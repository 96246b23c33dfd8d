"""2D slab scaling: c1, c2 and c3 at their BASELINE sizes and shipped knobs, cut into row slabs over the GPUs of one box
(GpuSlab, "p2p": drs_run_slab, one launch per sweep).  Run under torchrun at N = 1, 2, 4, 8:

    torchrun --nproc-per-node N tools/slab2d_scaling.py [--seconds 1.0] [--out result.json]

Per configuration: the single-GPU rate of Plan.run on the whole grid (rank 0, same knobs), then the slab run on every
rank -- warm-up calls, then timed calls of `iterations` timesteps (the .stc's) until at least --seconds have passed,
every rank making the same number of calls.  Reports GStencil/s (interior points x timesteps / wall time of the timed
calls, CUDA events, all ranks), parallel efficiency against N x the single-GPU rate, kernel launches per sweep, and
in-run parity: after the timed calls both buffers of every rank against the single-GPU run of the same number of
timesteps, bit for bit.  The card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
import torch.distributed as dist

import drstencil_b200 as drs
from drstencil_b200.presets import PRESETS
from drstencil_b200.slab import GpuSlab


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                        "-i", str(torch.cuda.current_device())], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return q.stdout.strip()


def interior(shape, halo):
    n = 1
    for d in shape:
        n *= max(0, d - 2 * halo)
    return n


def timed_calls(run, seconds, sync):
    """(calls, seconds) of back-to-back run() calls for at least `seconds` (the same call count on every rank)."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    run()
    e1.record()
    e1.synchronize()
    one = max(1e-6, e0.elapsed_time(e1) * 1e-3)
    calls = torch.tensor([max(2, int(seconds / one) + 1)], device="cuda")
    if sync:
        dist.all_reduce(calls, op=dist.ReduceOp.MAX)
        dist.barrier()
    calls = int(calls)
    e0.record()
    for _ in range(calls):
        run()
    e1.record()
    e1.synchronize()
    return calls, e0.elapsed_time(e1) * 1e-3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--configs", default="c1,c2,c3")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    results = {"world": world, "card": card() if rank == 0 else "", "configs": []}
    for name in a.configs.split(","):
        path, kn = PRESETS[name]
        st = drs.Stencil.from_file(path)
        shape, T = tuple(st.shape), st.iterations
        M, N = shape
        dt = torch.float32 if kn.dtype == drs.F32 else torch.float64
        g = torch.Generator(device="cuda")

        def row(yg):
            g.manual_seed(1000 + yg)
            return torch.rand((N,), dtype=dt, device="cuda", generator=g)

        slab = GpuSlab(path, kn, rank, world, halo="p2p", global_shape=shape)
        H, lo, hi = slab.geom.ghost, slab.geom.lo, slab.geom.hi
        slab.fill(row)
        n_sweeps = drs.sweep_count(T, kn.step)
        for _ in range(3):                                   # warm-up: module load, graph capture, clocks
            slab.run(T)
        slab.plan.sync_check()
        dist.barrier()
        l0 = slab.plan.launch_count
        calls, secs = timed_calls(lambda: slab.run(T), a.seconds, True)
        launches = (slab.plan.launch_count - l0) / float((calls + 1) * n_sweeps)
        slab.plan.sync_check()
        worst = torch.tensor([secs], device="cuda")
        dist.all_reduce(worst, op=dist.ReduceOp.MAX)
        total_calls = 3 + 1 + calls
        # in-run parity: the single-GPU run of the same timesteps from the same input, this rank's rows of both buffers
        ref = drs.Plan(drs.Stencil.from_file(path), kn)
        A = torch.stack([row(y) for y in range(M)])
        B = torch.zeros_like(A)
        for _ in range(total_calls):
            ref.run(A, B, T)
        ref.sync_check()
        same = bool(torch.equal(slab.owned(0), A[lo:hi])) and bool(torch.equal(slab.owned(1), B[lo:hi]))
        t = torch.tensor([1 if same else 0], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        # the single-GPU rate: Plan.run on the whole grid (rank 0), after the slab run, on the same buffers
        single = 0.0
        if rank == 0:
            for _ in range(3):
                ref.run(A, B, T)
            c1, s1 = timed_calls(lambda: ref.run(A, B, T), a.seconds, False)
            ref.sync_check()
            single = interior(shape, H) * T * c1 / s1 / 1e9
        del A, B
        rate = interior(shape, H) * T * calls / float(worst) / 1e9
        entry = {"config": name, "shape": list(shape), "knobs": str(kn), "halo": H, "timesteps_per_call": T,
                 "timed_calls": calls, "seconds": float(worst), "gstencil_s": rate, "single_gpu_gstencil_s": single,
                 "efficiency": rate / (world * single) if single else None, "gpu_launches_per_sweep": launches,
                 "rows_per_rank": hi - lo, "parity": "bit-exact" if int(t) else "MISMATCH"}
        if rank == 0:
            print(json.dumps(entry), flush=True)
            results["configs"].append(entry)
        slab.close()
        del ref
        torch.cuda.empty_cache()
        dist.barrier()
    if rank == 0:
        print(json.dumps(results), flush=True)
        if a.out:
            os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
            with open(a.out, "w") as f:
                json.dump(results, f, indent=1)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
