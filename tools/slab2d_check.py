"""Run under torchrun (one process per GPU, >= 2 GPUs): 2D grids cut into row slabs through GpuSlab against the
undecomposed single-GPU run of the same global grid, both buffers bit for bit, two calls in a row -- c1-, c2- and
c3-shaped configurations in the "p2p" mode (run and run_host) and in "p2p-flags".  Prints SLAB2D_CHECK_OK on success."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
import torch.distributed as dist

import drstencil_b200 as drs
from drstencil_b200.presets import PRESETS
from drstencil_b200.slab import GpuSlab


def agree(flag):
    t = torch.tensor([1 if flag else 0], device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    return bool(int(t))


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ok = True
    # (preset, global shape, timesteps per call, host block): shipped knobs, grids cut down so the check stays short
    for preset, shape, T, block in [("c1", (96 * world + 5, 1030), 4, 24),
                                    ("c2", (128 * world + 3, 2048), 8, 32),
                                    ("c3", (64 * world + 1, 1024), 4, 16)]:
        path, kn = PRESETS[preset]
        M, N = shape
        dt = torch.float32 if kn.dtype == drs.F32 else torch.float64
        g = torch.Generator(device="cuda")

        def row(yg):
            g.manual_seed(77 + yg)
            return torch.rand((N,), dtype=dt, device="cuda", generator=g)

        plan = drs.Plan(drs.Stencil.from_file(path).set_size(shape), kn)
        A = torch.stack([row(y) for y in range(M)])
        B = torch.zeros_like(A)
        refs = []
        for _ in range(2):                       # the reference after one call and after two
            plan.run(A, B, T)
            plan.sync_check()
            refs.append((A.clone(), B.clone()))
        for mode in ("p2p", "p2p-flags"):
            slab = GpuSlab(path, kn, rank, world, halo=mode, global_shape=shape)
            lo, hi = slab.geom.lo, slab.geom.hi
            if mode == "p2p":
                # the host-buffer path (drs_run_host_slab) against Plan.run_host, two calls on the same object: the
                # flag numbering carries over; then the device path on the same object
                slab.plan.set_host_block(block)
                ref_host = torch.stack([row(y) for y in range(M)]).cpu()
                plan.run_host(ref_host, None, T)
                same = True
                for call in range(2):
                    h = torch.stack([row(y) for y in range(lo, hi)]).cpu().pin_memory()
                    slab.run_host(h, T)
                    same = same and bool(torch.equal(h, ref_host[lo:hi]))
                same = agree(same)
                if rank == 0:
                    print("slab2d_check run_host %s %s block=%d world=%d -> %s" % (
                        preset, shape, block, world, "bit-exact" if same else "MISMATCH"), flush=True)
                ok = ok and same
            slab.fill(row)
            same = True
            for call in range(2):
                slab.run(T)
                slab.plan.sync_check()
                torch.cuda.synchronize()
                dist.barrier()
                for b in (0, 1):
                    same = same and bool(torch.equal(slab.owned(b), refs[call][b][lo:hi]))
            same = agree(same)
            if rank == 0:
                print("slab2d_check %s %s mode=%s world=%d -> %s" % (preset, shape, mode, world,
                                                                    "bit-exact" if same else "MISMATCH"), flush=True)
            ok = ok and same
            slab.close()
            dist.barrier()
    if rank == 0:
        print("SLAB2D_CHECK_OK" if ok else "SLAB2D_CHECK_FAILED", flush=True)
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
