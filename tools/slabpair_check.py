"""Run under torchrun (one process per GPU, >= 2 GPUs): 3D grids cut into PAIR slabs (GpuSlab(..., pairs=True): ghost
regions of 2 Halo planes, drs_run_slab as exact pair launches plus single sweeps) against the undecomposed single-GPU
Plan.run of the same global grid, both buffers bit for bit, two calls in a row -- c4- and c5-shaped configurations
(the shipped knobs, grids cut down so the check stays short), sweep counts with both shapes of the split.  Prints
SLABPAIR_CHECK_OK on success."""
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
    # (preset, global shape, timesteps per call): 6 sweeps = 2 pairs + 2 singles, 8 = 2 + 4, 10 = 4 + 2
    for preset, shape, T in [("c4", (37 * world + 3, 136, 264), 6),
                             ("c5", (41 * world + 1, 200, 256), 8),
                             ("c5", (23 * world + 2, 96, 128), 10)]:
        path, kn = PRESETS[preset]
        L, M, N = shape
        g = torch.Generator(device="cuda")

        def plane(zg):
            g.manual_seed(91 + zg)
            return torch.rand((M, N), dtype=torch.float64, device="cuda", generator=g)

        plan = drs.Plan(drs.Stencil.from_file(path).set_size(shape), kn)
        A = torch.stack([plane(z) for z in range(L)])
        B = torch.zeros_like(A)
        refs = []
        for _ in range(2):                       # the reference after one call and after two
            plan.run(A, B, T)
            plan.sync_check()
            refs.append((A.clone(), B.clone()))
        del A, B
        slab = GpuSlab(path, kn, rank, world, halo="p2p", global_shape=shape, pairs=True)
        lo, hi = slab.geom.lo, slab.geom.hi
        split = slab.plan.slab_split(T)
        slab.fill(plane)
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
            print("slabpair_check %s %s T=%d split=%s world=%d -> %s" % (preset, shape, T, split, world,
                                                                         "bit-exact" if same else "MISMATCH"), flush=True)
        ok = ok and same and split[0] > 0
        slab.close()
        dist.barrier()
    if rank == 0:
        print("SLABPAIR_CHECK_OK" if ok else "SLABPAIR_CHECK_FAILED", flush=True)
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
