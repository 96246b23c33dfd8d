"""One GPU: drs_run_slab on a middle rank of c5's N = 8 slab (1536^2 planes, 192 owned planes) with passive neighbours,
single sweeps (set_slab: Halo ghost planes, one launch per sweep) against pair launches (set_slab_pairs: 2 Halo ghost
planes, drs_plan_slab_split's pairs and singles).  The rank's own flag words are released in advance and its
neighbours are device arrays on the same GPU, so this is the per-GPU kernel rate of a slab rank: the peer stores go to
local memory, not over NVLink.  Alternates the two for >= 1 s per sample, three rounds; prints ms per 100 timesteps,
the card's name and its power limit.  Usage: python tools/slabpair_timing.py [timesteps=100] [rounds=3]"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch

import drstencil_b200 as drs
from drstencil_b200.presets import PRESETS
from drstencil_b200.slab import SlabGeometry


def setup(pairs, path, kn, G, rest, world=8, rank=3):
    H = 1
    g = SlabGeometry(G, world, rank, 2 * H if pairs else H, ring=H)
    shape = (g.local_planes,) + rest
    plan = drs.Plan(drs.Stencil.from_file(path).set_size(shape), kn)
    (plan.set_slab_pairs if pairs else plan.set_slab)(G, g.lo, g.hi)
    bufs = [torch.zeros(shape, dtype=torch.float64, device="cuda") for _ in range(2)]
    bufs[0].uniform_()
    nb = {}
    for side, r in (("lower", g.lower), ("upper", g.upper)):
        gn = SlabGeometry(G, world, r, g.ghost, ring=H)
        nb[side] = (gn, [torch.zeros((gn.local_planes,) + rest, dtype=torch.float64, device="cuda") for _ in range(2)])
    flags = torch.full((2,), 1 << 62, dtype=torch.int64, device="cuda")
    words = torch.zeros(4, dtype=torch.int64, device="cuda")
    plan.set_peers(bufs, nb["lower"][1], nb["upper"][1], nb["lower"][0].lo, nb["upper"][0].lo)
    plan.set_flags(flags.data_ptr(), words.data_ptr() + 8, words.data_ptr() + 16)
    return dict(plan=plan, keep=(bufs, nb, flags, words), g=g)


def sample(run, T, min_s=1.0):
    """ms per call of `T` timesteps over >= min_s seconds (CUDA events)."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    calls, ms = 0, 0.0
    while ms < 1000.0 * min_s:
        e0.record()
        for _ in range(3):
            run.run_slab(T)
        e1.record()
        e1.synchronize()
        ms += e0.elapsed_time(e1)
        calls += 3
    run.sync_check()
    return ms / calls


def main():
    T = int(sys.argv[1]) if len(sys.argv) > 1 else 100
    rounds = int(sys.argv[2]) if len(sys.argv) > 2 else 3
    torch.cuda.set_device(0)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       stdout=subprocess.PIPE, text=True).stdout.strip()
    print("device: %s (%s)" % (torch.cuda.get_device_name(0), q), flush=True)
    path, kn = PRESETS["c5"]
    shape = drs.Stencil.from_file(path).shape
    G, rest = shape[0], tuple(shape[1:])
    runs = {"singles": setup(False, path, kn, G, rest), "pairs": setup(True, path, kn, G, rest)}
    for name, r in runs.items():
        r["plan"].run_slab(T)                     # warm-up: module load, graph capture
        r["plan"].sync_check()
        print("%s: %d local planes of %dx%d, split %s" % (name, r["g"].local_planes, rest[0], rest[1],
                                                         r["plan"].slab_split(T)), flush=True)
    res = {n: [] for n in runs}
    for k in range(rounds):
        for name in (("singles", "pairs") if k % 2 == 0 else ("pairs", "singles")):
            ms = sample(runs[name]["plan"], T)
            res[name].append(ms * 100.0 / T)
            print("round %d %-7s %8.2f ms per 100 timesteps" % (k, name, res[name][-1]), flush=True)
    owned = 192 * rest[0] * rest[1]
    for name, v in res.items():
        best = min(v)
        print("%-7s min %.2f / max %.2f ms per 100 timesteps, %.1f GStencil/s of owned points" % (
            name, best, max(v), owned * 100 / (best * 1e-3) / 1e9), flush=True)
    print("pair/single time ratio (min over rounds): %.3f" % (min(res["pairs"]) / min(res["singles"])), flush=True)


if __name__ == "__main__":
    main()
