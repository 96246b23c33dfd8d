"""One GPU: c1 (2d5pt_star fp64 4096^2) and c3 (2d25pt_box fp32 16384^2) at their BASELINE sizes and preset knobs, drs_run
with single sweeps (the default) against drs_run with exact pair launches (Plan.set_pairs(True)), on the same plan and
the same buffers.  Each call runs 100 timesteps on c1 and 16 on c3 (c3's field overflows fp32 near 100 sweeps); A is
renormalised between calls, outside the timed region, so the field stays finite.  The two modes alternate in samples of
>= 1 s each, over three rounds.  Prints ms per call, GStencil/s (interior points x timesteps / s), the pair/single ratio,
whether both modes leave both buffers bit-identical (torch.equal), the card's name and its power limit.
Usage: python tools/pair2d_timing.py [rounds=3]"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch

import drstencil_b200 as drs
from drstencil_b200.presets import PRESETS

WORKLOADS = (("c1", 100), ("c3", 16))


def renormalise(A):
    A.mul_(1.0 / float(A.abs().max()))


def sample(plan, A, B, T, min_s=1.0):
    """ms per call of `T` timesteps over >= min_s seconds (CUDA events around each call)."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    calls, ms = 0, 0.0
    while ms < 1000.0 * min_s:
        renormalise(A)
        e0.record()
        plan.run(A, B, T)
        e1.record()
        e1.synchronize()
        ms += e0.elapsed_time(e1)
        calls += 1
    plan.sync_check()
    return ms / calls


def main():
    rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 3
    torch.cuda.set_device(0)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       stdout=subprocess.PIPE, text=True).stdout.strip()
    print("device: %s (%s)" % (torch.cuda.get_device_name(0), q), flush=True)
    for name, T in WORKLOADS:
        path, kn = PRESETS[name]
        plan = drs.Plan(drs.Stencil.from_file(path), kn)
        M, N = plan.stencil.shape
        H = plan.halo
        dt = torch.float64 if plan.info.dtype == 0 else torch.float32
        g = torch.Generator(device="cuda").manual_seed(7)
        A0 = torch.rand((M, N), generator=g, dtype=dt, device="cuda")
        B0 = torch.zeros_like(A0)
        # bit-identical results of the two modes from the same start
        outs = {}
        for pairs in (False, True):
            plan.set_pairs(pairs)
            A, B = A0.clone(), B0.clone()
            plan.run(A, B, T)
            plan.sync_check()
            outs[pairs] = (A, B)
        same = torch.equal(outs[False][0], outs[True][0]) and torch.equal(outs[False][1], outs[True][1])
        del outs
        print("%s: %dx%d %s, %d timesteps per call, split with pairs %s, A and B equal in both modes: %s" % (
            name, M, N, "fp64" if dt == torch.float64 else "fp32", T, plan.pair_split(T), same), flush=True)
        A, B = A0.clone(), B0.clone()
        res = {False: [], True: []}
        for k in range(rounds):
            for pairs in ((False, True) if k % 2 == 0 else (True, False)):
                plan.set_pairs(pairs)
                plan.run(A, B, T)                # warm-up: module load, graph capture (set_pairs drops the graphs)
                plan.sync_check()
                ms = sample(plan, A, B, T)
                res[pairs].append(ms)
                print("  round %d %-7s %9.3f ms per call" % (k, "pairs" if pairs else "singles", ms), flush=True)
        pts = (M - 2 * H) * (N - 2 * H) * T
        for pairs in (False, True):
            best = min(res[pairs])
            print("  %-7s min %.3f / max %.3f ms per call, %.1f GStencil/s" % (
                "pairs" if pairs else "singles", best, max(res[pairs]), pts / (best * 1e-3) / 1e9), flush=True)
        print("  %s pair/single speed ratio (min over rounds): %.3f" % (name, min(res[False]) / min(res[True])), flush=True)
        plan.set_pairs(False)
        del A, B, A0, B0
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
