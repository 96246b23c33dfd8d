"""Exact pair launches against the single-sweep loop on the c5 and c4 presets, in one process: five rounds, each runs
Plan.run (pair launches) and a loop of Plan.sweep (one launch per sweep) from the same seeded buffers, checks both
buffers with torch.equal and prints the time of each arm (CUDA events) as one JSON line per round.

    python tools/pair_check.py [--rounds 5] [--timesteps 100] [--presets c5,c4]
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--timesteps", type=int, default=100)
    ap.add_argument("--presets", default="c5,c4")
    args = ap.parse_args()
    import torch
    import drstencil_b200 as drs
    from drstencil_b200.presets import PRESETS
    torch.cuda.set_device(0)
    print(json.dumps({"device": torch.cuda.get_device_name(0)}), flush=True)
    ok_all = True
    for name in args.presets.split(","):
        path, kn = PRESETS[name]
        plan = drs.Plan(drs.Stencil.from_file(path), kn)
        shape, T = plan.stencil.shape, args.timesteps
        n = drs.sweep_count(T, 1)
        pairs, singles = plan.pair_split(T)
        g = torch.Generator(device="cuda")
        A = torch.empty(shape, dtype=torch.float64, device="cuda")
        B, rA, rB = torch.empty_like(A), torch.empty_like(A), torch.empty_like(A)

        def reset(seed):
            g.manual_seed(seed)
            torch.rand(shape, generator=g, dtype=torch.float64, device="cuda", out=A)
            B.fill_(-7.0)
            rA.copy_(A)
            rB.copy_(B)

        def timed(fn):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            return e0.elapsed_time(e1)

        def loop():
            bufs = [rA, rB]
            for s in range(n):
                plan.sweep(bufs[s % 2], bufs[(s + 1) % 2])

        reset(0)                      # warm-up: modules, tensor maps, the captured graph
        plan.run(A, B, T)
        loop()
        plan.sync_check()
        for r in range(args.rounds):
            reset(r + 1)
            first_pairs = r % 2 == 0  # alternate which arm runs first
            t_run = t_loop = None
            for arm in ((0, 1) if first_pairs else (1, 0)):
                if arm == 0:
                    l0 = plan.launch_count
                    t_run = timed(lambda: plan.run(A, B, T))
                    launches = plan.launch_count - l0
                else:
                    t_loop = timed(loop)
            plan.sync_check()
            ok = torch.equal(A, rA) and torch.equal(B, rB)
            ok_all &= ok and launches == pairs + singles
            print(json.dumps({"preset": name, "round": r, "timesteps": T, "pairs": pairs, "singles": singles,
                              "launches": launches, "run_ms": round(t_run, 3), "sweep_loop_ms": round(t_loop, 3),
                              "speedup": round(t_loop / t_run, 4), "equal": ok}), flush=True)
        del A, B, rA, rB, plan
        torch.cuda.empty_cache()
    sys.exit(0 if ok_all else 1)


if __name__ == "__main__":
    main()
