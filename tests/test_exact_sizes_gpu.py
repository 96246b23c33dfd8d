"""Exact-arithmetic parity at the grid sizes where size-gated kernel paths switch on (exact_ops.size_cases): the
shipped configurations at their sizes, both sides of the 1 GiB rule (L2 load hint, exact pair launches) and of the
flat 1 -> 2 rule of unaligned rows, arrays past 2^31 elements, and run_host at c4's size.  The input is procedural, so
each slow-axis window of both buffers is compared with torch.equal against a float64 reference computed on the device
from just the source window it depends on; device memory stays at the engine's two arrays plus one window.
test_exact_sizes.py checks every case's plan, thresholds and exactness budget on the CPU."""
import time

import numpy as np
import pytest

import exact_ops as X

pytestmark = pytest.mark.gpu

SEED = 11
# the reference of one window: both buffers, two levels of apply_levels, a product temporary and the hash's int64
# temporaries, in float64 / int64 units of the largest source window
WINDOW_COPIES = 12


def _free():
    import gc
    import torch
    gc.collect()
    torch.cuda.empty_cache()


def _report(shape, info, bad, first):
    lines = ["%s: %d of %d points differ" % (name, n, int(np.prod(shape))) for name, n in bad.items() if n]
    return "; ".join(lines) + "; first: " + " | ".join(first)


@pytest.mark.parametrize("cid", [c["id"] for c in X.size_cases()])
def test_exact_at_size(built, cid):
    import torch
    import drstencil_b200 as drs
    case = X.size_case(cid)
    _free()
    t0 = time.time()
    shape, op, step, sweeps, runner = case["shape"], X.OPS[case["op"]], X.step_of(case), case["sweeps"], case["runner"]
    dt = torch.float32 if case["dtype"] == "f32" else torch.float64
    plan = X.size_plan(case)
    info = plan.info
    assert X.size_markers(case, plan) == [], cid
    assert X.size_growth_ok(case)[0], cid
    nbytes = int(np.prod(shape)) * X.esize(case["dtype"])
    plane = int(np.prod(shape[1:]))
    wmax = max(np.subtract(*X.source_window(op, step, sweeps, shape[0], z0, z1)[::-1]) for z0, z1 in X.windows(shape))
    need = 2 * nbytes + WINDOW_COPIES * 8 * wmax * plane
    free = torch.cuda.mem_get_info()[0]
    if free < need:
        pytest.skip("%s needs %d bytes of free device memory, %d are free" % (cid, need, free))
    torch.cuda.reset_peak_memory_stats()
    dev = torch.empty(0, device="cuda")
    imps = X.impulses(shape, info)
    host = runner in ("host", "host_streamed")
    b_init = 0.0 if host else -7.0          # run_host's own second buffer starts as zeros
    T = sweeps * step
    if host:
        A, B = torch.empty(shape, dtype=dt, pin_memory=True), None
    else:
        A, B = torch.empty(shape, dtype=dt, device="cuda"), torch.full(shape, b_init, dtype=dt, device="cuda")
    for z0, z1 in X.windows(shape):
        A[z0:z1].copy_(X.gen_input(shape, z0, z1, SEED, imps, like=dev).to(dt))
    l0 = plan.launch_count
    if host:
        plan.set_host_block(-1 if runner == "host" else 0)
        plan.run_host(A, None, T)
        n = drs.sweep_count(T, step)
        if runner == "host":
            assert plan.host_schedule(T) == []
            assert plan.launch_count - l0 == sum(plan.pair_split(T))
        else:
            assert plan.host_schedule(T) != []
            assert plan.launch_count - l0 > n, "the streamed path did not run"
    else:
        if runner == "sweep":
            plan.sweep(A, B)
            n = 1
        else:
            n = plan.run(A, B, T)
        plan.sync_check()
        launches = plan.launch_count - l0
        if case["pair"]:
            pairs, singles = plan.pair_split(T)
            assert pairs > 0 and launches == pairs + singles, (launches, pairs, singles)
        elif case["path"] == "multi3d":
            assert launches == n * step
        elif runner == "run":
            assert launches == n
    assert n == sweeps
    t_run = time.time()

    def source(s0, s1):
        a = X.gen_input(shape, s0, s1, SEED, imps, like=dev)
        return a, torch.full_like(a, b_init)

    bad, first = {"A": 0, "B": 0}, []
    for z0, z1 in X.windows(shape):
        refs = X.window_run(op, step, sweeps, shape, z0, z1, source)
        for name, buf, ref in (("A", A, refs[0]), ("B", B, refs[1])):
            if buf is None:
                continue
            got = buf[z0:z1].to(device="cuda", dtype=torch.float64)
            if torch.equal(got, ref):
                continue
            diff = got != ref
            bad[name] += int(diff.sum())
            for idx in diff.nonzero()[:max(0, 4 - len(first))].tolist():
                g = (idx[0] + z0,) + tuple(idx[1:])
                first.append(name + " " + X.describe_mismatch(g, shape, info, float(got[tuple(idx)]),
                                                              float(ref[tuple(idx)])))
        del refs
    peak = torch.cuda.max_memory_allocated()
    print("%s %s %s: %d sweeps, %d launches, run %.1f s, check %.1f s, peak allocated %.2f GiB%s"
          % (cid, shape, case["dtype"], n, plan.launch_count - l0, t_run - t0, time.time() - t_run, peak / 2 ** 30,
             " (+ the plan's two device buffers)" if host else ""))
    del A, B, plan
    _free()
    assert not any(bad.values()), "%s: %s" % (cid, _report(shape, info, bad, first))
