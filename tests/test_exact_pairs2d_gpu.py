"""Opt-in exact pair launches on 2D plans, bit for bit: after set_pairs(True), Plan.run leaves in both buffers, ring
included, exactly what a loop of single sweeps (Plan.sweep) leaves there, and -- for the exact operators of
exact_ops.py, where growth_ok allows -- exactly the float64 reference exact_run.  B starts at -7, so the two buffers'
rings differ and a level that takes its ring from the wrong buffer shows.  test_exact_pairs2d.py checks the plans and
the generated units on the CPU."""
import numpy as np
import pytest

import drstencil_b200 as drs
import exact_ops as X
from drstencil_b200.presets import PRESETS

pytestmark = pytest.mark.gpu

EXACT_2D = ("star5", "box9", "box25", "mixed3x3", "onesided", "star3gap", "unit", "two", "sep121")


def _torch():
    import torch
    return torch


def _tdtype(dt):
    t = _torch()
    return t.float64 if dt == "f64" else t.float32


def _plan(op, shape, dt, name=None, knobs=None):
    o = X.OPS[op]
    offs = list(o)
    kn = dict(knobs or {}, dtype=dt)
    st = drs.Stencil.from_points(offs, [o[k] for k in offs], shape, 2, name=name or "pair2d_" + op)
    plan = drs.Plan(st, drs.Knobs(**kn))
    plan.set_pairs(True)
    return plan


def _geometry(plan, op, dt):
    """(halo, columns a warp strip stores, rows of a chunk) of the plan's pair unit."""
    src = plan.pair_source
    d = {k: int(v) for k, v in (l.split()[1:3] for l in src.splitlines() if l.startswith("#define DRS_") and
                                 len(l.split()) == 3 and l.split()[2].lstrip("-").isdigit())}
    vec = 2 if dt == "f64" else 4
    hw = -(-d["DRS_E"] // vec) * vec
    wu = 32 * d["DRS_VT"] * vec - 2 * hw
    o = X.OPS[op]
    st = drs.Stencil.from_points(list(o), list(o.values()), (4096, 1024), 2)
    chunk = drs.Plan(st, drs.Knobs(step=2, fuse="temporal", dtype=dt)).info.chunk
    return d["DRS_HALO"], wu, chunk


def _seams(shape, H, wu, chunk):
    """Impulse positions on strip seams (x), chunk seams (y) and the ring rows and columns."""
    M, N = shape
    xs = [H - 1, H, N - H - 1, N - H] + [H + q * wu + d for q in (1, 2) for d in (-1, 0)]
    ys = [H - 1, H, M - H - 1, M - H] + [H + q * chunk + d for q in (1, 2) for d in (-1, 0)]
    return [(y, x) for y in ys for x in xs if 0 <= y < M and 0 <= x < N]


def _inputs(shape, dt, seed, impulses=(), integer=True):
    torch = _torch()
    g = torch.Generator(device="cuda").manual_seed(seed)
    if integer:
        a = torch.randint(-X.UMAX, X.UMAX + 1, shape, generator=g, device="cuda").to(_tdtype(dt))
    else:
        a = torch.rand(shape, generator=g, dtype=_tdtype(dt), device="cuda") * 2 - 1
    for k, idx in enumerate(impulses):
        a[idx] = X.IMPULSE * (1 if k % 2 else -1)
    return a, torch.full(shape, -7.0, dtype=_tdtype(dt), device="cuda")


def _mismatch(name, got, ref):
    torch = _torch()
    bad = (got != ref).nonzero()
    return "%s: %d cells differ, first %s" % (name, bad.shape[0], bad[:4].tolist()) if not torch.equal(got, ref) else ""


def _check(plan, A0, B0, T, op=None, graph=True, stream=None):
    """run() with pair launches against the loop of single sweeps (and against exact_run when op is given)."""
    torch = _torch()
    n = drs.sweep_count(T, 1)
    pairs, singles = plan.pair_split(T)
    assert 2 * pairs + singles == n
    A, B, rA, rB = A0.clone(), B0.clone(), A0.clone(), B0.clone()
    torch.cuda.synchronize()            # the copies are on the current stream, run() may be on another
    plan.set_graph(graph)
    l0 = plan.launch_count
    assert plan.run(A, B, T, stream=stream) == n
    plan.sync_check(stream)
    assert plan.launch_count - l0 == pairs + singles
    bufs = [rA, rB]
    for s in range(n):
        plan.sweep(bufs[s % 2], bufs[(s + 1) % 2])
    plan.sync_check()
    errs = [e for e in (_mismatch("A", A, rA), _mismatch("B", B, rB)) if e]
    if op is not None:
        ref = X.exact_run(X.OPS[op], 1, A0, B0, n)
        errs += [e for e in (_mismatch("A vs exact", A.to(torch.float64), ref[0]),
                             _mismatch("B vs exact", B.to(torch.float64), ref[1])) if e]
    assert not errs, "T=%d pairs=%d: %s" % (T, pairs, errs)
    plan.set_graph(True)
    return pairs


def _exact_ok(op, dt, n, u):
    return X.growth_ok(dict(op=op, dtype=dt, knobs={}, sweeps=n), u.cpu().numpy())[0]


@pytest.mark.parametrize("dt", ["f64", "f32"])
@pytest.mark.parametrize("op", EXACT_2D)
def test_operators_with_seam_impulses(built, op, dt):
    """Several chunks with a one-row last chunk, a ragged last strip, impulses on the strip and chunk seams and on the
    ring rows and columns; 6 and 8 sweeps (both shapes of the split)."""
    probe = _plan(op, (300, 520), dt)
    H, wu, chunk = _geometry(probe, op, dt)
    shape = (2 * H + 2 * chunk + 1, 2 * H + 2 * wu + 5 - (2 * H + 2 * wu + 5) % (2 if dt == "f64" else 4))
    plan = _plan(op, shape, dt)
    for T in (6, 8):
        A0, B0 = _inputs(shape, dt, 17 + T, _seams(shape, H, wu, chunk))
        exact = _exact_ok(op, dt, drs.sweep_count(T, 1), A0)
        assert _check(plan, A0, B0, T, op if exact else None) > 0


@pytest.mark.parametrize("op,dt", [("star5", "f64"), ("box25", "f64"), ("onesided", "f32"), ("star3gap", "f64")])
def test_small_grids(built, op, dt):
    """A grid narrower than one strip, fewer rows than one chunk, and the smallest grid with an interior."""
    probe = _plan(op, (300, 520), dt)
    H, wu, chunk = _geometry(probe, op, dt)
    vec = 2 if dt == "f64" else 4

    def al(n):
        return -(-n // vec) * vec
    for shape in ((2 * H + chunk // 2, al(2 * H + wu // 2)), (2 * H + 3, al(2 * H + wu + vec)), (2 * H + 1, al(2 * H + 1))):
        plan = _plan(op, shape, dt)
        A0, B0 = _inputs(shape, dt, 5, _seams(shape, H, wu, chunk))
        _check(plan, A0, B0, 6, op if _exact_ok(op, dt, 6, A0) else None)


def test_sweep_counts_graphs_streams(built):
    """Sweep counts 2 and 4 (no pair launches), 6, 8, 10, 16 and 100; graph replay on and off; a non-default stream;
    set_pairs(False) returns to single sweeps."""
    torch = _torch()
    op, dt, shape = "star5", "f64", (390, 522)
    plan = _plan(op, shape, dt)
    H, wu, chunk = _geometry(plan, op, dt)
    for T in (2, 4, 6, 8, 10, 16, 100):
        A0, B0 = _inputs(shape, dt, T, _seams(shape, H, wu, chunk))
        n = drs.sweep_count(T, 1)
        pairs = _check(plan, A0, B0, T, op if _exact_ok(op, dt, n, A0) else None)
        assert (pairs > 0) == (n >= 6)
    A0, B0 = _inputs(shape, dt, 3, _seams(shape, H, wu, chunk))
    _check(plan, A0, B0, 10, op, graph=False)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        A1, B1 = A0.clone(), B0.clone()
    s.synchronize()
    _check(plan, A1, B1, 10, op, stream=s.cuda_stream)
    _check(plan, A1, B1, 10, op, graph=False, stream=s.cuda_stream)
    plan.set_pairs(False)
    assert plan.pair_split(10) == (0, 10)
    l0 = plan.launch_count
    A, B = A0.clone(), B0.clone()
    plan.run(A, B, 10)
    plan.sync_check()
    assert plan.launch_count - l0 == 10
    ref = X.exact_run(X.OPS[op], 1, A0, B0, 10)
    assert torch.equal(A.double(), ref[0]) and torch.equal(B.double(), ref[1])


def test_run_host_plain(built):
    """The plain drs_run_host sequence (h_b given) runs the pair schedule: A ends as after the single sweeps."""
    torch = _torch()
    op, dt, shape = "mixed3x3", "f64", (300, 522)
    plan = _plan(op, shape, dt)
    A0, B0 = _inputs(shape, dt, 9)
    h_a, h_b = A0.cpu().numpy().copy(), B0.cpu().numpy().copy()
    pairs, singles = plan.pair_split(10)
    assert pairs > 0
    l0 = plan.launch_count
    plan.run_host(h_a, h_b, 10)
    assert plan.launch_count - l0 == pairs + singles
    rA, rB = A0.clone(), B0.clone()
    bufs = [rA, rB]
    for s in range(10):
        plan.sweep(bufs[s % 2], bufs[(s + 1) % 2])
    plan.sync_check()
    assert np.array_equal(h_a, rA.cpu().numpy())
    ref = X.exact_run(X.OPS[op], 1, A0, B0, 10)
    assert torch.equal(torch.from_numpy(h_a).cuda().double(), ref[0])


@pytest.mark.parametrize("name,op", [("c1", "star5"), ("c3", "box25")])
def test_presets_at_size(built, name, op):
    """c1 (4096^2 fp64) and c3 (16384^2 fp32) at their sizes and knobs: the preset stencils on random values, and the
    shaped exact operators, against the single-sweep loop (and exact_run where growth_ok allows)."""
    torch = _torch()
    path, kn = PRESETS[name]
    real = drs.Plan(drs.Stencil.from_file(path), kn)
    shape = real.stencil.shape
    dt = "f64" if real.info.dtype == 0 else "f32"
    real.set_pairs(True)
    for T in ((6, 8, 10, 16, 100) if name == "c1" else (6, 8, 16)):
        A0, B0 = _inputs(shape, dt, 40 + T, integer=False)
        assert _check(real, A0, B0, T) > 0
        del A0, B0
        torch.cuda.empty_cache()
    o = X.OPS[op]
    shaped = drs.Plan(drs.Stencil.from_points(list(o), list(o.values()), shape, 2, name="shaped_" + op), kn)
    shaped.set_pairs(True)
    geom = ("DRS_T", "DRS_HALO", "DRS_RJ", "DRS_E", "DRS_NW", "DRS_ST", "DRS_RB", "DRS_VT", "DRS_MINB")
    defs = [{l.split()[1]: l.split()[2:] for l in p.pair_source.splitlines() if l.startswith("#define DRS_")}
            for p in (real, shaped)]
    assert [defs[0][k] for k in geom] == [defs[1][k] for k in geom], defs
    H, wu, chunk = _geometry(shaped, op, dt)
    for T in ((6, 10) if name == "c1" else (6,)):
        A0, B0 = _inputs(shape, dt, 60 + T, _seams(shape, H, wu, chunk))
        n = drs.sweep_count(T, 1)
        _check(shaped, A0, B0, T, op if _exact_ok(op, dt, n, A0) else None)
        del A0, B0
        torch.cuda.empty_cache()


def test_3d_plan_below_1gib(built):
    """One 3D plan below 1 GiB with set_pairs(True) runs the 3D pair unit, bit for bit."""
    op, dt, shape = "star7neg", "f64", (70, 72, 136)
    plan = _plan(op, shape, dt)
    assert '#include "drs_pair3d.cuh"' in plan.pair_source
    for T in (6, 8):
        A0, B0 = _inputs(shape, dt, T)
        _check(plan, A0, B0, T, op)
