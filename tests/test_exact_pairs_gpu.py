"""drs_run's exact pair launches, bit for bit: Plan.run on a plan with pair launches leaves in both buffers, ring
included, exactly what a loop of single sweeps (Plan.sweep, the kernel the other exact tests hold to the gold chain)
leaves there.  B starts at -7, so the two buffers' rings differ and a level that takes its ring from the wrong buffer
shows.  test_exact_pairs.py checks the plans and the generated units on the CPU."""
import pytest

import drstencil_b200 as drs
from drstencil_b200.presets import PRESETS
from helpers import stc_path

pytestmark = pytest.mark.gpu


def _fill(shape, dtype, seed, impulses=()):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    a = torch.rand(shape, generator=g, dtype=dtype, device="cuda") * 2 - 1
    for idx in impulses:
        a[idx] = 64.0 * (1 if sum(idx) % 2 else -1)
    return a, torch.full(shape, -7.0, dtype=dtype, device="cuda")


def _check(plan, shape, dtype, Ts, seed=1, impulses=()):
    import torch
    for T in Ts:
        A, B = _fill(shape, dtype, seed + T, impulses)
        rA, rB = A.clone(), B.clone()
        n = drs.sweep_count(T, 1)
        pairs, singles = plan.pair_split(T)
        assert pairs > 0 and 2 * pairs + singles == n
        l0 = plan.launch_count
        assert plan.run(A, B, T) == n
        plan.sync_check()
        assert plan.launch_count - l0 == pairs + singles
        bufs = [rA, rB]
        for s in range(n):
            plan.sweep(bufs[s % 2], bufs[(s + 1) % 2])
        plan.sync_check()
        okA, okB = torch.equal(A, rA), torch.equal(B, rB)
        if not (okA and okB):
            bad = [(name, int((X != R).sum()), (X != R).nonzero()[:4].tolist())
                   for name, X, R in (("A", A, rA), ("B", B, rB)) if not torch.equal(X, R)]
            pytest.fail("T=%d: %s" % (T, bad))
        del A, B, rA, rB
        torch.cuda.empty_cache()


def _seams(shape, plan):
    """Impulses on the pair kernel's tile seams (x, y) and chunk boundaries (z)."""
    H = plan.info.halo
    L, M, N = shape
    zs = [z for q in (0, 1, 2) for z in (H + 128 * q - 1, H + 128 * q) if 0 <= z < L] + [L - H - 1, L - H]
    ys = [H - 1, H, H + 29, H + 30, M - H - 1, M - H]
    xs = [H - 1, H, H + 59, H + 60, H + 63, H + 64, N - H - 1, N - H]
    return [(z, y, x) for z in zs for y in ys for x in xs if 0 <= z < L and 0 <= y < M and 0 <= x < N]


@pytest.mark.parametrize("name", ["c5", "c4"])
def test_pairs_equal_single_sweeps_presets(built, name):
    import torch
    path, kn = PRESETS[name]
    plan = drs.Plan(drs.Stencil.from_file(path), kn)
    assert plan.pair_source
    _check(plan, plan.stencil.shape, torch.float64, (6, 8, 10, 16, 100))


def test_pairs_equal_single_sweeps_fp32(built):
    import torch
    shape = (512, 520, 1024)
    plan = drs.Plan(drs.Stencil.from_file(stc_path("3d7pt_star")).set_size(shape), drs.Knobs(dtype="f32"))
    assert plan.pair_source
    _check(plan, shape, torch.float32, (6, 8, 14), impulses=_seams(shape, plan))


@pytest.mark.parametrize("op", ["box27", "aniso", "kside", "star7neg"])
def test_pairs_equal_single_sweeps_operators(built, op):
    import torch
    import exact_ops as X
    o = X.OPS[op]
    offs = list(o)
    shape = (520, 512, 516)
    plan = drs.Plan(drs.Stencil.from_points(offs, [o[k] for k in offs], shape, 2, name="pair_" + op), drs.Knobs())
    assert plan.pair_source
    _check(plan, shape, torch.float64, (6, 8), impulses=_seams(shape, plan))
