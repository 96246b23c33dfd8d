"""Exact-arithmetic parity of every kernel path on non-smoothing operators (exact_ops.py): mixed signs, coefficients of
+-1, zero gaps, one-sided and anisotropic extents, fp32 and fp64, temporal depth up to 6.  Inputs and coefficients are
short dyadics, so every correct evaluation order gives the exact answer and the whole of both buffers -- interior,
frozen ring, ping-pong partner -- is compared with array_equal.  test_exact_operators.py proves each case's
preconditions and path markers on the CPU.

The range tests hold operators with a tiny leading coefficient, whose deferred scale would leave the dtype's range, to a
pointwise condition-aware bound against a higher-precision reference."""
import numpy as np
import pytest

import exact_ops as X

pytestmark = pytest.mark.gpu


def _dev(a):
    import torch
    return torch.from_numpy(a).cuda()


def _mismatch(got, ref, H):
    """Count and first few indices of the differing points, with whether they sit in the frozen ring."""
    bad = np.argwhere(got != ref)
    shape = got.shape
    first = [(tuple(int(v) for v in i), "ring" if any(v < H or v >= n - H for v, n in zip(i, shape)) else "interior",
              float(got[tuple(i)]), float(ref[tuple(i)])) for i in bad[:4]]
    return "%d of %d points differ, first %s" % (len(bad), got.size, first)


@pytest.mark.parametrize("cid", [c["id"] for c in X.CASES])
def test_exact_operator_bit_for_bit(built, cid, monkeypatch):
    import torch
    import drstencil_b200 as drs
    case = X.CASE_BY_ID[cid]
    X.set_env(case, monkeypatch)
    op, step, sweeps, runner = X.OPS[case["op"]], X.step_of(case), case["sweeps"], case["runner"]
    dt = np.float32 if case["dtype"] == "f32" else np.float64
    for n_shape, shape in enumerate(X.shapes(case)):
        plan = X.make_plan(case, shape)
        info = plan.info
        H = info.halo
        assert X.markers(case, plan, shape, bool(case["env"])) == [], (cid, shape)
        a0 = X.make_input(case, shape, info, seed=1000 + n_shape)
        assert X.growth_ok(case, a0)[0]
        b0 = np.full(shape, -7, dt)
        l0 = plan.launch_count
        if runner in ("host", "host_streamed"):
            b0 = np.zeros(shape, dt)            # run_host's own second buffer starts as zeros
            a = torch.from_numpy(a0.copy()).pin_memory()
            block = 4 * H + 1
            plan.set_host_block(-1 if runner == "host" else block)
            plan.run_host(a, None, sweeps * step)
            n = drs.sweep_count(sweeps * step, step)
            if runner == "host_streamed" and shape[0] >= 4 * block:
                assert plan.launch_count - l0 > n, "the streamed path did not run"
            got_a, got_b = a.numpy(), None
        else:
            A, B = _dev(a0), _dev(b0)
            if runner == "sweep":
                assert sweeps == 1
                plan.sweep(A, B)
                n = 1
            elif runner == "gold":
                n = plan.gold_run(A, B, sweeps * step)
            else:
                n = plan.run(A, B, sweeps * step)
            plan.sync_check()
            got_a, got_b = A.cpu().numpy(), B.cpu().numpy()
            if case["path"] == "multi3d":
                assert plan.launch_count - l0 == n * step
        assert n == sweeps
        exA, exB = X.exact_run(op, step, a0, b0, sweeps)
        assert np.array_equal(got_a, exA), (cid, shape, "A", _mismatch(got_a, exA, H))
        if got_b is not None:
            assert np.array_equal(got_b, exB), (cid, shape, "B", _mismatch(got_b, exB, H))


@pytest.mark.parametrize("name", sorted(X.RANGE_OPS))
def test_deferred_scale_stays_in_range(built, name):
    """|got - ref| <= (P ts + 4) eps |K|^ts |u| pointwise, every value finite, the ring untouched: an operator whose
    leading coefficient is tiny must not be evaluated as K / eta with levels growing like eta^-s."""
    op, shape, dtype, step, factored = X.RANGE_OPS[name]
    plan = X.range_plan(name)
    src = plan.source
    assert "#define DRS_TS %d\n" % step in src and ("#define DRS_FACTORED 1" in src) == factored
    assert ("drs_sweep3d_t.cuh" in src) == (len(shape) == 3)
    dt = np.float32 if dtype == "f32" else np.float64
    ref_dt = np.float64 if dtype == "f32" else np.longdouble
    a0 = np.random.default_rng(5).uniform(0.5, 1.5, size=shape).astype(dt)
    b0 = np.zeros(shape, dt)
    A, B = _dev(a0), _dev(b0)
    plan.sweep(A, B)
    plan.sync_check()
    got = B.cpu().numpy()
    inner = X.interior(shape, plan.info.halo)
    ref = X.apply_levels(a0, op, step, dtype=ref_dt)[inner]
    mag = X.apply_levels(a0, op, step, mag=True, dtype=ref_dt)[inner]
    assert np.all(np.isfinite(got)), "%d of %d values not finite" % (np.sum(~np.isfinite(got)), got.size)
    bound = (len(op) * step + 4) * ref_dt(np.finfo(dt).eps) * mag
    err = np.abs(got[inner].astype(ref_dt) - ref)
    assert np.all(err <= bound), "max error / bound %.3g" % float(np.max(err / bound))
    ring = np.ones(shape, bool)
    ring[inner] = False
    assert np.array_equal(got[ring], b0[ring])
