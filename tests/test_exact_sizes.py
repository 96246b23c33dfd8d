"""CPU half of the exact parity tests at size (exact_ops.size_cases, test_exact_sizes_gpu.py): every case's plan takes
the path it is about, the operators shaped like the shipped stencils generate the presets' own units, each threshold
pair sits one step either side of the generator's size rule, every schedule stays exact, the procedural input is the
same in numpy and torch, and the windowed reference equals exact_run."""
import numpy as np
import pytest

import exact_ops as X

SHAPED = {"c1": "star5", "c1t2": "star5", "c2": "box9", "c3": "box25", "c3t2": "box25", "c4": "star7neg",
          "c4t2": "star7neg", "c5": "star7neg", "c5t2": "star7neg"}


@pytest.mark.parametrize("cid", [c["id"] for c in X.size_cases()])
def test_size_case_plan_and_exactness(built, cid):
    case = X.size_case(cid)
    plan = X.size_plan(case)
    assert plan.stencil.shape == case["shape"]
    assert X.size_markers(case, plan) == [], cid
    ok, why = X.size_growth_ok(case)
    assert ok, (cid, why)
    assert X.literals_exact(plan.source, X.ARITH_MACROS, case["dtype"]) == [], cid
    assert X.literals_exact(plan.pair_source, ("DRS_SCATTER3",), case["dtype"]) == [], cid
    assert plan.info.halo == X.halo_of(X.OPS[case["op"]], X.step_of(case))


@pytest.mark.parametrize("preset", sorted(SHAPED))
def test_shaped_operator_generates_the_preset_unit(built, preset):
    """With the preset's knobs, size and stencil name, the shaped operator's translation units (main and pair) are the
    preset's, literal for literal once the coefficient values are blanked out: same header, DRS_TS, factorisation and
    residual terms, deferred scale, DRS_FLAT / DRS_LD_HINT and tile defines."""
    import drstencil_b200 as drs
    from drstencil_b200.presets import PRESETS
    path, kn = PRESETS[preset]
    ref = drs.Plan(drs.Stencil.from_file(path), kn)
    case = X.size_case(preset)
    assert case["op"] == SHAPED[preset]
    plan = X.size_plan(case)
    assert plan.note == "" and ref.note == ""
    assert X.normalise_literals(plan.source) == X.normalise_literals(ref.source)
    assert X.normalise_literals(plan.pair_source) == X.normalise_literals(ref.pair_source)
    assert plan.info.kernel_name == ref.info.kernel_name


def test_threshold_pairs_flip_the_generator_rules(built):
    """The two shapes of each threshold pair differ by one slow-axis plane / row, and the plan's markers flip there:
    DRS_LD_HINT and the pair unit at 1 GiB per 3D array, DRS_FLAT 1 -> 2 of unaligned rows."""
    cases = {c["id"]: c for c in X.size_cases()}
    for kernel in ("gather3d", "fused3d", "multi3d"):
        off, on = cases["l2-off-" + kernel], cases["l2-on-" + kernel]
        assert on["shape"][0] == off["shape"][0] + 1 and on["shape"][1:] == off["shape"][1:]
        assert not X.far_beyond_l2(off["shape"], "f64") and X.far_beyond_l2(on["shape"], "f64")
        p_off, p_on = X.size_plan(off), X.size_plan(on)
        assert "DRS_LD_HINT" not in p_off.source and "#define DRS_LD_HINT 1" in p_on.source
        assert p_off.pair_source == "" and bool(p_on.pair_source) == (kernel == "gather3d")
    for what in ("2d-gather2d", "2d-temporal2d", "3d-gather3d", "3d-multi3d"):
        f1, f2 = cases["flat1-" + what], cases["flat2-" + what]
        assert f2["shape"][0] == f1["shape"][0] + 1 and f2["shape"][1:] == f1["shape"][1:]
        assert (f1["flat"], f2["flat"]) == (1, 2)
        assert "#define DRS_FLAT 1\n" in X.size_plan(f1).source and "#define DRS_FLAT 2\n" in X.size_plan(f2).source
        assert np.prod(f2["shape"]) < 2 ** 31          # flat 2 by the tile overrun rule, not by the element count
    for cid in ("big-2d-gather2d", "big-2d-temporal2d", "big-3d-gather3d", "big-3d-fused3d",
                "big-3d-unaligned-gather3d", "c5", "c5t2"):
        assert np.prod(cases[cid]["shape"]) > 2 ** 31, cid
    assert cases["big-3d-unaligned-gather3d"]["flat"] == 2


def test_size_case_ids_are_unique():
    ids = [c["id"] for c in X.size_cases()]
    assert len(ids) == len(set(ids))


def test_generator_numpy_equals_torch():
    """The same values from numpy and torch (CPU), windows around the flat index 2^31 included; values in
    -UMAX..UMAX, all of them taken; impulses land where they are listed."""
    import torch
    shape = (1040, 1024, 2048)
    like = torch.empty(0)
    imps = [((1023, 5, 7), 3), ((1024, 0, 0), -3)]
    for lo, hi in ((0, 2), (1022, 1026), (1038, 1040)):
        a = X.gen_input(shape, lo, hi, 11, imps)
        t = X.gen_input(shape, lo, hi, 11, imps, like=like)
        assert a.dtype == np.float64 and t.dtype == torch.float64
        assert np.array_equal(a, t.numpy()), (lo, hi)
        vals = set(np.unique(a).tolist())
        assert set(range(-X.UMAX, X.UMAX + 1)) <= vals <= set(range(-X.UMAX, X.UMAX + 1)) | {-3, 3}
    whole = X.gen_input((6, 7, 9), 0, 6, 3, [])
    assert np.array_equal(np.concatenate([X.gen_input((6, 7, 9), z, z + 1, 3, []) for z in range(6)]), whole)
    assert not np.array_equal(whole, X.gen_input((6, 7, 9), 0, 6, 4, []))
    flat = np.arange(2 ** 31 - 4, 2 ** 31 + 4, dtype=np.int64)
    assert np.array_equal(X.gen_values(flat, 5), X.gen_values(torch.from_numpy(flat), 5).numpy())


def _reference_params():
    """Every (operator, step, sweeps) of the size cases, plus one-sided operators whose slow-axis reach differs below
    and above (r- != r+)."""
    out = {(c["op"], X.step_of(c), c["sweeps"]) for c in X.size_cases()}
    out |= {("onesided", 1, 3), ("onesided", 2, 2), ("kside", 1, 4), ("kside", 2, 3)}
    return sorted(out)


@pytest.mark.parametrize("op,step,sweeps", _reference_params())
def test_window_run_equals_exact_run(op, step, sweeps):
    """window_run over windows that cut the frozen ring at either end, single planes and the whole grid equals the
    matching planes of exact_run, in numpy and in torch."""
    import torch
    o = X.OPS[op]
    H = X.halo_of(o, step)
    shape = (4 * H + 9, 37) if X.op_dim(op) == 2 else (4 * H + 9, 11, 17)
    imps = [((H, 3, 4)[:len(shape)], 3), ((shape[0] - H - 1, 5, 6)[:len(shape)], -3)]
    a0 = X.gen_input(shape, 0, shape[0], 7, imps)
    b0 = np.full(shape, -7.0)
    exA, exB = X.exact_run(o, step, a0, b0, sweeps)
    L = shape[0]
    wins = [(0, 1), (0, H + 1), (H - 1, H + 2), (H, L - H), (L // 2, L // 2 + 1), (L - H - 1, L), (L - 1, L), (0, L)]

    def source_np(s0, s1):
        return X.gen_input(shape, s0, s1, 7, imps), np.full((s1 - s0,) + shape[1:], -7.0)

    def source_torch(s0, s1):
        a = X.gen_input(shape, s0, s1, 7, imps, like=torch.empty(0))
        return a, torch.full_like(a, -7.0)

    rm, rp = X.reach(o)
    for z0, z1 in wins:
        s0, s1 = X.source_window(o, step, sweeps, L, z0, z1)
        assert (s0, s1) == (max(0, z0 - sweeps * step * rm), min(L, z1 + sweeps * step * rp))
        wa, wb = X.window_run(o, step, sweeps, shape, z0, z1, source_np)
        assert np.array_equal(wa, exA[z0:z1]) and np.array_equal(wb, exB[z0:z1]), (z0, z1)
        ta, tb = X.window_run(o, step, sweeps, shape, z0, z1, source_torch)
        assert np.array_equal(ta.numpy(), wa) and np.array_equal(tb.numpy(), wb), (z0, z1)
    # a window one plane too narrow on the side the operator reaches to is wrong somewhere (the margin is tight)
    if rp and sweeps * step * rp < L // 2:
        z0, z1 = L // 2, L // 2 + 1
        s0, s1 = X.source_window(o, step, sweeps, L, z0, z1)

        def short(lo, hi):
            a, b = source_np(lo, hi)
            a[-1] = 0.0
            b[-1] = 0.0
            return a, b
        wa, wb = X.window_run(o, step, sweeps, shape, z0, z1, short)
        assert not (np.array_equal(wa, exA[z0:z1]) and np.array_equal(wb, exB[z0:z1]))


def test_mismatch_report_names_the_place(built):
    case = X.size_case("big-3d-gather3d")
    plan = X.size_plan(case)
    shape, info = case["shape"], plan.info
    msg = X.describe_mismatch((1024, 0, 1), shape, info, 1.0, 2.0)
    assert "(>= 2^31)" in msg and "ring" in msg and "seam" in msg
    msg = X.describe_mismatch((5, 6, info.halo + info.tile_x), shape, info, 1.0, 2.0)
    assert "interior" in msg and "(>= 2^31)" not in msg and "axis 2 seam %d at distance 0" % (info.halo + info.tile_x) in msg
