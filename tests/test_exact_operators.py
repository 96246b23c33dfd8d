"""CPU half of the exact-arithmetic parity suite (exact_ops.py): the reference is cross-checked against the oracle's C
sweep, and every case of test_exact_operators_gpu.py is planned here (NVRTC needs no GPU), so that its exactness
preconditions and the markers of the kernel path it means to test are known to hold before a GPU sees it."""
import numpy as np
import pytest

import exact_ops as X


def _oracle_terms(op):
    offs = np.array(X._offsets3(op), dtype=np.int32)
    order = np.lexsort(offs.T[::-1])
    return offs[order], np.array(list(op.values()))[order]


@pytest.mark.parametrize("op", sorted(X.OPS))
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_exact_reference_equals_the_oracle_sweep(built, op, dtype):
    """On exact inputs the numpy reference (float64, any summation order) and the oracle's gold chain (the reference's
    contracted order, in the dtype) must agree bit for bit, ring included, over a ping-pong pair of sweeps."""
    from oracle import oracle
    o = X.OPS[op]
    shape = (23, 37) if X.op_dim(op) == 2 else (13, 11, 17)
    rng = np.random.default_rng(3)
    a0 = rng.integers(-X.UMAX, X.UMAX + 1, size=shape).astype(dtype)
    b0 = np.full(shape, -7, dtype)
    offs, coefs = _oracle_terms(o)
    H = X.halo_of(o, 1)
    refA, refB = a0.copy(), b0.copy()
    oracle.sweep(refA, refB, offs, coefs, H)
    oracle.sweep(refB, refA, offs, coefs, H)
    exA, exB = X.exact_run(o, 1, a0, b0, 2)
    assert np.array_equal(exB, refB) and np.array_equal(exA, refA)
    # and the composed operator of the oracle (step 2, exact dyadic products) equals two levels of the reference
    comp = oracle.compose({((0,) + k) if len(k) == 2 else k: c for k, c in o.items()}, 2)
    keys = sorted(comp)
    ra, rb = a0.astype(np.float64), b0.astype(np.float64)
    oracle.sweep(ra, rb, np.array(keys, np.int32), np.array([comp[k] for k in keys]), X.halo_of(o, 2))
    _, exB2 = X.exact_run(o, 2, a0, b0, 1)
    assert np.array_equal(exB2, rb)


def test_reference_is_sensitive():
    """A coefficient off by one ulp of fp32, and a neighbour moved by one column, change the exact answer."""
    o = X.OPS["mixed3x3"]
    a = np.random.default_rng(1).integers(-2, 3, size=(20, 30)).astype(np.float64)
    base = X.apply_levels(a, o, 2)[X.interior(a.shape, 2)]
    o2 = dict(o)
    o2[(0, 1)] = float(np.nextafter(np.float32(o[(0, 1)]), np.float32(1)))
    assert not np.array_equal(X.apply_levels(a, o2, 2)[X.interior(a.shape, 2)], base)
    o3 = dict(o)
    o3[(0, 0)], o3[(0, -1)] = o[(0, -1)], o[(0, 0)]
    assert not np.array_equal(X.apply_levels(a, o3, 2)[X.interior(a.shape, 2)], base)


@pytest.mark.parametrize("cid", [c["id"] for c in X.CASES])
def test_case_preconditions_and_path_markers(built, cid, monkeypatch):
    """For every shape of every GPU case: (a) the values stay exact over the whole schedule, (b) every literal the
    kernel multiplies by is an exact short dyadic, (c) the plan really takes the kernel path the case is about."""
    case = X.CASE_BY_ID[cid]
    X.set_env(case, monkeypatch)
    shapes = X.shapes(case)
    assert len(shapes) >= 3
    for shape in shapes:
        plan = X.make_plan(case, shape)
        info = plan.info
        u = X.make_input(case, shape, info, 0)
        ok, why = X.growth_ok(case, u)
        assert ok, (cid, shape, why)
        assert X.literals_exact(plan.source, X.arith_names(case), case["dtype"]) == [], (cid, shape)
        assert X.markers(case, plan, shape, bool(case["env"])) == [], (cid, shape)
        assert info.halo == X.halo_of(X.OPS[case["op"]], X.step_of(case))


@pytest.mark.parametrize("name", sorted(X.RANGE_OPS))
def test_no_deferred_scale_outside_the_dtype_range(built, name):
    """A leading coefficient of 1e-10 / 1e-7 / 1e-100 at depth 4 / 6 / 4 would make eta^ts 1e-40 / 1e-42 (fp32
    subnormals) / 1e-400 (0 in fp64): such operators are evaluated unscaled, on the same temporal path."""
    _, shape, _, step, factored = X.RANGE_OPS[name]
    src = X.range_plan(name).source
    assert "#define DRS_TS %d\n" % step in src and ("#define DRS_FACTORED 1" in src) == factored
    assert "DRS_OUT_SCALE" not in src


# fnv1a of the generated translation unit of every preset (the part of Plan.cache_key before the NVRTC version): the
# workloads bench.py times compile to exactly this code.  A deliberate change of the generated code updates the table.
PRESET_SOURCE_HASHES = {
    "2d5pt_star": "e351bd6c31cfcf86", "2d5pt_cross": "f374a5c08b4b685a", "2d9pt_star": "39d87ee3af77b0f2",
    "2d9pt_box": "87eb910a4c5f4ed3", "2d9pt_cross": "caa17f2df6b27d3a", "2d25pt_box": "de93ec3d01299749",
    "3d7pt_star": "62de5be265dc493d", "3d9pt_cross": "aca3e94023dd89e1",
    "c1": "eae70d9b3cd6c2bc", "c2": "641cf9ae69d6c7f9", "c3": "58acac6a2876ae7f", "c4": "c894c64fca08059d",
    "c5": "04d7f1f09be682e7", "c4t2": "8c6ebed1c83eb74b", "c5t2": "0c47239c26f940dc", "c1t2": "efe08a5d228469ea",
    "c3t2": "88decef99846a493",
}


def test_presets_keep_their_deferred_scale_and_their_code(built):
    import drstencil_b200 as drs
    from drstencil_b200.presets import PRESETS
    assert set(PRESETS) == set(PRESET_SOURCE_HASHES)
    for name, (path, kn) in PRESETS.items():
        plan = drs.Plan(drs.Stencil.from_file(path), kn)
        assert ("#define DRS_OUT_SCALE" in plan.source) == (name in ("c2", "c1t2", "c3t2", "c4t2", "c5t2")), name
        assert plan.cache_key.split("_")[0] == PRESET_SOURCE_HASHES[name], name
