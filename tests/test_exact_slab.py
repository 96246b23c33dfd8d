"""CPU twin of test_exact_slab_gpu.py: every GPU case's preconditions without a GPU -- the exactness budget, the
kernel path (header, DRS_FLAT, DRS_TS, the drslab_ entry), the geometry property the case exists for (restating
fill_params' face counting), the host schedule's flag bits, pair_split on slab plans, and the frozen-ghost reference
itself against the global one."""
import numpy as np
import pytest

import exact_ops as X
import exact_slab as S


def _plans(case, monkeypatch):
    X.set_env(case, monkeypatch)
    gs = S.geoms(case)
    ranks = range(case["world"]) if case["runner"] == "emulated" else [case["rank"]]
    return gs, [(gs[r], S.make_plan(case, gs[r])) for r in ranks]


@pytest.mark.parametrize("cid", [c["id"] for c in S.CASES])
def test_case_preconditions(built, cid, monkeypatch):
    case = S.CASE_BY_ID[cid]
    ok, why = S.growth_ok(case)
    assert ok, (cid, why)
    gs, plans = _plans(case, monkeypatch)
    chunks = {g.rank: p.info.chunk for g, p in plans}
    for g, p in plans:
        assert p.halo == S.ghost_of(case) == g.ghost, cid
        assert X.markers(case, p, S.local_shape(case, g), bool(case["env"])) == [], cid
        assert "#define DRS_SLAB_NAME drslab_" in p.source, cid
    for claim in case["claims"]:
        assert S.claim_holds(case, claim, chunks), (cid, claim, [S.faces(gs[r], c) for r, c in chunks.items()])
    if case["runner"] != "emulated":
        g = gs[case["rank"]]
        assert [g.lower is not None, g.upper is not None] == [case["rank"] > 0, case["rank"] < case["world"] - 1]


def test_ranks_covered():
    """drs_run_slab: the lowest, a middle, the highest and an alone rank; drs_run_host_slab: both skews."""
    kinds = set()
    for c in S.RUN_SLAB:
        kinds.add("alone" if c["world"] == 1 else "lowest" if c["rank"] == 0 else
                  "highest" if c["rank"] == c["world"] - 1 else "middle")
    assert kinds == {"alone", "lowest", "middle", "highest"}
    assert {c["blocks"][1] for c in S.HOST_SLAB} == {0, 1}
    assert {c["path"] for c in S.EMULATED} == {"gather3d", "cta3d", "fused3d"}
    assert {S.step_of(c) for c in S.EMULATED if c["path"] == "fused3d"} == {2, 3, 4}
    assert {c["world"] for c in S.EMULATED} == {2, 3, 4}
    assert {"thin", "chunk<ghost", "both-faces", "ring-ghost"} <= {k for c in S.EMULATED for k in c["claims"]}
    assert all(c["sweeps"] >= 4 for c in S.EMULATED)
    for c in S.EMULATED:
        sizes = [h - l for l, h in S.geoms(c)[0].bounds]
        if c["world"] > 1 and c["G"] % c["world"]:
            assert len(set(sizes)) > 1


@pytest.mark.parametrize("cid", [c["id"] for c in S.HOST_SLAB])
def test_host_schedule_flags(built, cid):
    """The step list is non-empty and has wait, signal and init bits exactly on the sides that have neighbours."""
    case = S.CASE_BY_ID[cid]
    g = S.geoms(case)[case["rank"]]
    plan = S.make_plan(case, g)
    units, up_skew = case["blocks"]
    plan.set_host_block(units)
    recs = plan.slab_schedule(case["calls"] * S.step_of(case), bool(up_skew))
    assert recs, cid
    bits = 0
    for r in recs:
        bits |= r[5]
    for has, side in ((g.lower is not None, (1, 4, 16)), (g.upper is not None, (2, 8, 32))):
        for b in side:
            assert bool(bits & b) == has, (cid, b, bits)
    assert bits & ~63 == 0


@pytest.mark.parametrize("cid", [c["id"] for c in S.RUN])
def test_pair_split_on_slab_plans(built, cid):
    """drs_run on a slab plan runs single sweeps only, also where the plain plan of that size has pair launches."""
    case = S.CASE_BY_ID[cid]
    g = S.geoms(case)[case["rank"]]
    plan = S.make_plan(case, g)
    T = case["sweeps"] * S.step_of(case)
    assert plan.pair_split(T) == (0, case["sweeps"])
    big = X.far_beyond_l2(S.local_shape(case, g), case["dtype"])
    assert bool(plan.pair_source) == big, cid          # the plan has a pair unit exactly when its size qualifies
    if big:
        import drstencil_b200 as drs
        op = X.OPS[case["op"]]
        offs = list(op)
        st = drs.Stencil.from_points(offs, [op[o] for o in offs], S.local_shape(case, g), T, name="exact_" + case["op"])
        plain = drs.Plan(st, drs.Knobs(**case["knobs"]))
        assert plain.pair_split(T)[0] > 0, "the same plan without set_slab has pair launches"


@pytest.mark.parametrize("name", sorted(S.PRESET_SLABS))
def test_preset_slab_plan(built, name):
    """The middle rank of the N = 8 slab of c5 / c5t2 runs the preset's kernel with the L2 hint and a drslab_ entry;
    its arrays are >= 1 GiB, and the exactness budget covers both calls."""
    import drstencil_b200 as drs
    from drstencil_b200.presets import PRESETS
    from drstencil_b200.slab import SlabGeometry
    spec = S.PRESET_SLABS[name]
    shape = X._stc_shape(PRESETS[spec["preset"]][0])
    stname, kn = X._preset_stencil(spec["preset"])
    op, step = X.OPS["star7neg"], kn.values["step"]
    H = X.halo_of(op, step)
    g = SlabGeometry(shape[0], spec["world"], spec["rank"], H)
    lshape = (g.local_planes,) + shape[1:]
    assert g.hi - g.lo == shape[0] // spec["world"] and g.lower is not None and g.upper is not None
    offs = list(op)
    plan = drs.Plan(drs.Stencil.from_points(offs, [op[o] for o in offs], lshape, 2 * step, name=stname), kn)
    plan.set_slab(shape[0], g.lo, g.hi)
    src = plan.source
    assert plan.halo == H
    assert "#define DRS_SLAB_NAME drslab_" in src and "#define DRS_LD_HINT 1" in src
    assert X.HEADERS[spec["path"]] in src and ("drs_sweep3d_cta.cuh" in src) == (spec["path"] == "cta3d")
    assert "#define DRS_TS %d\n" % (step if spec["path"] == "fused3d" else 1) in src
    assert X.far_beyond_l2(lshape, "f64")
    n = spec["sweeps_per_call"]
    assert plan.pair_split(n * step) == (0, n)
    assert X.growth_ok(dict(op="star7neg", dtype="f64", knobs=dict(step=step), sweeps=2 * n), np.array([X.IMPULSE]))[0]


@pytest.mark.parametrize("cid", [c["id"] for c in S.EMULATED])
def test_frozen_reference_self_check(built, cid, monkeypatch):
    """The frozen-ghost reference with every rank's ghost planes refreshed from the global reference after each
    sweep equals the global reference cut into the rank's window."""
    case = S.CASE_BY_ID[cid]
    _, plans = _plans(case, monkeypatch)
    assert S.self_check(case, {g.rank: p.info.chunk for g, p in plans}) == []


def test_faces_restatement():
    """faces() on hand-checked geometries: a middle rank of 3 planes with Halo 1 and chunks of 2 has one chunk per
    face; with one chunk for the whole slab, that chunk is on both faces and counted once in the prefix."""
    from drstencil_b200.slab import SlabGeometry
    g = SlabGeometry(12, 4, 1, 1)           # planes [3, 6), local 5, outputs [1, 4), faces end 2 / begin 3
    assert (g.out_lo, g.out_hi, g.local_planes) == (1, 4, 5)
    assert S.faces(g, 2) == dict(nzs=2, nlo=1, nhi=1, face_lo_chunks=1, face_hi_chunks=1, both=False)
    assert S.faces(g, 16) == dict(nzs=1, nlo=1, nhi=1, face_lo_chunks=1, face_hi_chunks=0, both=True)
    g0 = SlabGeometry(12, 4, 0, 1)          # no lower neighbour: no lower-face chunks
    assert S.faces(g0, 1)["nlo"] == 0 and S.faces(g0, 1)["nhi"] == 1
