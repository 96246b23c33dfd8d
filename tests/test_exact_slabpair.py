"""CPU twin of test_exact_slabpair_gpu.py: every GPU case's preconditions without a GPU -- the exactness budget, the
slab pair unit set_slab_pairs generates, the geometry property the case exists for, the reference restated for pairs
against the global one -- plus the refusals of drs_plan_set_slab_pairs, drs_run_slab's split on every rank, the cache
keys of the shipped pair units, and the slab pair units of c4- and c5-shaped middle ranks: NVRTC compile health and SASS
(cuobjdump), and the textual guard that keeps their plane loop the plain pair kernel's."""
import collections
import os
import re
import shutil
import subprocess

import pytest

import exact_ops as X
import exact_slab as S
import exact_slabpair as SP

# drs_run's pair units of the shipped configurations: the slab pair unit lives in its own header and header table,
# so these keys (NVRTC 12.8, the pinned compiler) are those of the parent of the change that added it
PAIR_CACHE_KEYS = {"c4": "a38c2c0103afcffe_12_8", "c5": "12edf83ba8e0a12e_12_8"}

KDIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "drstencil_b200", "csrc", "kernels")


def _define(src, name):
    m = re.search(r"^#define %s\b(.*)$" % name, src, re.M)
    return m.group(1).strip() if m else None


@pytest.mark.parametrize("cid", [c["id"] for c in SP.CASES])
def test_case_preconditions(built, cid):
    case = SP.CASE_BY_ID[cid]
    ok, why = SP.growth_ok(case)
    assert ok, (cid, why)
    gs = SP.geoms(case)
    ranks = range(case["world"]) if case["runner"] == "emulated" else [case["rank"]]
    chunks = {}
    for r in ranks:
        g = gs[r]
        p = SP.make_plan(case, g)
        chunks[r] = p.info.chunk
        H = SP.halo_of(case)
        assert p.halo == H and g.ghost == 2 * H and g.local_planes == g.hi - g.lo + 4 * H, cid
        assert p.info.kernel_name.startswith("dr_") and X.HEADERS["gather3d"] in p.source, cid
        src = p.slab_pair_source
        assert '#include "drs_slabpair3d.cuh"' in src and "#define DRS_SLABPAIR_NAME drslabpair_exact_" in src, cid
        assert p.slab_pair_cache_key and p.slab_pair_cache_key not in (p.cache_key, p.pair_cache_key), cid
        assert p.slab_source == "", cid
        n = case["sweeps"]
        assert p.slab_split(n) == SP.pair_split(n) and SP.pair_split(n)[0] > 0 and p.pair_split(n) == (0, n), cid
    for claim in case["claims"]:
        assert SP.claim_holds(case, claim, chunks), (cid, claim, chunks)


def test_cases_cover_the_ground():
    """Operators for which the depth-2 tile fits, fp64 and fp32, worlds 2-4 with uneven splits, sweep counts 6, 8, 10
    and more (both shapes of the split), every geometry claim; drs_run_slab on the lowest, a middle, the highest and an
    alone rank."""
    em = SP.EMULATED
    assert {c["op"] for c in em} == {"box27", "aniso", "kside", "star7neg", "star7asym", "diag2k"}
    assert {c["dtype"] for c in em} == {"f64", "f32"}
    assert {c["world"] for c in em} == {2, 3, 4}
    assert {6, 8, 10} <= {c["sweeps"] for c in em} and max(c["sweeps"] for c in em) > 10
    assert {SP.pair_split(c["sweeps"])[1] for c in em} == {2, 4}
    assert {"thin", "chunk<ghost", "both-faces", "ring-ghost"} <= {k for c in em for k in c["claims"]}
    for c in em:
        if c["G"] % c["world"]:
            assert len({h - l for l, h in SP.geoms(c)[0].bounds}) > 1
    kinds = {"alone" if c["world"] == 1 else "lowest" if c["rank"] == 0 else
             "highest" if c["rank"] == c["world"] - 1 else "middle" for c in SP.RUN_SLAB}
    assert kinds == {"alone", "lowest", "middle", "highest"}
    assert {SP.pair_split(c["sweeps"])[1] for c in SP.RUN_SLAB} == {2, 4}


@pytest.mark.parametrize("cid", [c["id"] for c in SP.EMULATED])
def test_pair_reference_self_check(built, cid):
    """The reference restated for pairs (schedule_ref), with every rank's ghost planes refreshed from the global
    reference after each launch, equals the global reference cut into the rank's window."""
    case = SP.CASE_BY_ID[cid]
    gs = SP.geoms(case)
    chunks = {g.rank: SP.make_plan(case, g).info.chunk for g in gs}
    assert SP.self_check(case, chunks) == []


def _plan(op, shape, **kn):
    import drstencil_b200 as drs
    return drs.Plan(drs.Stencil.from_points(list(op), list(op.values()), shape, 2, name="sp"), drs.Knobs(**kn))


def test_refusals(built):
    """drs_plan_set_slab_pairs refuses with DRS_E_ARG what has no slab pair launch and a plan that already is a slab;
    drs_plan_slab_schedule refuses pair slabs, drs_sweep_pair a pair slab without peers."""
    import drstencil_b200 as drs
    star = X.OPS["star7neg"]
    G, lo, hi = 40, 13, 27
    L = hi - lo + 4
    # radius 32 along x (and a slow-axis offset of 32, the largest x offset a plan accepts): no depth-2 tile
    wide = {(0, 0, 0): -1 / 2, (0, 0, -32): 1 / 4, (0, 0, 32): 1 / 4, (32, 0, 0): 1 / 8, (-1, 0, 0): -1 / 8}
    # radius 8 along k and y: the plane ring does not fit in shared memory
    deep = {(0, 0, 0): -1 / 2, (-8, 0, 0): 1 / 4, (8, 0, 0): 1 / 4, (0, -8, 0): 1 / 8, (0, 8, 0): 1 / 8}
    cases = [
        ("2D plan", _plan({(0, 0): -1 / 2, (-1, 0): 1 / 4, (1, 0): 1 / 4}, (L, 264)), "3D only"),
        ("step 2", _plan(star, (L + 4, 20, 72), step=2, fuse="temporal"), "step-1"),
        ("sub-step launches", _plan(star, (L + 4, 20, 72), step=2, fuse="temporal", no_fused3d=1), "step-1"),
        ("unaligned pitch", _plan(star, (L, 20, 71)), "row pitch"),
        ("fuse reuse", _plan(star, (L, 20, 72), fuse="reuse"), "reuse"),
        ("naive kernel", _plan(deep, (hi - lo + 32, 40, 72)), "naive kernel"),
        ("tile", _plan(wide, (hi - lo + 128, 70, 200)), "depth-2 tile"),
        ("local size", _plan(star, (L - 2, 20, 72)), "4*Halo"),
    ]
    for what, p, msg in cases:
        with pytest.raises(drs.DrsError) as e:
            p.set_slab_pairs(G, lo, hi)
        assert e.value.code == drs.E_ARG and msg in str(e.value), (what, str(e.value))
        assert p.slab_pair_source == "" and p.slab_pair_cache_key == "", what
    p = _plan(star, (L - 2, 20, 72))
    p.set_slab(G, lo, hi)
    with pytest.raises(drs.DrsError) as e:
        p.set_slab_pairs(G, lo, hi)
    assert e.value.code == drs.E_ARG and "already a slab" in str(e.value)
    p = _plan(star, (L, 20, 72))
    p.set_slab_pairs(G, lo, hi)
    with pytest.raises(drs.DrsError) as e:
        p.set_slab_pairs(G, lo, hi)
    assert e.value.code == drs.E_ARG and "already a slab" in str(e.value)
    with pytest.raises(drs.DrsError) as e:
        p.slab_schedule(6, False)
    assert e.value.code == drs.E_ARG and "pair slab" in str(e.value)
    with pytest.raises(drs.DrsError) as e:
        p.sweep_pair(16, 32)
    assert e.value.code == drs.E_ARG and "set_peers" in str(e.value)


def test_refused_plans_take_their_paths(built):
    """The plans of test_refusals stand for what they are refused for."""
    star = X.OPS["star7neg"]
    deep = {(0, 0, 0): -1 / 2, (-8, 0, 0): 1 / 4, (8, 0, 0): 1 / 4, (0, -8, 0): 1 / 8, (0, 8, 0): 1 / 8}
    assert _plan(deep, (46, 40, 72)).info.kernel_name.startswith("gold_")
    assert "drs_reuse.cuh" in _plan(star, (18, 20, 72), fuse="reuse").source
    assert "drs_sweep3d_t.cuh" in _plan(star, (22, 20, 72), step=2, fuse="temporal").source
    assert "one single-step launch per sub-step" in _plan(star, (22, 20, 72), step=2, fuse="temporal", no_fused3d=1).note
    assert "#define DRS_FLAT 1" in _plan(star, (18, 20, 71)).source


def test_only_pair_slabs_have_the_unit(built):
    """slab_pair_source / slab_pair_cache_key are "" on plain plans, on big plans with drs_run pair launches and on
    slabs of set_slab; slab_split is (0, n) there, and pair_split stays (0, n) on pair slabs."""
    from drstencil_b200.slab import SlabGeometry
    star = X.OPS["star7neg"]
    g1, g2 = SlabGeometry(40, 3, 1, 1), SlabGeometry(40, 3, 1, 2, ring=1)
    plain = _plan(star, (g1.local_planes, 20, 72))
    big = _plan(star, (512, 512, 512))
    slab = _plan(star, (g1.local_planes, 20, 72))
    slab.set_slab(40, g1.lo, g1.hi)
    for p in (plain, big, slab):
        assert p.slab_pair_source == "" and p.slab_pair_cache_key == ""
        assert p.slab_split(10) == (0, 10)
    assert big.pair_split(10) == (4, 2)
    pair = _plan(star, (g2.local_planes, 20, 72))
    pair.set_slab_pairs(40, g2.lo, g2.hi)
    assert pair.slab_split(10) == (4, 2) and pair.pair_split(10) == (0, 10)
    assert [pair.slab_split(n) for n in (2, 4, 6, 8, 10)] == [(0, 2), (0, 4), (2, 2), (2, 4), (4, 2)]


@pytest.mark.parametrize("world", [2, 3, 4])
def test_slab_split_is_the_same_on_every_rank(built, world):
    """Uneven splits; each rank's slab_split equals pair_split of the sweep count whether or not its local arrays are
    >= 1 GiB (the 1 GiB rule of drs_run's pair launches does not apply to pair slabs)."""
    import drstencil_b200 as drs
    from drstencil_b200.slab import SlabGeometry
    star = X.OPS["star7neg"]
    # 1024^2 fp64 planes are 8 MiB: local arrays of 127 and 128 planes sit either side of 1 GiB
    for G, M, N in ((37 * world + 1, 20, 72), (124 * world - 1, 1024, 1024)):
        sizes = set()
        for r in range(world):
            g = SlabGeometry(G, world, r, 2, ring=1)
            p = _plan(star, (g.local_planes, M, N))
            sizes.add(X.far_beyond_l2((g.local_planes, M, N), "f64"))
            p.set_slab_pairs(G, g.lo, g.hi)
            for T in range(0, 41):
                n = drs.sweep_count(T, 1)
                assert p.slab_split(T) == SP.pair_split(n), (world, r, T)
        assert len({h - l for l, h in SlabGeometry(G, world, 0, 2, ring=1).bounds}) > 1
        if M == 1024:
            assert sizes == {True, False}, "the big world has ranks on both sides of 1 GiB"


def test_shipped_pair_units_unchanged(built):
    """c4's and c5's drs_run pair units: the parent's cache keys."""
    import drstencil_b200 as drs
    from drstencil_b200.presets import PRESETS
    for name, key in PAIR_CACHE_KEYS.items():
        path, kn = PRESETS[name]
        plan = drs.Plan(drs.Stencil.from_file(path), kn)
        assert plan.pair_cache_key == key, (name, plan.pair_cache_key)


# ---- the slab pair units of c4- and c5-shaped middle ranks (N = 8) -----------------------------------------------

def _preset_pair_slab(name, world=8, rank=3):
    import drstencil_b200 as drs
    from drstencil_b200.presets import PRESETS
    from drstencil_b200.slab import SlabGeometry
    path, kn = PRESETS[name]
    st = drs.Stencil.from_file(path)
    full = drs.Plan(st, kn)
    G = st.shape[0]
    H = full.halo
    g = SlabGeometry(G, world, rank, 2 * H, ring=H)
    plan = drs.Plan(drs.Stencil.from_file(path).set_size((g.local_planes,) + tuple(st.shape[1:])), kn)
    plan.set_slab_pairs(G, g.lo, g.hi)
    return full, plan


def _cache(key, ext):
    import drstencil_b200 as drs
    return os.path.join(os.path.dirname(drs.__file__), "_jitcache", key + ext)


def _resources(log, fn):
    m = re.search(r"Function properties for %s\n.*?(\d+) bytes spill stores, (\d+) bytes spill loads.*?Used (\d+) "
                  r"registers" % fn, log, re.S)
    assert m, log[:2000]
    return int(m.group(1)) + int(m.group(2)), int(m.group(3))


@pytest.mark.parametrize("name", ["c4", "c5"])
def test_preset_slabpair_unit_compiles_without_spills(built, name):
    full, plan = _preset_pair_slab(name)
    fn = "drslabpair_" + full.info.kernel_name[len("dr_"):]
    spill, regs = _resources(open(_cache(plan.slab_pair_cache_key, ".log")).read(), fn)
    assert spill == 0 and regs <= 128, (name, spill, regs)
    src = plan.slab_pair_source
    assert (_define(src, "DRS_NW"), _define(src, "DRS_MINB")) == ("8", "2"), name
    # the slab pair unit is drs_run's pair unit with another entry point: same macros, same literals
    ref = full.pair_source
    for m in ("DRS_RK", "DRS_RJ", "DRS_E", "DRS_NW", "DRS_ST", "DRS_RY", "DRS_MINB", "DRS_HALO"):
        assert _define(src, m) == _define(ref, m), (name, m)
    # the L2 hint follows the rank's own array size (c4's 100 planes of 768^2 are below 1 GiB, c5's 196 of 1536^2 not)
    assert (_define(src, "DRS_LD_HINT") == "1") == X.far_beyond_l2((plan.info.L, plan.info.M, plan.info.N), "f64"), name
    assert X.literals(src, X.ARITH_MACROS) == X.literals(ref, X.ARITH_MACROS)


def _mnemonics(fn, key):
    sass = subprocess.run(["cuobjdump", "-sass", "-fun", fn, _cache(key, ".cubin")],
                          stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True).stdout
    ops = collections.Counter()
    for line in sass.splitlines():
        m = re.match(r"\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", line)
        if m:
            ops[m.group(1)] += 1
    assert sum(ops.values()) > 200, sass[:400]
    return ops


def _count(ops, prefix):
    return sum(n for k, n in ops.items() if k.startswith(prefix))


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not on PATH")
@pytest.mark.parametrize("name", ["c4", "c5"])
def test_preset_slabpair_unit_sass(built, name):
    """TMA plane loads and 128-bit stores, no local memory.  The per-thread global loads are exactly those of drpair_
    (the ring cells of A and B, the watchdog word) plus the protocol's: the sequence base (slab_wait, slab_arrive: two
    LDG.E.64), the two flag slots (a first read and the spin loop each: four LDG.E.64.STRONG.SYS) and the fault word of
    slab_wait's spin loops (two LDG.E.STRONG.SYS)."""
    full, plan = _preset_pair_slab(name)
    nm = full.info.kernel_name[len("dr_"):]
    ops = _mnemonics("drslabpair_" + nm, plan.slab_pair_cache_key)
    assert _count(ops, "UTMALDG.3D") >= 2
    assert _count(ops, "STG.E.128") >= 3        # own planes and the two pushes
    assert _count(ops, "LDL") == 0 and _count(ops, "STL") == 0
    main = _mnemonics("drpair_" + nm, full.pair_cache_key)
    want = collections.Counter({k: n for k, n in main.items() if k.startswith("LDG")})
    want.update({"LDG.E.64": 2, "LDG.E.64.STRONG.SYS": 4, "LDG.E.STRONG.SYS": 2})
    assert {k: n for k, n in ops.items() if k.startswith("LDG")} == dict(want), (name, ops, main)


def _body(text, sig, start=None, end=None):
    """The text of the braced block after `sig` (or between the markers start / end inside it), comments and
    whitespace dropped, namespace qualifiers removed."""
    i = text.index(sig)
    depth = 0
    for k in range(text.index("{", i), len(text)):
        depth += {"{": 1, "}": -1}.get(text[k], 0)
        if depth == 0:
            block = text[i:k + 1]
            break
    if start is not None:
        block = block[block.index(start):block.index(end, block.index(start))]
    return " ".join(re.sub(r"//[^\n]*", "", block).replace("s3p::", "").replace("s3sp::", "").split())


def test_slabpair_plane_loop_is_the_pair_kernels():
    """drs_slabpair3d.cuh carries a copy of drs_pair3d.cuh's plane loop.  The parts that must stay the same text --
    the level-0 patch, the shuffles and the scatter, the publication of level 1's edge rows, the stage hand-back after
    the iteration's __syncthreads, the phase recursion -- are compared here; what differs is where the ring planes are
    (ring_lo / ring_hi), the peer stores and the step flags."""
    plain = open(os.path.join(KDIR, "pair", "drs_pair3d.cuh")).read()
    slab = open(os.path.join(KDIR, "slabpair", "drs_slabpair3d.cuh")).read()
    parts = [("void patch_level0(", None, None),
             ("bool phases(", None, None),
             ("bool iteration(", "const real* mine =", "// ---- the plane of level 1 completed by this iteration"),
             ("bool iteration(", "// ---- its edge rows are published", "} else if (n >= c.n_first"),
             ("bool iteration(", "// published planes visible to every warp", "return true;")]
    for sig, a, b in parts:
        assert _body(plain, sig, a, b) == _body(slab, sig, a, b), (sig, a)
        assert len(_body(plain, sig, a, b)) > 90, (sig, a)
