"""CPU half of the opt-in exact pair launches on 2D plans (kernels/pair2d/drs_pair2d.cuh, Plan.set_pairs): which plans
get a 2D pair unit and which are refused, that the unit evaluates exactly the single-step chain, that no existing cache
key moves, and the NVRTC cubins of the c1- and c3-shaped units (spills, occupancy, SASS).  test_exact_pairs2d_gpu.py
holds the results bit for bit against the single-sweep loop and the float64 reference."""
import collections
import os
import re
import shutil
import subprocess

import pytest

import drstencil_b200 as drs
import exact_ops as X
from drstencil_b200.presets import PRESETS
from helpers import stc_path

KDIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "drstencil_b200", "csrc", "kernels")

# main units and drs_run pair units of every preset (NVRTC 12.8, the pinned compiler): the keys of the parent of the
# change that added the 2D pair unit, whose header table enters only the 2D pair keys
PARENT_CACHE_KEYS = {  # preset -> [main key, pair key]
    "2d5pt_star": ["e351bd6c31cfcf86_12_8", ""],
    "2d5pt_cross": ["f374a5c08b4b685a_12_8", ""],
    "2d9pt_star": ["39d87ee3af77b0f2_12_8", ""],
    "2d9pt_box": ["87eb910a4c5f4ed3_12_8", ""],
    "2d9pt_cross": ["caa17f2df6b27d3a_12_8", ""],
    "2d25pt_box": ["de93ec3d01299749_12_8", ""],
    "3d7pt_star": ["62de5be265dc493d_12_8", "b84f8ac02d67c2fa_12_8"],
    "3d9pt_cross": ["aca3e94023dd89e1_12_8", "63aaff16dda1bbc0_12_8"],
    "c1": ["eae70d9b3cd6c2bc_12_8", ""],
    "c2": ["641cf9ae69d6c7f9_12_8", ""],
    "c3": ["58acac6a2876ae7f_12_8", ""],
    "c4": ["c894c64fca08059d_12_8", "a38c2c0103afcffe_12_8"],
    "c5": ["04d7f1f09be682e7_12_8", "12edf83ba8e0a12e_12_8"],
    "c4t2": ["8c6ebed1c83eb74b_12_8", ""],
    "c5t2": ["0c47239c26f940dc_12_8", ""],
    "c1t2": ["efe08a5d228469ea_12_8", ""],
    "c3t2": ["88decef99846a493_12_8", ""],
}
PAIR_CACHE_KEYS = {"c4": "a38c2c0103afcffe_12_8", "c5": "12edf83ba8e0a12e_12_8"}

EXACT_2D = ("star5", "box9", "box25", "mixed3x3", "onesided", "star3gap", "unit", "two", "sep121")


def _preset(name):
    path, kn = PRESETS[name]
    return drs.Plan(drs.Stencil.from_file(path), kn)


def _plan_file(name, shape, **kn):
    return drs.Plan(drs.Stencil.from_file(stc_path(name)).set_size(shape), drs.Knobs(**kn))


def _plan_op(op, shape, name="p2", **kn):
    o = X.OPS[op] if isinstance(op, str) else op
    offs = list(o)
    return drs.Plan(drs.Stencil.from_points(offs, [o[k] for k in offs], shape, 2, name=name), drs.Knobs(**kn))


def _qualifying():
    """(label, plan factory) of every plan that must have a 2D pair unit after set_pairs(True)."""
    out = [("c1", lambda: _preset("c1")), ("c3", lambda: _preset("c3"))]
    for name in ("2d5pt_star", "2d9pt_box", "2d25pt_box"):
        for dt in ("f64", "f32"):
            out.append(("%s-%s" % (name, dt), lambda name=name, dt=dt: _plan_file(name, (520, 1032), dtype=dt)))
    for op in EXACT_2D:
        for dt in ("f64", "f32"):
            out.append(("%s-%s" % (op, dt), lambda op=op, dt=dt: _plan_op(op, (300, 520), name="exact_" + op, dtype=dt)))
    return out


QUALIFYING = _qualifying()


@pytest.mark.parametrize("label", [q[0] for q in QUALIFYING])
def test_set_pairs_gives_a_2d_pair_unit(built, label):
    plan = dict(QUALIFYING)[label]()
    assert plan.pair_source == "" and plan.pair_cache_key == ""
    for T in (1, 2, 5, 10, 100):
        assert plan.pair_split(T) == (0, drs.sweep_count(T, 1))
    plan.set_pairs(True)
    src = plan.pair_source
    assert '#include "drs_pair2d.cuh"' in src and "drs_pair3d.cuh" not in src
    assert "#define DRS_PAIR_NAME drpair_" in src and "#define DRS_TS 2\n" in src
    assert "#define DRS_HALO %d\n" % plan.info.halo in src
    assert plan.pair_cache_key and plan.pair_cache_key != plan.cache_key
    for T in range(0, 41):
        n = drs.sweep_count(T, 1)
        assert plan.pair_split(T) == X_pair_split(n), (label, T)
    plan.set_pairs(True)                 # idempotent
    assert plan.pair_source == src
    plan.set_pairs(False)
    assert plan.pair_source == "" and plan.pair_cache_key == "" and plan.pair_split(10) == (0, 10)


def X_pair_split(n):
    """generate.hpp: pair_split -- p pairs (p even), then 2 or 4 single sweeps."""
    s = n if n < 2 else (2 if ((n - 2) // 2) % 2 == 0 else 4)
    s = min(s, n)
    return (n - s) // 2, s


def test_refusals(built):
    """drs_plan_set_pairs refuses, with DRS_E_ARG and the reason, every 2D plan that has no pair kernel, and slab plans;
    the refused plan keeps no pair unit."""
    star = X.OPS["star5"]
    # radius 9 along x (and a slow-axis offset of 9, the largest x offset a plan accepts): E = 9 > 8 columns per lane
    wide = {(0, 0): -1 / 2, (0, -9): 1 / 4, (0, 9): 1 / 4, (9, 0): 1 / 8, (-1, 0): -1 / 8}
    slab = _plan_op(star, (42, 264))
    slab.set_slab(40, 0, 40)
    cases = [
        ("c2 (step 4)", _preset("c2"), "step-1"),
        ("fuse reuse", _plan_op(star, (300, 264), fuse="reuse"), "reuse"),
        ("unaligned pitch", _plan_op(star, (300, 263)), "row pitch"),
        ("naive kernel", _plan_op(star, (300, 264), rows_per_stage=256), "naive kernel"),
        ("slab", slab, "drs_plan_set_slab_pairs"),
        ("too wide", _plan_op(wide, (300, 520)), "x extent"),
        ("too wide f32", _plan_op({(0, 0): -1 / 2, (0, -5): 1 / 4, (0, 5): 1 / 4, (5, 0): 1 / 8, (-1, 0): -1 / 8},
                                  (300, 520), dtype="f32"), "x extent"),
    ]
    for what, p, msg in cases:
        with pytest.raises(drs.DrsError) as e:
            p.set_pairs(True)
        assert e.value.code == drs.E_ARG and msg in str(e.value), (what, str(e.value))
        assert p.pair_source == "" and p.pair_cache_key == "" and p.pair_split(10)[0] == 0, what


def test_refused_plans_take_their_paths(built):
    """The plans of test_refusals stand for what they are refused for."""
    star = X.OPS["star5"]
    assert _preset("c2").info.step == 4
    assert "drs_reuse.cuh" in _plan_op(star, (300, 264), fuse="reuse").source
    assert "#define DRS_FLAT 1" in _plan_op(star, (300, 263)).source
    assert _plan_op(star, (300, 264), rows_per_stage=256).info.kernel_name.startswith("gold_")
    wide = {(0, 0): -1 / 2, (0, -9): 1 / 4, (0, 9): 1 / 4, (9, 0): 1 / 8, (-1, 0): -1 / 8}
    p = _plan_op(wide, (300, 520))
    assert p.info.kernel_name.startswith("dr_") and "#define DRS_E 9\n" in p.source


def test_3d_plan_below_1gib_pairs_on_request(built):
    """A 3D step-1 plan below 1 GiB gets the existing 3D pair unit (the 1 GiB rule dropped); set_pairs(False) restores
    the rule.  On a plan that already pairs, set_pairs(True) changes nothing."""
    small = _plan_file("3d7pt_star", (64, 64, 128))
    assert small.pair_source == ""
    small.set_pairs(True)
    assert '#include "drs_pair3d.cuh"' in small.pair_source and small.pair_split(10) == (4, 2)
    small.set_pairs(False)
    assert small.pair_source == "" and small.pair_split(10) == (0, 10)
    c5 = _preset("c5")
    key = c5.pair_cache_key
    c5.set_pairs(True)
    assert c5.pair_cache_key == key
    c5.set_pairs(False)
    assert c5.pair_cache_key == key and c5.pair_split(100) == (48, 4)
    with pytest.raises(drs.DrsError) as e:
        _preset("c4t2").set_pairs(True)
    assert e.value.code == drs.E_ARG and "step-1" in str(e.value)


# ---- the exact scatter ---------------------------------------------------------------------------------------------

def _chain(src):
    body = src.split("#define DRS_CHAIN(MUL, FMA)", 1)[1].split("\n#define", 1)[0]
    return [(op, (int(b), int(c)), lit)
            for op, a, b, c, lit in re.findall(r"(MUL|FMA)\((-?\d+), (-?\d+), (-?\d+), ([^)]+)\)", body)]


def _scatter_order(src):
    """Per output, the operations the exact 2D scatter applies, in row-arrival order: [(MUL|FMA, (dj, di), literal)],
    for an output whose slots all start empty (each output's first statement must assign)."""
    body = src.split("#define DRS_SCATTER(P, U)", 1)[1].split("\n#", 1)[0]
    ops, carry, assigned = [], None, set()
    lit = r"\(real\)\(([^)]+)\)"
    u = r"U\((-?\d+)\)"
    for stmt in [s.strip(" \\\n") for s in body.split(";") if s.strip(" \\\n")]:
        m = re.fullmatch(r"P\((-?\d+)\) = (.*)", stmt)
        assert m, stmt
        dj, rhs = int(m.group(1)), m.group(2)
        if re.fullmatch(u, rhs):
            assert not assigned
            carry = (dj, int(re.fullmatch(u, rhs).group(1)))
        elif re.fullmatch(r"rmul\(%s, %s\)" % (u, lit), rhs):
            assert not assigned
            di, c = re.fullmatch(r"rmul\(%s, %s\)" % (u, lit), rhs).groups()
            ops.append(("MUL", (dj, int(di)), c))
        elif re.fullmatch(r"rfma\(P\(%d\), %s, rmul\(%s, %s\)\)" % (dj, lit, u, lit), rhs):
            c0, di, c1 = re.fullmatch(r"rfma\(P\(%d\), %s, rmul\(%s, %s\)\)" % (dj, lit, u, lit), rhs).groups()
            assert carry is not None and carry[0] < dj and not assigned
            ops += [("MUL", (dj, int(di)), c1), ("FMA", carry, c0)]
        elif re.fullmatch(r"rfma\(%s, %s, rmul\(%s, %s\)\)" % (u, lit, u, lit), rhs):
            assert not assigned
            di0, c0, di, c1 = re.fullmatch(r"rfma\(%s, %s, rmul\(%s, %s\)\)" % (u, lit, u, lit), rhs).groups()
            ops += [("MUL", (dj, int(di)), c1), ("FMA", (dj, int(di0)), c0)]
        else:
            m = re.fullmatch(r"rfma\(%s, %s, P\(%d\)\)" % (u, lit, dj), rhs)
            assert m and ops, stmt
            ops.append(("FMA", (dj, int(m.group(1))), m.group(2)))
        if ops:
            assigned.add(dj)
    return ops


@pytest.mark.parametrize("label", [q[0] for q in QUALIFYING])
def test_pair_unit_evaluates_the_single_step_chain(built, label):
    """No deferred scale, no row factorisation, no radd, and per output exactly DRS_CHAIN: same terms, same order, same
    literal text."""
    plan = dict(QUALIFYING)[label]()
    plan.set_pairs(True)
    src = plan.pair_source
    for banned in ("DRS_OUT_SCALE", "DRS_FACTORED", "DRS_HROW", "radd"):
        assert banned not in src, (label, banned)
    chain = _chain(plan.source)
    assert len(chain) == plan.info.npoints
    assert _scatter_order(src) == chain


# ---- cache keys ----------------------------------------------------------------------------------------------------

def test_existing_cache_keys_unchanged(built):
    """Every preset's main unit and c4's and c5's pair units keep their keys; a 2D pair key is none of them."""
    pinned = PARENT_CACHE_KEYS
    assert set(pinned) == set(PRESETS)
    for name in PRESETS:
        p = _preset(name)
        assert [p.cache_key, p.pair_cache_key] == pinned[name], name
    for name, key in PAIR_CACHE_KEYS.items():
        assert pinned[name][1] == key
    keys = {k for v in pinned.values() for k in v if k}
    for name in ("c1", "c3"):
        p = _preset(name)
        p.set_pairs(True)
        assert p.pair_cache_key not in keys


# ---- the c1- and c3-shaped units: NVRTC compile health and SASS ----------------------------------------------------

def _cache(key, ext):
    return os.path.join(os.path.dirname(drs.__file__), "_jitcache", key + ext)


def _resources(log, fn):
    m = re.search(r"Function properties for %s\n.*?(\d+) bytes spill stores, (\d+) bytes spill loads.*?Used (\d+) "
                  r"registers" % fn, log, re.S)
    assert m, log[:2000]
    return int(m.group(1)) + int(m.group(2)), int(m.group(3))


def _define(src, name):
    m = re.search(r"^#define %s\b(.*)$" % name, src, re.M)
    return m.group(1).strip() if m else None


def _paired(name):
    p = _preset(name)
    p.set_pairs(True)
    return p, "drpair_" + p.info.kernel_name[len("dr_"):]


@pytest.mark.parametrize("name", ["c1", "c3"])
def test_preset_pair2d_unit_compiles_without_spills(built, name):
    """No spills, and the registers allow the planned occupancy: DRS_MINB CTAs of DRS_NW warps per SM.  The geometry is
    choose_spec's at step 2 (the c1t2 / c3t2 shapes) with the ring of one step."""
    p, fn = _paired(name)
    src = p.pair_source
    spill, regs = _resources(open(_cache(p.pair_cache_key, ".log")).read(), fn)
    nw, minb = int(_define(src, "DRS_NW")), int(_define(src, "DRS_MINB"))
    assert spill == 0 and regs * nw * 32 * minb <= 65536, (name, spill, regs, nw, minb)
    t2 = _preset(name + "t2").source
    for m in ("DRS_NW", "DRS_ST", "DRS_RB", "DRS_VT", "DRS_RJ", "DRS_E"):
        assert _define(src, m) == _define(t2, m), (name, m)
    assert int(_define(src, "DRS_HALO")) * 2 == int(_define(t2, "DRS_HALO"))


def _mnemonics(fn, key):
    sass = subprocess.run(["cuobjdump", "-sass", "-fun", fn, _cache(key, ".cubin")],
                          stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True).stdout
    ops = collections.Counter()
    for line in sass.splitlines():
        m = re.match(r"\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\w+\s+)?([A-Z0-9_.]+)", line)
        if m:
            ops[m.group(1)] += 1
    assert sum(ops.values()) > 200, sass[:400]
    return ops


def _count(ops, prefix):
    return sum(n for k, n in ops.items() if k.startswith(prefix))


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not on PATH")
@pytest.mark.parametrize("name,mul,fma,other", [("c1", "DMUL", "DFMA", ("FMUL", "FFMA")), ("c3", "FMUL", "FFMA", ("DMUL", "DFMA"))])
def test_preset_pair2d_unit_sass(built, name, mul, fma, other):
    """TMA row loads, no local memory, floating-point arithmetic only multiplies and fused multiply-adds of the dtype
    (no adds: no row factorisation, no radd), one MUL per output and level (the chain's first term), and global loads
    that are the ring-patch loads (read-only, one width: the dtype's) plus the pipeline watchdog's fault word."""
    p, fn = _paired(name)
    ops = _mnemonics(fn, p.pair_cache_key)
    assert _count(ops, "UTMALDG.2D") >= 1
    assert _count(ops, "LDL") == 0 and _count(ops, "STL") == 0
    assert _count(ops, "DADD") == 0 and _count(ops, "FADD") == 0
    for o in other:
        assert _count(ops, o) == 0, (name, o)
    R2 = 2 * int(_define(p.pair_source, "DRS_RJ")) + 1
    C = int(_define(p.pair_source, "DRS_VT")) * (2 if mul == "DMUL" else 4)
    npts = p.info.npoints
    # the row loop is unrolled by R2 phases; each phase runs two levels of C outputs
    assert ops[mul] == R2 * 2 * C and ops[fma] == R2 * 2 * C * (npts - 1), (name, ops[mul], ops[fma])
    loads = {k: n for k, n in ops.items() if k.startswith("LDG")}
    ring = "LDG.E.64.CONSTANT" if mul == "DMUL" else "LDG.E.CONSTANT"     # read-only (ld.global.nc): rings are never written
    assert set(loads) == {ring, "LDG.E.STRONG.SYS"}, (name, loads)
    main = _mnemonics(p.info.kernel_name, p.cache_key)
    assert "LDG.E.STRONG.SYS" in main and ring not in main


# ---- textual guard: the copied parts of drs_sweep2d.cuh --------------------------------------------------------------

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
        block = block[block.index(start):block.index(end, block.index(start)) + len(end)]
    return " ".join(re.sub(r"//[^\n]*", "", block).replace("s2d::", "").split())


def test_pair2d_copies_of_the_sweep2d_row_loop():
    """drs_pair2d.cuh copies drs_sweep2d.cuh's stage handling (the wait of a stage's first row, the hand-back after its
    last row), the level-2 shuffles, the level-2 store's guard and the tile setup of sweep(); those parts must stay
    the same text."""
    plain = open(os.path.join(KDIR, "drs_sweep2d.cuh")).read()
    pair = open(os.path.join(KDIR, "pair2d", "drs_pair2d.cuh")).read()
    parts = [("bool iteration(", "const int rr =", "(drs_u32)((c / ST) & 1), st.fault)) return false;"),
             ("bool iteration(", "if (rr == RB - 1) {", "return true;"),
             ("void row_step(", "const real (&src)[", "__shfl_down_sync(0xffffffffu, src[e], 1);"),
             ("void sweep(", "extern __shared__", "st.N = p.N;"),
             ("void sweep(", "const int X0 =", "st.NCH = (st.NIT + RB - 1) / RB;"),
             ("void sweep(", "Tile t;", "t.out = p.out;"),
             ("void sweep(", "#pragma unroll 1", "return;")]
    for sig, a, b in parts:
        x, y = _body(plain, sig, a, b), _body(pair, sig, a, b)
        # the pair kernel has no unaligned-pitch forms (DRS_FLAT == 0) and one level feeding the next
        x = x.replace("#if DRS_FLAT == 2 if (c + ST < st.NCH) st.issue(c + ST); #else ", "").replace(" #endif", "")
        x = x.replace("DRS_FLAT == 2 ? 32 : 1", "1")
        x = x.replace("const real (&src)[SW]", "const real (&src)[C]").replace("w[s >= 2 ? s - 2 : 0]", "w[0]")
        y = y.replace("phases<0>(w, rb, st, t, g, n0)", "phases<0>(w, st, t, n0)")
        assert x == y, (sig, a, x, y)
        assert len(x) > 60, (sig, a)


def test_cli_run_pairs_refusal(built, tmp_path):
    """`drstencil --run --pairs` on a plan with no pair kernel prints the library's reason and exits non-zero before it
    touches a GPU."""
    from helpers import ROOT
    cli = os.path.join(ROOT, "drstencil_b200", "bin", "drstencil")
    r = subprocess.run([cli, "--run", "--pairs", "--step", "4", stc_path("2d5pt_star")], cwd=tmp_path,
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode != 0 and "step-1" in r.stdout, (r.returncode, r.stdout)
