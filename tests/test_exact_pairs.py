"""CPU half of the exact pair launches (kernels/pair/drs_pair3d.cuh): which plans get a pair unit, that the unit
evaluates exactly the single-step chain, and how drs_run splits its sweeps.  test_exact_pairs_gpu.py holds the
results bit for bit against the single-sweep loop."""
import re

import pytest

import drstencil_b200 as drs
from drstencil_b200.presets import PRESETS
from helpers import stc_path

GIB = 1 << 30


def _plan(name, shape=None, **kn):
    st = drs.Stencil.from_file(stc_path(name) if "/" not in name else name)
    if shape is not None:
        st.set_size(shape)
    return drs.Plan(st, drs.Knobs(**kn))


def _preset(name):
    path, kn = PRESETS[name]
    return drs.Plan(drs.Stencil.from_file(path), kn)


def test_pair_unit_exactly_for_qualifying_plans(built, monkeypatch):
    assert _preset("c5").pair_source and _preset("c4").pair_source
    for name in ("c4t2", "c5t2", "c1", "c2", "c3"):
        assert _preset(name).pair_source == "", name
    # >= 1 GiB per array, and not one element less (fp64: 2^27 elements, fp32: 2^28)
    assert _plan("3d7pt_star", (512, 512, 512)).pair_source
    assert _plan("3d7pt_star", (510, 512, 512)).pair_source == ""
    assert _plan("3d7pt_star", (512, 512, 1024), dtype="f32").pair_source
    assert _plan("3d7pt_star", (512, 512, 512), dtype="f32").pair_source == ""
    # row pitch not a multiple of 16 bytes, step 2, data-reuse mode, 2D
    assert _plan("3d7pt_star", (520, 512, 513)).pair_source == ""
    assert _plan("3d7pt_star", (512, 512, 512), step=2).pair_source == ""
    assert _plan("3d7pt_star", (512, 512, 512), fuse="reuse").pair_source == ""
    assert _plan("2d5pt_star", (16384, 16384)).pair_source == ""
    # the size rule does not depend on the L2 policy switch
    monkeypatch.setenv("DRS_NO_LD_HINT", "1")
    assert _plan("3d7pt_star", (512, 512, 512)).pair_source


def test_main_unit_is_untouched_by_the_pair_unit(built):
    for name in ("c4", "c5"):
        p = _preset(name)
        assert "drs_pair3d.cuh" not in p.source and "drs_sweep3d_t.cuh" not in p.source
        assert '#include "drs_pair3d.cuh"' in p.pair_source and "drs_sweep3d" not in p.pair_source
        assert p.pair_cache_key and p.pair_cache_key != p.cache_key


def _chain(src):
    body = src.split("#define DRS_CHAIN(MUL, FMA)", 1)[1].split("\n#define", 1)[0]
    return [(op, (int(a), int(b), int(c)), lit)
            for op, a, b, c, lit in re.findall(r"(MUL|FMA)\((-?\d+), (-?\d+), (-?\d+), ([^)]+)\)", body)]


def _scatter_order(src):
    """Per output, the operations the exact scatter applies, in plane-arrival order: [(MUL|FMA, (dk, dj, di), literal)]."""
    body = src.split("#define DRS_SCATTER3(P, U)", 1)[1].split("\n#", 1)[0]
    ops, carry = [], None
    lit = r"\(real\)\(([^)]+)\)"
    u = r"U\((-?\d+), (-?\d+)\)"
    for stmt in [s.strip(" \\\n") for s in body.split(";") if s.strip(" \\\n")]:
        m = re.fullmatch(r"P\((-?\d+)\) = (.*)", stmt)
        assert m, stmt
        dk, rhs = int(m.group(1)), m.group(2)
        if re.fullmatch(u, rhs):
            dj, di = map(int, re.fullmatch(u, rhs).groups())
            carry = (dk, dj, di)
        elif re.fullmatch(r"rmul\(%s, %s\)" % (u, lit), rhs):
            dj, di, c = re.fullmatch(r"rmul\(%s, %s\)" % (u, lit), rhs).groups()
            ops.append(("MUL", (dk, int(dj), int(di)), c))
        elif re.fullmatch(r"rfma\(P\(%d\), %s, rmul\(%s, %s\)\)" % (dk, lit, u, lit), rhs):
            c0, dj, di, c1 = re.fullmatch(r"rfma\(P\(%d\), %s, rmul\(%s, %s\)\)" % (dk, lit, u, lit), rhs).groups()
            assert carry is not None and carry[0] < dk
            ops += [("MUL", (dk, int(dj), int(di)), c1), ("FMA", carry, c0)]
        elif re.fullmatch(r"rfma\(%s, %s, rmul\(%s, %s\)\)" % (u, lit, u, lit), rhs):
            dj0, di0, c0, dj, di, c1 = re.fullmatch(r"rfma\(%s, %s, rmul\(%s, %s\)\)" % (u, lit, u, lit), rhs).groups()
            ops += [("MUL", (dk, int(dj), int(di)), c1), ("FMA", (dk, int(dj0), int(di0)), c0)]
        else:
            m = re.fullmatch(r"rfma\(%s, %s, P\(%d\)\)" % (u, lit, dk), rhs)
            assert m, stmt
            ops.append(("FMA", (dk, int(m.group(1)), int(m.group(2))), m.group(3)))
    return ops


@pytest.mark.parametrize("case", ["c4", "c5", "box27", "aniso", "kside", "star7neg", "f32"])
def test_pair_unit_evaluates_the_single_step_chain(built, case):
    """No deferred scale, no row factorisation, and per output exactly DRS_CHAIN: same terms, same order, same
    literal text."""
    import exact_ops as X
    if case in PRESETS:
        plan = _preset(case)
    elif case == "f32":
        plan = _plan("3d7pt_star", (512, 512, 1024), dtype="f32")
    else:
        op = X.OPS[case]
        offs = list(op)
        plan = drs.Plan(drs.Stencil.from_points(offs, [op[o] for o in offs], (512, 512, 512), 2, name="exact_" + case),
                        drs.Knobs())
    src = plan.pair_source
    assert src and "DRS_OUT_SCALE" not in src and "DRS_FACTORED" not in src
    assert "#define DRS_HALO %d\n" % plan.info.halo in src
    chain = _chain(plan.source)
    assert len(chain) == plan.info.npoints
    assert _scatter_order(src) == chain


def test_pair_split_rule(built):
    """n sweeps = p pairs + s singles: p even, s = 2 when (n - 2) / 2 is even and 4 otherwise; plans without pair
    launches keep n single sweeps."""
    c5, small = _preset("c5"), _plan("3d7pt_star", (64, 64, 64))
    for T in range(1, 201):
        n = drs.sweep_count(T, 1)
        p, s = c5.pair_split(T)
        assert 2 * p + s == n and p % 2 == 0 and s == (2 if ((n - 2) // 2) % 2 == 0 else 4), (T, p, s)
        assert small.pair_split(T) == (0, n)
    assert c5.pair_split(100) == (48, 4)
