"""Exact-arithmetic parity: operators whose every coefficient is k / 2^f (f <= 6, a `%g` literal that is exact) applied
to small integer inputs.  While |K|^s |u| stays far below 2^p (p = 53, or 24 in fp32), every partial sum of every
evaluation order -- gather chain, scatter, row factorisation w (x) h + residual, a deferred power-of-two scale,
forward/backward partial sums, the composed operator -- is exactly representable.  Any correct kernel then equals the
exact answer bit for bit, at any temporal depth and in fp32 too, and a wrong neighbour, a stale stage, a mis-rotated
level or a one-ulp coefficient shows up as a mismatch instead of hiding behind a tolerance.

Shared by test_exact_operators.py (CPU: the preconditions and path markers of every case) and
test_exact_operators_gpu.py (the comparisons) on small grids, and by test_exact_sizes.py / test_exact_sizes_gpu.py at
the sizes where size-gated kernel paths switch on (procedural input, a reference computed one slow-axis window at a
time)."""
import re
from fractions import Fraction

import numpy as np

# ------------------------------------------------------------------------------------------------------------------
# operators: {offset: coefficient}, offsets (dj, di) in 2D and (dk, dj, di) in 3D
# ------------------------------------------------------------------------------------------------------------------


def _box27():
    rng = np.random.default_rng(27)
    pts = {(k, j, i): float(rng.choice([-2, -1, 1, 2])) / 16 for k in (-1, 0, 1) for j in (-1, 0, 1) for i in (-1, 0, 1)}
    pts[(-1, -1, -1)] = -1 / 8          # the leading coefficient (deferred scale) is a power of two
    pts[(0, 0, 0)] = -1.0
    return pts


OPS = {
    # 3x3, negative centre: factorises as (1, 2, 2) (x) (1, 2, 1) / 16 with a residual -1 at the centre
    "mixed3x3": {(-1, -1): 1 / 16, (-1, 0): 2 / 16, (-1, 1): 1 / 16, (0, -1): 2 / 16, (0, 0): -12 / 16, (0, 1): 2 / 16,
                 (1, -1): 1 / 8, (1, 0): 2 / 8, (1, 1): 1 / 8},
    # separable (1, 2, 1) (x) (1, 2, 1) / 16: factorised, no residual, deferred scale 1/16
    "sep121": {(j, i): (2 - abs(j)) * (2 - abs(i)) / 16 for j in (-1, 0, 1) for i in (-1, 0, 1)},
    # one-sided in both axes: rows j .. j+2, columns i-2 .. i (no term at dj = -RJ: no deferred scale, empty P rows)
    "onesided": {(0, 0): -1 / 2, (0, -1): 1 / 4, (0, -2): -1 / 8, (1, 0): 3 / 8, (1, -1): -1 / 4, (1, -2): 1 / 8,
                 (2, 0): 1 / 8, (2, -1): -1 / 8, (2, -2): 1 / 4},
    # radius-3 star with zero gaps at +-2: E = 3 > one fp64 vector, so a lane owns two
    "star3gap": {(0, 0): -1.0, (0, -1): 1 / 4, (0, 1): 1 / 4, (0, -3): 1 / 8, (0, 3): 1 / 8,
                 (-1, 0): 1 / 4, (1, 0): 1 / 4, (-3, 0): 1 / 8, (3, 0): 1 / 8},
    # coefficients of exactly +1 and -1, a leading +1 (no deferred scale): the copy / radd branches of the scatter
    "unit": {(-1, 0): 1.0, (0, -1): -1.0, (0, 0): 1 / 4, (0, 1): 1.0, (1, 0): -1 / 2},
    # two terms: the P == 2 order of the gather chain
    "two": {(0, 0): 3 / 4, (1, -1): -1 / 2},
    "box27": _box27(),
    # RK = 3, RJ = 2, E = 2, gaps at dk = +-2 and dj = +-1
    "aniso": {(0, 0, 0): -1.0, (-1, 0, 0): 1 / 4, (1, 0, 0): 1 / 4, (-3, 0, 0): 1 / 8, (3, 0, 0): 1 / 8,
              (0, -2, 0): 1 / 8, (0, 2, 0): 1 / 8, (0, 0, -1): 1 / 4, (0, 0, 1): 1 / 4, (0, 0, -2): 1 / 8, (0, 0, 2): 1 / 8},
    # planes k and k+1 only
    "kside": {(0, 0, 0): -1 / 2, (0, 0, -1): 1 / 4, (0, 0, 1): 1 / 4, (0, -1, 0): 1 / 8, (0, 1, 0): 1 / 8,
              (1, 0, 0): 1 / 2, (1, -1, 1): -1 / 8},
    # the 7-point star of c4 / c5: one centre and six equal arms
    "star7neg": {(0, 0, 0): -1 / 2, (-1, 0, 0): 1 / 8, (1, 0, 0): 1 / 8, (0, -1, 0): 1 / 8, (0, 1, 0): 1 / 8,
                 (0, 0, -1): 1 / 8, (0, 0, 1): 1 / 8},
    # a 7-point star whose arms differ in sign along every axis (a mirrored neighbour shows), sum |K| = 1: exact in
    # fp32 over six sweeps
    "star7asym": {(0, 0, 0): -1 / 4, (-1, 0, 0): 1 / 8, (1, 0, 0): -1 / 8, (0, -1, 0): -1 / 8, (0, 1, 0): 1 / 8,
                  (0, 0, -1): 1 / 8, (0, 0, 1): -1 / 8},
    # two terms of +-1/2 on a diagonal through k, j and i: sum |K| = 1 with f = 1, so values stay multiples of 2^-d
    # below 3 -- exact over the 16 to 24 levels of the deep fused slab runs (test_exact_slab*.py), fp32 included
    "diag2k": {(-1, 0, 0): 1 / 2, (1, 1, -1): -1 / 2},
    # shaped like the shipped 2D stencils (same offsets, same classes of equal coefficients, hence the same kernel
    # path as the preset: test_exact_sizes.py compares the generated units).  Composed coefficients must print
    # exactly with 6 digits (generate.hpp), which rules out deep dyadic fractions: c2 and c3 use small integers with a
    # power-of-two leading coefficient.
    # c1: 5-point star
    "star5": {(0, 0): -1 / 2, (-1, 0): 1 / 8, (0, -1): 1 / 8, (0, 1): 1 / 8, (1, 0): 1 / 8},
    # c2: 3x3 box, corners 2, edges 4 = 2 x 2, centre -6: rows (2, 4, 2) (x) (1, 2, 1) plus a residual at the centre
    "box9": {(j, i): {0: -6.0, 1: 4.0, 2: 2.0}[abs(j) + abs(i)] for j in (-1, 0, 1) for i in (-1, 0, 1)},
    # c3: 5x5 box with the preset's five classes -- centre, |d| = 1 edges, (+-2, 0) / (0, +-2) / diagonals, knights,
    # corners -- in the preset's row proportions: rows (2, 4, 8, 4, 2), a half row plus corner residuals, twice the
    # row plus a centre residual
    "box25": {(j, i): {(0, 0): -8.0, (0, 1): 8.0, (0, 2): 4.0, (1, 1): 4.0, (1, 2): 2.0, (2, 2): -1.0}[
        tuple(sorted((abs(j), abs(i))))] for j in range(-2, 3) for i in range(-2, 3)},
}


def op_dim(op):
    return len(next(iter(OPS[op])))


# ------------------------------------------------------------------------------------------------------------------
# cases: (id, operator, dtype, knobs, runner, sweeps, path, factored, env)
#   runner  "run" (Plan.run), "sweep" (Plan.sweep), "gold" (Plan.gold_run), "host" / "host_streamed" (Plan.run_host)
#   sweeps  of the ping-pong schedule (1: A -> B only)
#   path    the kernel that must run: gather2d, gather3d, cta3d, temporal2d, fused3d, multi3d, reuse
#   factored  2D temporal: whether the row factorisation must be in use (None: not applicable)
# ------------------------------------------------------------------------------------------------------------------

def _c(op, dtype="f64", runner="run", sweeps=2, path=None, factored=None, env=None, **kn):
    step = kn.get("step", 1)
    cid = "%s-%s-s%d-%s" % (op, dtype, step, runner)
    if "fuse" in kn:
        cid += "-" + kn["fuse"]
    for k in sorted(kn):
        if k not in ("step", "fuse"):
            cid += "-%s%s" % (k, kn[k])
    if env:
        cid += "-flatmode2"
    return dict(id=cid, op=op, dtype=dtype, knobs=dict(kn, dtype=dtype), runner=runner, sweeps=sweeps, path=path,
                factored=factored, env=env or {})


T = "temporal"
FLAT2 = {"DRS_FLAT_MODE": "2"}

CASES = [
    # single step, fp64 and fp32
    *[_c(op, dt, path="gather2d") for op in ("mixed3x3", "sep121", "onesided", "star3gap", "unit", "two")
      for dt in ("f64", "f32")],
    *[_c(op, dt, path="gather3d") for op in ("box27", "aniso", "kside", "star7neg") for dt in ("f64", "f32")],
    _c("mixed3x3", path="gather2d", env=FLAT2), _c("two", "f32", path="gather2d", env=FLAT2),
    _c("box27", path="gather3d", env=FLAT2),
    # 2D temporal blocking
    *[_c("mixed3x3", step=s, fuse=T, path="temporal2d", factored=True) for s in (2, 3, 4)],
    _c("mixed3x3", step=6, fuse=T, sweeps=1, runner="sweep", path="temporal2d", factored=True),
    _c("mixed3x3", step=3, fuse=T, no_factor=1, path="temporal2d", factored=False),
    _c("mixed3x3", step=2, fuse=T, vectors=1, path="temporal2d", factored=True),
    _c("mixed3x3", "f32", step=2, fuse=T, runner="sweep", sweeps=1, path="temporal2d", factored=True),
    *[_c("sep121", step=s, fuse=T, path="temporal2d", factored=True) for s in (2, 3, 4)],
    _c("sep121", step=6, fuse=T, runner="sweep", sweeps=1, path="temporal2d", factored=True),
    _c("sep121", step=4, fuse=T, no_factor=1, path="temporal2d", factored=False),
    _c("sep121", step=2, fuse=T, vectors=2, path="temporal2d", factored=True),
    _c("sep121", "f32", step=2, fuse=T, path="temporal2d", factored=True),
    _c("sep121", "f32", step=4, fuse=T, runner="sweep", sweeps=1, path="temporal2d", factored=True),
    _c("sep121", step=3, fuse=T, path="temporal2d", factored=True, env=FLAT2),
    *[_c("onesided", step=s, fuse=T, path="temporal2d", factored=False) for s in (2, 3, 4)],
    _c("onesided", step=6, fuse=T, runner="sweep", sweeps=1, path="temporal2d", factored=False),
    _c("onesided", "f32", step=3, fuse=T, runner="sweep", sweeps=1, path="temporal2d", factored=False),
    *[_c("star3gap", step=s, fuse=T, path="temporal2d", factored=False) for s in (2, 3, 4)],
    _c("star3gap", step=6, fuse=T, runner="sweep", sweeps=1, path="temporal2d", factored=False),
    _c("star3gap", step=2, fuse=T, vectors=1, path="temporal2d", factored=False),
    _c("star3gap", "f32", step=2, fuse=T, path="temporal2d", factored=False),
    _c("star3gap", step=3, fuse=T, path="temporal2d", factored=False, env=FLAT2),
    *[_c("unit", step=s, fuse=T, path="temporal2d", factored=False) for s in (2, 3, 4, 6)],
    _c("unit", "f32", step=3, fuse=T, runner="sweep", sweeps=1, path="temporal2d", factored=False),
    *[_c("two", step=s, fuse=T, path="temporal2d", factored=False) for s in (2, 4, 6)],
    _c("two", "f32", step=4, fuse=T, runner="sweep", sweeps=1, path="temporal2d", factored=False),
    # 3D temporal: fused in one kernel, or one launch per sub-step
    *[_c("box27", step=s, fuse=T, path="fused3d") for s in (2, 3)],
    _c("box27", step=4, fuse=T, runner="sweep", sweeps=1, path="fused3d"),
    _c("box27", "f32", step=2, fuse=T, runner="sweep", sweeps=1, path="fused3d"),
    _c("box27", step=2, fuse=T, no_fused3d=1, path="multi3d"),
    *[_c("aniso", step=s, fuse=T, path="fused3d") for s in (2, 3)],
    _c("aniso", step=3, fuse=T, no_fused3d=1, path="multi3d"),
    *[_c("kside", step=s, fuse=T, path="fused3d") for s in (2, 4)],
    _c("kside", step=2, fuse=T, no_fused3d=1, path="multi3d"),
    *[_c("star7neg", "f32", step=s, fuse=T, path="fused3d") for s in (2,)],
    *[_c("star7neg", "f32", step=s, fuse=T, runner="sweep", sweeps=1, path="fused3d") for s in (3, 4)],
    _c("star7neg", "f32", step=3, fuse=T, runner="sweep", sweeps=1, no_fused3d=1, path="multi3d"),
    _c("star7neg", step=4, fuse=T, path="fused3d"),
    # 3D single step with one input ring shared by the CTA's warps
    _c("box27", share_x=2, share_y=2, path="cta3d"), _c("star7neg", "f32", share_x=1, share_y=4, path="cta3d"),
    _c("aniso", share_x=1, share_y=2, path="cta3d"),
    # the composed operator evaluated literally / forward-backward data reuse (composed literals stay exact)
    _c("unit", step=2, fuse="algebraic", path="gather2d"), _c("two", step=2, fuse="algebraic", path="gather2d"),
    _c("star7neg", step=2, fuse="algebraic", path="gather3d"),
    _c("unit", fuse="reuse", path="reuse"), _c("unit", step=2, fuse="reuse", path="reuse"),
    _c("star3gap", fuse="reuse", path="reuse"), _c("star7neg", step=2, fuse="reuse", path="reuse"),
    _c("box27", fuse="reuse", path="reuse"),
    # the gold kernel (the reference's gold_ expression of the composed operator)
    _c("mixed3x3", runner="gold", path="gold"), _c("unit", step=2, runner="gold", path="gold"),
    _c("star7neg", step=2, runner="gold", path="gold"), _c("kside", "f32", runner="gold", path="gold"),
    # host buffers: plain and streamed (time-skewed blocks)
    _c("mixed3x3", step=2, fuse=T, runner="host", path="temporal2d", factored=True),
    _c("mixed3x3", step=2, fuse=T, runner="host_streamed", path="temporal2d", factored=True),
    _c("box27", runner="host", sweeps=4, path="gather3d"), _c("box27", runner="host_streamed", sweeps=4, path="gather3d"),
]
CASE_BY_ID = {c["id"]: c for c in CASES}
assert len(CASE_BY_ID) == len(CASES)

HEADERS = {"gather2d": "drs_sweep2d.cuh", "temporal2d": "drs_sweep2d.cuh", "gather3d": "drs_sweep3d.cuh",
           "multi3d": "drs_sweep3d.cuh", "cta3d": "drs_sweep3d_cta.cuh", "fused3d": "drs_sweep3d_t.cuh",
           "reuse": "drs_reuse.cuh"}


def step_of(case):
    return case["knobs"].get("step", 1)


def make_plan(case, shape):
    import drstencil_b200 as drs
    op = OPS[case["op"]]
    offs = list(op)
    st = drs.Stencil.from_points(offs, [op[o] for o in offs], shape, 2 * step_of(case), name="exact_" + case["op"])
    return drs.Plan(st, drs.Knobs(**case["knobs"]))


def shapes(case):
    """Grids cut to the plan's own tiles: interior widths of one and two warp tiles, minus one, exact and plus one; a
    slow extent whose last chunk holds a single output row / plane; the minimal grid 2 * Halo + 1."""
    dim = op_dim(case["op"])
    probe = make_plan(case, (300, 520) if dim == 2 else (300, 40, 200))
    info = probe.info
    H, tx, ty = info.halo, info.tile_x, info.tile_y
    # the chunk of a grid with enough rows / planes for several chunks
    last = 2 * H + 2 * info.chunk + 1
    if dim == 2:
        out = [(last, 2 * H + tx - 1), (2 * H + 3, 2 * H + tx), (last, 2 * H + tx + 1),
               (2 * H + 5, 2 * H + 2 * tx - 1), (2 * H + 2, 2 * H + 2 * tx), (last, 2 * H + 2 * tx + 1), (2 * H + 1, 2 * H + 1)]
    else:
        out = [(last, 2 * H + ty + 1, 2 * H + tx - 1), (2 * H + 3, 2 * H + 2 * ty, 2 * H + tx),
               (2 * H + 2, 2 * H + ty - 1, 2 * H + 2 * tx + 1), (2 * H + 1, 2 * H + 1, 2 * H + 1)]
    if case["path"] == "cta3d":         # the shared ring has no unaligned-pitch form: widths rounded up to a 16-byte pitch
        vec = 2 if case["dtype"] == "f64" else 4
        out = list(dict.fromkeys(s[:-1] + (-(-s[-1] // vec) * vec,) for s in out))
    return out


# ------------------------------------------------------------------------------------------------------------------
# inputs and the exact reference
# ------------------------------------------------------------------------------------------------------------------

UMAX = 2          # |u| of the random field
IMPULSE = 3       # seeded impulses on tile and lane seams


def make_input(case, shape, info, seed):
    """Small seeded integers, plus impulses on the seams of the warp tiles (x) and of the lanes' columns and on the
    first and last row / plane of the chunks (slow axis), so that a mismatch there names the seam."""
    rng = np.random.default_rng(seed)
    a = rng.integers(-UMAX, UMAX + 1, size=shape).astype(np.float64)
    H = info.halo
    cols = 2 if case["dtype"] == "f64" else 4
    xs = [H + q * info.tile_x + d for q in (0, 1, 2) for d in (-1, 0)] + [H + cols * q for q in range(1, 40, 7)]
    slow = [H + q * info.chunk + d for q in (0, 1, 2) for d in (-1, 0)]
    sign = 1.0
    for x in xs:
        for y in slow:
            if 0 <= x < shape[-1] and 0 <= y < shape[0]:
                idx = (y, rng.integers(0, shape[1]), x) if len(shape) == 3 else (y, x)
                a[idx] = sign * IMPULSE
                sign = -sign
    return a.astype(np.float32 if case["dtype"] == "f32" else np.float64)


def _as3(a):
    return a.reshape((1,) + a.shape) if a.ndim == 2 else a


def _offsets3(op):
    return [((0,) + o) if len(o) == 2 else o for o in op]


def _is_np(u):
    return isinstance(u, np.ndarray)


def _torch():
    import torch
    return torch


def apply_levels(u, op, ts, mag=False, dtype=None):
    """ts applications of the operator on shrinking valid regions (in `dtype`, float64 by default; |K| on |u| when
    mag).  Returns the last level as a full-size array; only the region every level could compute is meaningful.
    `u` is a numpy array or a torch tensor (on any device); the result is of the same kind."""
    xp = np if _is_np(u) else _torch()
    if dtype is None:
        dtype = xp.float64
    cur = _as3(abs(u) if mag else u)
    cur = cur.astype(dtype) if xp is np else cur.to(dtype)
    offs = _offsets3(op)
    lo, hi = [0, 0, 0], list(cur.shape)
    for _ in range(ts):
        nlo = [lo[a] + max(0, -min(o[a] for o in offs)) for a in range(3)]
        nhi = [hi[a] - max(0, max(o[a] for o in offs)) for a in range(3)]
        nxt = xp.zeros_like(cur)
        dst = tuple(slice(nlo[a], nhi[a]) for a in range(3))
        if all(nlo[a] < nhi[a] for a in range(3)):
            for o, c in zip(offs, op.values()):
                src = tuple(slice(nlo[a] + o[a], nhi[a] + o[a]) for a in range(3))
                c = abs(c) if mag else c
                nxt[dst] += (dtype(c) if xp is np else c) * cur[src]
        cur, lo, hi = nxt, nlo, nhi
    return cur.reshape(u.shape)


def halo_of(op, step):
    return step * max(0, max(o[0] for o in op))


def interior(shape, H):
    return tuple(slice(H, n - H) for n in shape)


def _f64(u):
    return u.astype(np.float64) if _is_np(u) else u.to(_torch().float64).clone()


def exact_run(op, step, A, B, sweeps, slow=None):
    """The ping-pong schedule of Plan.run: sweep s writes interior(Halo) of buffer (s + 1) % 2 from buffer s % 2,
    every sweep applying the operator `step` times; the destination's ring keeps its contents.  float64 copies (numpy
    or torch, like the inputs).  slow = (lo, hi): the sweeps write slow-axis planes / rows [lo, hi) instead of
    [Halo, n - Halo) -- a slab's output range, everything outside it (its ghost planes) frozen."""
    bufs = [_f64(A), _f64(B)]
    H = halo_of(op, step)
    lo, hi = (H, A.shape[0] - H) if slow is None else slow
    inner = (slice(lo, hi),) + interior(A.shape[1:], H)
    for s in range(sweeps):
        src, dst = bufs[s & 1], bufs[(s & 1) ^ 1]
        if hi > lo and all(n > 2 * H for n in A.shape[1:]):
            dst[inner] = apply_levels(src, op, step)[inner]
    return bufs


# ------------------------------------------------------------------------------------------------------------------
# preconditions
# ------------------------------------------------------------------------------------------------------------------

def _dyadic(v):
    """(k, q) with v == k / 2^q exactly, or None."""
    f = Fraction(v)
    d = f.denominator
    if d & (d - 1):
        return None
    return f.numerator, d.bit_length() - 1


def growth_ok(case, u):
    """(a): with every coefficient a multiple of 2^-f, the values of depth d are multiples of 2^-(f d) bounded by
    max(1, sum|K|)^d max|u|; in units of 2^-(f d) that is max(2^f, sum|K| 2^f)^d max|u|, which must stay below
    2^(p - 4) over the whole schedule (the margin covers the factorised and deferred-scale intermediates)."""
    op = OPS[case["op"]]
    f = max(_dyadic(c)[1] for c in op.values())
    knum = sum(abs(_dyadic(c)[0]) << (f - _dyadic(c)[1]) for c in op.values())
    depth = step_of(case) * case["sweeps"]
    umax = int(np.max(np.abs(u)))
    p = 53 if case["dtype"] == "f64" else 24
    return max(1 << f, knum) ** depth * umax < 2 ** (p - 4), (max(1 << f, knum), depth, umax)


_MACRO = re.compile(r"^#define (\w+)(?:\([^)]*\))?((?:.*\\\n)*.*)$", re.M)
_LIT = re.compile(r"\(real\)\(([^)]*)\)")
_CHAIN_ARG = re.compile(r"(?:MUL|FMA)\(\s*-?\d+,\s*-?\d+,\s*-?\d+,\s*([^)]*)\)")
ARITH_MACROS = ("DRS_CHAIN", "DRS_SCATTER", "DRS_SCATTER3", "DRS_HROW", "DRS_OUT_SCALE", "DRS_FWD_SLOW", "DRS_FWD_MID",
                "DRS_FWD_FAST", "DRS_BWD")


def literals(source, names):
    """{macro: [literal texts]} of the arithmetic macros `names` in a generated translation unit."""
    out = {}
    for m in _MACRO.finditer(source):
        name, body = m.group(1), m.group(2)
        if name not in names:
            continue
        if name == "DRS_OUT_SCALE":
            out[name] = [body.strip().strip("()")]
        else:
            out[name] = _LIT.findall(body) + _CHAIN_ARG.findall(body)
    return out


def literals_exact(source, names, dtype):
    """(b): every literal the kernel multiplies by reads back as k / 2^q with a short k (exact in fp32 too) and a
    power of two q inside the dtype's normal range.  Returns the offending (macro, text) pairs."""
    bad = []
    for name, texts in literals(source, names).items():
        for t in texts:
            try:
                v = Fraction(t)          # the decimal text itself, not the double it rounds to
            except ValueError:
                bad.append((name, t))
                continue
            kq = _dyadic(v) if v.denominator & (v.denominator - 1) == 0 else None
            lim = 100 if dtype == "f32" else 900
            if kq is None or abs(kq[0]) >= 1 << 16 or abs(kq[1]) > lim or (v != 0 and abs(v) > Fraction(2) ** 60):
                bad.append((name, t))
    return bad


def markers(case, plan, shape, env_flat2):
    """(c): the markers of the intended kernel path in plan.source.  Returns a list of failures."""
    src, info = plan.source, plan.info
    path, step = case["path"], step_of(case)
    fails = []
    if path == "gold":          # the gold kernel is in every translation unit, whatever the sweep kernel
        return fails if info.kernel_name.startswith("dr_") else ["kernel " + info.kernel_name]
    ts = step if path in ("temporal2d", "fused3d") else 1
    if "#define DRS_TS %d\n" % ts not in src:
        fails.append("DRS_TS %d" % ts)
    if HEADERS[path] not in src:
        fails.append(HEADERS[path])
    if path in ("gather2d", "gather3d", "multi3d", "cta3d") and "drs_sweep3d_t.cuh" in src:
        fails.append("fused kernel present")
    if path == "gather3d" and "drs_sweep3d_cta.cuh" in src:
        fails.append("shared ring present")
    if case["factored"] is not None and ("#define DRS_FACTORED 1" in src) != case["factored"]:
        fails.append("DRS_FACTORED != %s" % case["factored"])
    if path != "reuse":
        vec = 2 if case["dtype"] == "f64" else 4
        flat = 0 if shape[-1] % vec == 0 else (2 if env_flat2 or path == "fused3d" else 1)
        if flat and "#define DRS_FLAT %d\n" % flat not in src:
            fails.append("DRS_FLAT %d" % flat)
        if not flat and "DRS_FLAT" in src:
            fails.append("unexpected DRS_FLAT")
    if not info.kernel_name.startswith("dr_"):
        fails.append("kernel " + info.kernel_name)
    if "naive kernel" in plan.note or "composed operator used" in plan.note:
        fails.append("note: " + plan.note)
    return fails


def arith_names(case):
    return ARITH_MACROS + (("DRS_GOLD_CHAIN",) if case["runner"] == "gold" else ())


def set_env(case, monkeypatch):
    for k, v in case["env"].items():
        monkeypatch.setenv(k, v)


# ------------------------------------------------------------------------------------------------------------------
# operators whose deferred scale eta^ts would leave the dtype's range (levels carry eta^-s, the store multiplies by
# eta^ts): (name, offsets -> coefficient, shape, dtype, step, factorised)
# ------------------------------------------------------------------------------------------------------------------

RANGE_OPS = {
    # 3D 7-point, fp32, depth 4, leading coefficient 1e-10: eta^4 = 1e-40 (a float subnormal), levels ~1e40
    "star7_tiny_lead_f32": ({(-1, 0, 0): 1e-10, (1, 0, 0): 0.4, (0, -1, 0): 0.1, (0, 1, 0): 0.2, (0, 0, -1): 0.3,
                             (0, 0, 1): 0.1, (0, 0, 0): 0.25}, (24, 30, 72), "f32", 4, False),
    # 3x3 box, fp32, depth 6, factorised with h = the row dj = -1: eta^6 = 1e-42
    "box9_tiny_row_f32": ({(j, i): {-1: 1e-7, 0: 0.2, 1: 0.1}[j] for j in (-1, 0, 1) for i in (-1, 0, 1)},
                          (60, 150), "f32", 6, True),
    # 5-point star, fp64, depth 4, leading coefficient 1e-100: eta^4 = 1e-400 -> 0, levels ~1e400
    "star5_tiny_lead_f64": ({(-1, 0): 1e-100, (0, -1): 0.3, (0, 0): 0.2, (0, 1): 0.3, (1, 0): 0.1},
                            (50, 140), "f64", 4, False),
}


def range_plan(name):
    import drstencil_b200 as drs
    op, shape, dtype, step, _ = RANGE_OPS[name]
    offs = list(op)
    st = drs.Stencil.from_points(offs, [op[o] for o in offs], shape, 2 * step, name="range_" + name.split("_")[0])
    return drs.Plan(st, drs.Knobs(step=step, fuse="temporal", dtype=dtype))


# ------------------------------------------------------------------------------------------------------------------
# grids of any size (test_exact_sizes.py / test_exact_sizes_gpu.py): the engine's kernels choose some paths by grid
# size alone -- the L2 load hint and the exact pair launches from 1 GiB per 3D array, the cp.async fill of unaligned
# rows past a 2^31 flat coordinate, 64-bit addressing past 2^31 elements.  The input below is a function of the global
# index, so it is made one slow-axis window at a time on the device, and the reference of each window is computed from
# the source window it depends on: no full-size copy of anything besides the engine's own two buffers.
# ------------------------------------------------------------------------------------------------------------------

_M31 = 0x7fffffff


def gen_values(flat, seed):
    """Small integers in -UMAX..UMAX from an integer hash of the flat index and the seed.  `flat` is an int64 numpy
    array or torch tensor; every product stays below 2^62, so numpy and torch (any device) agree exactly."""
    h = ((flat & _M31) * 0x2545F491 + (flat >> 31) * 0x9E3779B + (seed & 0xffff) * 0x3C6EF35) & _M31
    h = h ^ (h >> 15)
    h = (h * 0x2C1B3C6D) & _M31
    h = h ^ (h >> 12)
    h = (h * 0x297A2D39) & _M31
    h = h ^ (h >> 15)
    return h % (2 * UMAX + 1) - UMAX


def seams(shape, info):
    """{axis: sorted seam coordinates}: the first and last interior index of every warp tile along x (and y in 3D) and
    of every chunk along the slow axis, for the first three and the last tile / chunk of the grid."""
    H = info.halo
    out = {}
    periods = {0: info.chunk, len(shape) - 1: info.tile_x}
    if len(shape) == 3:
        periods[1] = info.tile_y
    for ax, per in periods.items():
        n = shape[ax]
        last = H + max(0, (n - 2 * H - 1) // per) * per
        qs = {H + q * per for q in (0, 1, 2, 3)} | {last, last + per}
        out[ax] = sorted(v for q in qs for v in (q - 1, q) if 0 <= v < n) + [n - H - 1, n - H]
    return out


def impulses(shape, info):
    """[(index, value)]: +-IMPULSE on pairs of seams (slow axis x fast axis, the middle axis of a 3D grid from a
    hash), and around the flat index 2^31 when the array reaches it."""
    s = seams(shape, info)
    slow, fast = s[0], s[len(shape) - 1]
    out, sign = [], 1
    for z in slow:
        for x in fast:
            if not (0 <= z < shape[0] and 0 <= x < shape[-1]):
                continue
            idx = (z, (z * 7919 + x * 104729) % shape[1], x) if len(shape) == 3 else (z, x)
            out.append((idx, sign * IMPULSE))
            sign = -sign
    total = int(np.prod(shape))
    for f in (2 ** 31 - 1, 2 ** 31, 2 ** 31 + shape[-1]):
        if f < total:
            out.append((tuple(int(v) for v in np.unravel_index(f, shape)), sign * IMPULSE))
            sign = -sign
    return out


def gen_input(shape, lo, hi, seed, imps, like=None):
    """Planes / rows [lo, hi) of the procedural input, float64: a numpy array, or a torch tensor on the device of the
    tensor `like`."""
    plane = int(np.prod(shape[1:]))
    if like is None:
        flat = np.arange(lo * plane, hi * plane, dtype=np.int64)
    else:
        torch = _torch()
        flat = torch.arange(lo * plane, hi * plane, dtype=torch.int64, device=like.device)
    u = gen_values(flat, seed).reshape((hi - lo,) + tuple(shape[1:]))
    u = u.astype(np.float64) if like is None else u.to(_torch().float64)
    for idx, v in imps:
        if lo <= idx[0] < hi:
            u[(idx[0] - lo,) + tuple(idx[1:])] = v
    return u


def reach(op):
    """(r-, r+): how far the operator reaches down and up the slow axis."""
    return max(0, -min(o[0] for o in op)), max(0, max(o[0] for o in op))


def source_window(op, step, sweeps, n_slow, z0, z1):
    """Slow-axis range [s0, s1) of the initial buffers that planes [z0, z1) of both buffers depend on after `sweeps`
    sweeps of depth `step`."""
    rm, rp = reach(op)
    return max(0, z0 - sweeps * step * rm), min(n_slow, z1 + sweeps * step * rp)


def window_run(op, step, sweeps, shape, z0, z1, source, slow=None):
    """exact_run restricted to slow-axis planes / rows [z0, z1) of both buffers: `source(s0, s1)` gives (A, B) over
    source_window(), float64 (numpy or torch); sweeps write the interior of the global grid (slow: exact_run's
    slow-axis output range instead), the frozen ring keeps its contents.  Planes the window's cut edges make wrong
    after sweep s lie within s * step * r of the cut, outside [z0, z1).  Returns the float64 windows (A, B)."""
    s0, s1 = source_window(op, step, sweeps, shape[0], z0, z1)
    bufs = list(source(s0, s1))
    H = halo_of(op, step)
    olo, ohi = (H, shape[0] - H) if slow is None else slow
    if ohi > olo and all(n > 2 * H for n in shape[1:]):
        lo, hi = max(olo, s0) - s0, min(ohi, s1) - s0
        inner = (slice(lo, max(lo, hi)),) + interior(shape[1:], H)
        for s in range(sweeps):
            src, dst = bufs[s & 1], bufs[(s & 1) ^ 1]
            dst[inner] = apply_levels(src, op, step)[inner]
    return bufs[0][z0 - s0:z1 - s0], bufs[1][z0 - s0:z1 - s0]


def windows(shape, elems=1 << 27):
    """Slow-axis windows of about `elems` points."""
    per = max(1, elems // int(np.prod(shape[1:])))
    return [(z, min(shape[0], z + per)) for z in range(0, shape[0], per)]


def describe_mismatch(idx, shape, info, got, ref):
    """One differing point: global index, ring or interior, flat index past 2^31, nearest seam, values."""
    H = info.halo
    ring = any(v < H or v >= n - H for v, n in zip(idx, shape))
    flat = int(np.ravel_multi_index(idx, shape))
    near = None
    for ax, coords in seams(shape, info).items():
        c = min(coords, key=lambda v: abs(v - idx[ax]))
        if near is None or abs(c - idx[ax]) < near[0]:
            near = (abs(c - idx[ax]), "axis %d seam %d" % (ax, c))
    return "%s %s flat %d%s, %s at distance %d: got %r, exact %r" % (
        tuple(idx), "ring" if ring else "interior", flat, " (>= 2^31)" if flat >= 2 ** 31 else "", near[1], near[0],
        got, ref)


# --- the size predicates of generate.hpp (choose_spec, far_beyond_l2), restated to place shapes on their thresholds

def esize(dtype):
    return 8 if dtype == "f64" else 4


def far_beyond_l2(shape, dtype):
    return len(shape) == 3 and int(np.prod(shape)) * esize(dtype) >= 1 << 30


def flat_mode(shape, dtype):
    """DRS_FLAT of a plan without DRS_FLAT_MODE and outside the fused 3D temporal kernel."""
    if shape[-1] % (16 // esize(dtype)) == 0:
        return 0
    total = (shape[0] + 64 if len(shape) == 3 else 1) * (shape[-2] + 256) * shape[-1]
    return 1 if total < 2 ** 31 - 1 else 2


def last_below(pred, make, lo, hi):
    """The largest v in [lo, hi) with pred(make(v)) false, given pred(make(lo)) false and pred(make(hi)) true."""
    assert not pred(make(lo)) and pred(make(hi))
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (lo, mid) if pred(make(mid)) else (mid, hi)
    return lo


# --- cases at size

def _preset_stencil(name):
    import os
    from drstencil_b200.presets import PRESETS
    path, kn = PRESETS[name]
    return os.path.splitext(os.path.basename(path))[0], kn


def _s(cid, op, shape, dtype="f64", runner="run", sweeps=2, path=None, factored=None, preset=None, hint=False,
       pair=False, flat=None, **kn):
    step = kn.get("step", 1)
    if preset is not None:
        step = _preset_stencil(preset)[1].values["step"]
    return dict(id=cid, op=op, shape=tuple(shape), dtype=dtype, runner=runner, sweeps=sweeps, path=path,
                factored=factored, preset=preset, kn=dict(kn, dtype=dtype), knobs=dict(kn, dtype=dtype, step=step),
                hint=hint, pair=pair, flat=flat_mode(shape, dtype) if flat is None else flat, env={})


def _stc_shape(path):
    """(M, N) or (L, M, N) from the header line of a .stc file."""
    with open(path) as f:
        w = f.readline().split()
    ext = dict(zip(w[0::2], w[1::2]))
    return tuple(int(ext[k]) for k in ("L", "M", "N") if k in ext)


def _size_cases():
    from drstencil_b200.presets import PRESETS
    shape = lambda p: _stc_shape(PRESETS[p][0])
    out = [
        # A: the shipped configurations at their sizes, with operators shaped like theirs
        _s("c1", "star5", shape("c1"), preset="c1", sweeps=4, path="gather2d"),
        _s("c1t2", "star5", shape("c1t2"), preset="c1t2", sweeps=4, path="temporal2d", factored=False),
        _s("c2", "box9", shape("c2"), preset="c2", sweeps=2, path="temporal2d", factored=True),
        _s("c3", "box25", shape("c3"), "f32", preset="c3", sweeps=2, path="gather2d"),
        _s("c3t2", "box25", shape("c3t2"), "f32", "sweep", 1, preset="c3t2", path="temporal2d", factored=True),
        _s("c4", "star7neg", shape("c4"), preset="c4", sweeps=6, path="cta3d", hint=True, pair=True),
        _s("c4t2", "star7neg", shape("c4t2"), preset="c4t2", path="fused3d", hint=True),
        _s("c5", "star7neg", shape("c5"), preset="c5", sweeps=6, path="cta3d", hint=True, pair=True),
        _s("c5t2", "star7neg", shape("c5t2"), preset="c5t2", path="fused3d", hint=True),
    ]
    # B: both sides of the 1 GiB rule, fp64 (512 x 512 planes: the rule is met from 512 planes on)
    l_off = last_below(lambda s: far_beyond_l2(s, "f64"), lambda v: (v, 512, 512), 1, 4096)
    for L in (l_off, l_off + 1):
        on = far_beyond_l2((L, 512, 512), "f64")
        side = "on" if on else "off"
        out += [
            _s("l2-%s-gather3d" % side, "box27", (L, 512, 512), sweeps=6, path="gather3d", hint=on, pair=on),
            _s("l2-%s-fused3d" % side, "star7neg", (L, 512, 512), path="fused3d", hint=on, step=2, fuse="temporal"),
            _s("l2-%s-multi3d" % side, "box27", (L, 512, 512), path="multi3d", hint=on, step=2, fuse="temporal",
               no_fused3d=1),
        ]
    # B: both sides of the flat 1 -> 2 rule of unaligned rows, chosen by size alone
    m_off = last_below(lambda s: flat_mode(s, "f32") == 2, lambda v: (v, 32770), 1, 1 << 17)
    l3_off = last_below(lambda s: flat_mode(s, "f64") == 2, lambda v: (v, 512, 1023), 1, 1 << 14)
    for d in (0, 1):
        side = "flat%d" % (1 + d)
        s2, s3 = (m_off + d, 32770), (l3_off + d, 512, 1023)
        out += [
            _s("%s-2d-gather2d" % side, "star5", s2, "f32", path="gather2d"),
            _s("%s-2d-temporal2d" % side, "star5", s2, "f32", path="temporal2d", factored=False, step=2,
               fuse="temporal"),
            _s("%s-3d-gather3d" % side, "star7asym", s3, path="gather3d"),
            _s("%s-3d-multi3d" % side, "star7asym", s3, path="multi3d", step=2, fuse="temporal", no_fused3d=1),
        ]
    # C: past 2^31 elements where no preset goes
    out += [
        _s("big-2d-gather2d", "box9", (65600, 32768), "f32", path="gather2d"),
        _s("big-2d-temporal2d", "box9", (65600, 32768), "f32", "sweep", 1, path="temporal2d", factored=True,
           step=2, fuse="temporal"),
        _s("big-3d-gather3d", "star7asym", (1040, 1024, 2048), "f32", sweeps=6, path="gather3d", hint=True,
           pair=True),
        _s("big-3d-fused3d", "star7asym", (1040, 1024, 2048), "f32", path="fused3d", hint=True, step=2,
           fuse="temporal"),
        _s("big-3d-unaligned-gather3d", "star7asym", (1040, 1024, 2047), "f32", path="gather3d"),
        # D: the host data path at c4's size: plain (pair launches) and streamed with the automatic block
        _s("c4-host", "star7neg", shape("c4"), runner="host", preset="c4", sweeps=6, path="cta3d", hint=True,
           pair=True),
        _s("c4-host-streamed", "star7neg", shape("c4"), runner="host_streamed", preset="c4", sweeps=6, path="cta3d",
           hint=True, pair=True),
    ]
    return out


SIZE_CASES = None


def size_cases():
    global SIZE_CASES
    if SIZE_CASES is None:
        SIZE_CASES = _size_cases()
    return SIZE_CASES


def size_case(cid):
    return {c["id"]: c for c in size_cases()}[cid]


def size_plan(case):
    """The case's plan: Stencil.from_points with the case's operator and size; for a shipped configuration also the
    preset's knobs and stencil name, so that the generated unit is the preset's (see preset_equivalent)."""
    import drstencil_b200 as drs
    op = OPS[case["op"]]
    offs = list(op)
    if case["preset"]:
        name, kn = _preset_stencil(case["preset"])
    else:
        name, kn = "exact_" + case["op"], drs.Knobs(**case["kn"])
    st = drs.Stencil.from_points(offs, [op[o] for o in offs], case["shape"], 2 * step_of(case), name=name)
    return drs.Plan(st, kn)


def normalise_literals(src):
    """A generated unit with every coefficient literal replaced by '#': the `(real)(...)` operands, the chains' last
    arguments and the DRS_OUT_SCALE value."""
    src = re.sub(r"\(real\)\([^)]*\)", "(real)(#)", src)
    src = re.sub(r"(MUL|FMA)\((-?\d+), (-?\d+), (-?\d+), [^)]*\)", r"\1(\2, \3, \4, #)", src)
    return re.sub(r"#define DRS_OUT_SCALE \(.*\)", "#define DRS_OUT_SCALE (#)", src)


def size_markers(case, plan):
    """markers() at the case's size, plus the load hint, the pair unit and the DRS_FLAT the size predicates give."""
    src = plan.source
    fails = markers(case, plan, case["shape"], case["flat"] == 2)
    if case["flat"] == 1 and case["path"] == "fused3d":
        fails.append("the fused 3D kernel has no flat-1 form")
    if ("#define DRS_LD_HINT 1" in src) != case["hint"]:
        fails.append("DRS_LD_HINT != %s" % case["hint"])
    if bool(plan.pair_source) != case["pair"]:
        fails.append("pair unit != %s" % case["pair"])
    if ("drs_sweep3d_cta.cuh" in src) != (case["path"] == "cta3d"):
        fails.append("shared ring")
    if case["path"] == "multi3d" and "#define DRS_TS 1\n" not in src:
        fails.append("multi3d DRS_TS")
    if plan.note and case["path"] != "multi3d":
        fails.append("note: " + plan.note)
    return fails


def size_growth_ok(case):
    """growth_ok over the case's whole schedule with the generator's largest |u|."""
    return growth_ok(case, np.array([IMPULSE]))
