"""Exact-arithmetic parity of pair slabs (drs_plan_set_slab_pairs: ghost regions of 2 * Halo planes, drs_run_slab as
pair launches plus single sweeps) on one GPU, against the float64 reference of exact_ops.py.  Shared by
test_exact_slabpair.py (CPU: every case's preconditions) and test_exact_slabpair_gpu.py.

Two ways to run, as in exact_slab.py:
- emulated: every rank is a plan of this process, its neighbours' arrays live on the same device, and for each launch
  index every rank runs its Plan.sweep_pair / Plan.sweep back to back on one stream (no flags).  Every rank's whole
  local arrays, deep ghost planes included, then equal the global reference cut into the rank's window.
- passive neighbours: ONE rank runs drs_run_slab with its flag words released in advance while its neighbours are
  SENTINEL-filled device arrays.  Nothing writes its ghost planes during a call, so its arrays follow the schedule of
  schedule_ref: the ghost planes frozen as inputs, and -- the difference to the single-sweep frozen-ghost reference --
  a pair launch's level 1 computed on the ghost planes [Halo, 2 Halo) from them.

Never two ranks' flagged launches at once on one GPU: a spinning face CTA could starve the other rank."""
import numpy as np

import exact_ops as X
import exact_slab as S

SENTINEL = S.SENTINEL
RELEASED = S.RELEASED


# ------------------------------------------------------------------------------------------------------------------
# cases
#   runner  "emulated" (all ranks, Plan.sweep_pair / Plan.sweep) or "run_slab" (one rank, passive neighbours)
#   sweeps  sweeps per drs_run_slab call (>= 6: pairs start there); emulated cases run one such schedule
#   claims  geometry properties the case exists for, proved on the CPU (test_exact_slabpair.py):
#           thin          some rank is exactly 2 Halo planes thick
#           chunk<ghost   the single sweeps' chunk (sn) is below the ghost depth 2 Halo
#           both-faces    a rank with two neighbours has a pair chunk that touches both faces
#           ring-ghost    rank 1's deep lower ghost planes reach the global ring
# ------------------------------------------------------------------------------------------------------------------

def _k(op, dtype, runner, world, G, rank=None, M=20, N=72, sweeps=6, claims=(), **kn):
    cid = "%s-%s-%s-w%d" % (runner, op, dtype, world)
    if rank is not None:
        cid += "-r%d" % rank
    cid += "-G%d-N%d-n%d" % (G, N, sweeps)
    for k in sorted(kn):
        cid += "-%s%s" % (k, kn[k])
    return dict(id=cid, op=op, dtype=dtype, path="gather3d", runner=runner, world=world, G=G, rank=rank, M=M, N=N,
                sweeps=sweeps, claims=tuple(claims), knobs=dict(kn, dtype=dtype), env={})


EMULATED = [
    _k("box27", "f64", "emulated", 2, 40, sweeps=6),
    _k("star7asym", "f32", "emulated", 3, 31, sweeps=6),
    _k("aniso", "f64", "emulated", 3, 29, sweeps=8, sn=2),
    _k("kside", "f64", "emulated", 4, 27, sweeps=10),
    _k("star7neg", "f64", "emulated", 4, 9, sweeps=8, sn=1, claims=("thin", "ring-ghost", "chunk<ghost")),
    _k("star7asym", "f64", "emulated", 3, 30, N=76, sweeps=10),
    _k("star7neg", "f64", "emulated", 3, 14, sweeps=6, claims=("both-faces",)),
    _k("diag2k", "f32", "emulated", 3, 26, N=68, sweeps=12),
    _k("diag2k", "f64", "emulated", 2, 33, sweeps=14),
    _k("star7asym", "f64", "emulated", 2, 24, M=24, N=72, sweeps=6, sn=3),
]

# drs_run_slab as one rank with passive neighbours: two calls of `sweeps` sweeps each
RUN_SLAB = [
    _k("star7neg", "f64", "run_slab", 3, 30, rank=0, sweeps=6, sn=2),
    _k("diag2k", "f64", "run_slab", 3, 30, rank=1, sweeps=8, sn=5),
    _k("star7neg", "f64", "run_slab", 3, 30, rank=2, sweeps=6, sn=3),
    _k("diag2k", "f64", "run_slab", 1, 20, rank=0, sweeps=10),
    _k("star7neg", "f64", "run_slab", 4, 16, rank=1, sweeps=6, claims=("both-faces",)),
    _k("diag2k", "f32", "run_slab", 3, 30, rank=1, sweeps=8, sn=4),
    _k("star7asym", "f64", "run_slab", 3, 40, rank=2, N=76, sweeps=6),
]

CASES = EMULATED + RUN_SLAB
CASE_BY_ID = {c["id"]: c for c in CASES}
assert len(CASE_BY_ID) == len(CASES)

# the timed configuration: a middle rank of c5's N = 8 slab at full plane size (192 owned planes + 2 x 2 ghosts)
PRESET_SLAB = dict(preset="c5", world=8, rank=3, sweeps_per_call=6)


def halo_of(case):
    return X.halo_of(X.OPS[case["op"]], 1)


def geoms(case):
    from drstencil_b200.slab import SlabGeometry
    H = halo_of(case)
    return [SlabGeometry(case["G"], case["world"], r, 2 * H, ring=H) for r in range(case["world"])]


def local_shape(case, g):
    return (g.local_planes, case["M"], case["N"])


def make_plan(case, g):
    import drstencil_b200 as drs
    op = X.OPS[case["op"]]
    offs = list(op)
    st = drs.Stencil.from_points(offs, [op[o] for o in offs], local_shape(case, g), 2, name="exact_" + case["op"])
    p = drs.Plan(st, drs.Knobs(**case["knobs"]))
    p.set_slab_pairs(g.g_slow, g.lo, g.hi)
    return p


def pair_split(n):
    """generate.hpp: pair_split, restated."""
    singles = n if n < 2 else (2 if ((n - 2) // 2) % 2 == 0 else 4)
    singles = min(singles, n)
    return (n - singles) // 2, singles


def total_sweeps(case):
    return case["sweeps"] * (2 if case["runner"] == "run_slab" else 1)


def growth_ok(case):
    return X.growth_ok(dict(case, sweeps=total_sweeps(case)), np.array([X.IMPULSE, X.UMAX]))


def pair_chunk(g, H):
    """The pair launch's chunk (generate.hpp: pair_spec): 128 planes, at most the local array less its ring."""
    return min(128, max(1, g.local_planes - 2 * H))


def ring_bounds(g, H):
    """(ring_lo, ring_hi): local planes outside are global ring or out-of-grid planes (capi.cpp: launch_slabpair)."""
    L = g.local_planes
    return min(L, max(0, H - g.origin)), min(L, max(0, g.g_slow - H - g.origin))


def faces(g, chunk):
    """exact_slab.faces with this slab's ghost depth (the rule of fill_params: face_lo_end = 2 ghost)."""
    return S.faces(g, chunk)


def claim_holds(case, claim, chunks):
    """chunks: {rank: the single sweeps' chunk}."""
    gs = geoms(case)
    H = halo_of(case)
    if claim == "thin":
        return any(g.hi - g.lo == 2 * H for g in gs)
    if claim == "chunk<ghost":
        return all(c < 2 * H for c in chunks.values())
    if claim == "both-faces":
        return any(faces(g, pair_chunk(g, H))["both"] for g in gs if g.lower is not None and g.upper is not None)
    if claim == "ring-ghost":
        return len(gs) > 1 and gs[1].lo - 2 * H < H
    raise KeyError(claim)


# ------------------------------------------------------------------------------------------------------------------
# inputs and references
# ------------------------------------------------------------------------------------------------------------------

def impulses(shape, gs, chunks, H):
    """exact_slab.impulses on a deep slab: its planes follow the ranks' ghost depth 2H (the faces and +-2H around them,
    face_lo_end / face_hi_begin, the chunk seams of `chunks`), its rows and columns the ring width H."""
    return S.impulses(shape, gs, chunks, H)


def _clone(u):
    return u.copy() if isinstance(u, np.ndarray) else u.clone()


def schedule_ref(op, bufs, s0, g, H, launches):
    """The arrays of rank g after `launches` ([("pair" | "single", input buffer index)]), with everything outside its
    owned output range frozen (passive neighbours).  bufs = [A, B]: float64 windows of local planes [s0, s0 + n)
    (numpy or torch), updated in place; planes within the launches' reach of a cut window edge are wrong.
      pair: level 0 = the input with the global ring and the lateral ring taken from A; level 1 = B with the
            operator applied on planes [max(Halo, ring_lo), min(L - Halo, ring_hi)) (ghost planes included) and the
            lateral interior; level 2 = the operator on level 1, stored on the owned output range of the output.
      single: the operator on the input, stored on the owned output range of the output (exact_run)."""
    n = bufs[0].shape[0]
    M, N = bufs[0].shape[1:]
    L = g.local_planes
    rlo, rhi = ring_bounds(g, H)
    lat = (slice(H, M - H), slice(H, N - H))

    def planes(a, b):
        a, b = max(a - s0, 0), min(b - s0, n)
        return slice(a, max(a, b))

    out_sl = (planes(g.out_lo, g.out_hi),) + lat
    for kind, src in launches:
        dst = src ^ 1
        if kind == "single":
            bufs[dst][out_sl] = X.apply_levels(bufs[src], op, 1)[out_sl]
            continue
        lv0 = _clone(bufs[src])
        if src == 1:
            ring = _clone(bufs[0])
            ring[(planes(rlo, rhi),) + lat] = lv0[(planes(rlo, rhi),) + lat]
            lv0 = ring
        lv1 = _clone(bufs[1])
        in1 = (planes(max(H, rlo), min(L - H, rhi)),) + lat
        lv1[in1] = X.apply_levels(lv0, op, 1)[in1]
        bufs[dst][out_sl] = X.apply_levels(lv1, op, 1)[out_sl]
    return bufs


def run_launches(n):
    """drs_run_slab's launches for n sweeps: [("pair" | "single", input buffer index)]."""
    p, s = pair_split(n)
    return [("pair", i & 1) for i in range(p)] + [("single", j & 1) for j in range(s)]


def pushed_planes(g, side):
    """Local planes of rank g stored into the `side` neighbour's ghost planes: the 2 Halo owned planes next to it that
    are outputs (global ring planes are never stored)."""
    ghost = g.ghost
    a, b = (ghost, 2 * ghost) if side == "lower" else (g.local_planes - 2 * ghost, g.local_planes - ghost)
    return max(a, g.out_lo), min(b, g.out_hi)


def global_levels(op, A0, B0, n):
    """[level 0 .. level n] of the global ping-pong schedule: level k is buffer k % 2 after k sweeps (its ring is that
    buffer's)."""
    bufs, out = [X._f64(A0), X._f64(B0)], [X._f64(A0)]
    for s in range(n):
        bufs = X.exact_run(op, 1, bufs[s & 1], bufs[(s & 1) ^ 1], 1)
        if s & 1:
            bufs = bufs[::-1]
        out.append(bufs[(s + 1) & 1])
    return out


def self_check(case, chunks):
    """schedule_ref run on every rank with its ghost planes refreshed from the global reference after every launch
    (what the neighbours' pushes do) equals the global reference cut into the rank's window, both buffers.  Returns a
    list of failures."""
    op, H = X.OPS[case["op"]], halo_of(case)
    gs = geoms(case)
    shape = (case["G"], case["M"], case["N"])
    A0, B0 = S.global_input(shape, impulses(shape, gs, chunks, H))
    n = case["sweeps"]
    lv = global_levels(op, A0, B0, n)
    fails = []
    for g in gs:
        loc = [S.to_local(A0, g), S.to_local(B0, g)]
        level = 0
        for kind, src in run_launches(n):
            schedule_ref(op, loc, 0, g, H, [(kind, src)])
            level += 2 if kind == "pair" else 1
            a, z = max(g.ring, g.origin), min(g.g_slow - g.ring, g.origin + g.local_planes)
            for zg in list(range(a, g.lo)) + list(range(g.hi, z)):
                loc[src ^ 1][zg - g.origin][H:-H, H:-H] = lv[level][zg][H:-H, H:-H]
        for b in (0, 1):                # n is even: A holds level n, B level n - 1
            fails += S.compare(loc[b], S.to_local(lv[n - b], g), g, "AB"[b], H, chunks[g.rank])
    return fails
