"""Exact-arithmetic parity of the 2D slab path (row slabs, the slab unit drslab_<name> of kernels/slab2d/) on one GPU,
against the float64 reference of exact_ops.py.  Shared by test_exact_slab2d.py (CPU: every case's preconditions, the
slab units' compile health and SASS) and test_exact_slab2d_gpu.py.  The harness is exact_slab.py's -- emulated ranks
and passive neighbours, same sentinel, same released flag words -- on (rows, N) arrays; its geometry, flag and
reference helpers take these cases as they are."""
import numpy as np

import exact_ops as X
import exact_slab as S

T = "temporal"
FLAT2 = X.FLAT2


def _k(op, dtype, path, runner, world, G, fuse=None, N=264, **kw):
    """A case of exact_slab._k on a 2D operator (N columns, three or more warp strips); fuse = the knob, "algebraic"
    tags the id."""
    kn = dict(kw, N=N)
    if path == "temporal2d":
        kn["fuse"] = T
    if fuse:
        kn["fuse"] = fuse
        kn["tag"] = (kn.get("tag", "") + "-" if kn.get("tag") else "") + fuse
    c = S._k(op, dtype, path, runner, world, G, **kn)
    c["factored"] = None if path != "temporal2d" else c["knobs"].get("no_factor") is None and op in ("mixed3x3", "sep121")
    return c


# every rank emulated (Plan.sweep with peer stores): worlds 2-4, uneven splits
EMULATED = [
    # gather (DRS_TS == 1), fp64 and fp32
    _k("mixed3x3", "f64", "gather2d", "emulated", 2, 41),
    _k("sep121", "f32", "gather2d", "emulated", 3, 31),
    _k("onesided", "f64", "gather2d", "emulated", 3, 29, sn=1, claims=("chunk<ghost",)),
    _k("star3gap", "f64", "gather2d", "emulated", 4, 38),
    _k("two", "f64", "gather2d", "emulated", 4, 5, claims=("thin", "ring-ghost")),
    _k("unit", "f32", "gather2d", "emulated", 3, 12, claims=("both-faces",)),
    # unaligned rows: per-row TMA (DRS_FLAT 1) and the cp.async fill (DRS_FLAT 2)
    _k("mixed3x3", "f64", "gather2d", "emulated", 3, 30, N=263),
    _k("sep121", "f64", "gather2d", "emulated", 2, 23, N=263, env=FLAT2),
    # scatter (DRS_TS > 1): depths 2, 3, 4, 6; factored and not; one and two vectors per thread
    _k("mixed3x3", "f64", "temporal2d", "emulated", 2, 40, step=2, vectors=1),
    _k("mixed3x3", "f64", "temporal2d", "emulated", 3, 37, step=3, sweeps=2),
    _k("mixed3x3", "f64", "temporal2d", "emulated", 3, 37, step=3, no_factor=1, sweeps=2),
    _k("sep121", "f64", "temporal2d", "emulated", 3, 50, step=4, vectors=2, sweeps=2),
    _k("sep121", "f32", "temporal2d", "emulated", 4, 46, step=2, sweeps=2),
    _k("onesided", "f64", "temporal2d", "emulated", 2, 45, step=3, sn=4, sweeps=2, claims=("chunk<ghost",)),
    _k("star3gap", "f64", "temporal2d", "emulated", 3, 41, step=2),
    _k("unit", "f64", "temporal2d", "emulated", 4, 45, step=4, sweeps=2),
    _k("two", "f64", "temporal2d", "emulated", 3, 47, step=6, sweeps=2),
    _k("mixed3x3", "f64", "temporal2d", "emulated", 3, 12, step=2, claims=("both-faces",)),
    _k("sep121", "f64", "temporal2d", "emulated", 3, 7, step=2, claims=("thin", "ring-ghost")),
    _k("sep121", "f64", "temporal2d", "emulated", 3, 40, N=263, step=3, sweeps=2),
    _k("star3gap", "f64", "temporal2d", "emulated", 2, 35, N=263, step=2, env=FLAT2),
    # `--fuse algebraic`: the composed operator as a gather plan with a wider halo
    _k("unit", "f64", "gather2d", "emulated", 3, 30, step=2, fuse="algebraic"),
    _k("two", "f32", "gather2d", "emulated", 2, 25, step=3, sweeps=2, fuse="algebraic"),
]

# drs_run_slab as one rank: two calls, a Plan.sweep pair, a third call (calls = sweeps per drs_run_slab call)
RUN_SLAB = [
    _k("mixed3x3", "f64", "gather2d", "run_slab", 3, 30, rank=0, calls=2, sn=2),
    _k("mixed3x3", "f64", "gather2d", "run_slab", 3, 30, rank=1, calls=2, sn=5, claims=("hi-fills",)),
    _k("mixed3x3", "f64", "gather2d", "run_slab", 3, 30, rank=2, calls=2, sn=3),
    _k("mixed3x3", "f64", "gather2d", "run_slab", 1, 20, rank=0, calls=2),
    _k("sep121", "f64", "gather2d", "run_slab", 4, 40, rank=2, calls=2, sn=2),
    _k("two", "f64", "temporal2d", "run_slab", 3, 40, rank=1, calls=2, step=2, sn=3),
    _k("two", "f64", "temporal2d", "run_slab", 3, 48, rank=2, calls=2, step=2, sn=4, vectors=1),
    _k("star3gap", "f64", "gather2d", "run_slab", 3, 40, rank=1, N=263, calls=2),
    _k("unit", "f64", "gather2d", "run_slab", 4, 12, rank=1, calls=2, claims=("both-faces", "hi<nhi")),
    _k("two", "f64", "temporal2d", "run_slab", 3, 16, rank=1, calls=2, step=2, claims=("both-faces", "hi<nhi")),
]

# drs_run_host_slab as one rank: two calls, then one drs_run_slab.  blocks = (host block units, up_skew); 0 units =
# the engine's choice, which needs rows of more than 32 MiB per block
HOST_SLAB = [
    _k("mixed3x3", "f64", "gather2d", "run_host_slab", 3, 60, rank=1, calls=2, blocks=(2, 0), tag="block2H"),
    _k("mixed3x3", "f64", "gather2d", "run_host_slab", 3, 60, rank=1, calls=2, blocks=(7, 1), tag="ragged"),
    _k("mixed3x3", "f64", "gather2d", "run_host_slab", 3, 3600, rank=1, N=4096, calls=2, blocks=(0, 0), tag="auto"),
    _k("mixed3x3", "f64", "gather2d", "run_host_slab", 3, 3600, rank=2, N=4096, calls=2, blocks=(0, 1), tag="auto"),
    _k("unit", "f64", "temporal2d", "run_host_slab", 3, 60, rank=0, calls=2, step=2, sn=4, blocks=(4, 0), tag="block2H"),
    _k("unit", "f64", "temporal2d", "run_host_slab", 3, 61, rank=2, calls=2, step=2, sn=5, blocks=(9, 1), tag="ragged"),
]

# drs_run on a slab plan against the loop of drs_sweep on the same plan, alone and as a passive middle rank
RUN = [
    _k("mixed3x3", "f64", "gather2d", "run", 1, 20, rank=0, sweeps=6),
    _k("mixed3x3", "f64", "gather2d", "run", 3, 60, rank=1, sweeps=6),
    _k("sep121", "f64", "temporal2d", "run", 3, 60, rank=1, step=2, sweeps=4),
]

CASES = EMULATED + RUN_SLAB + HOST_SLAB + RUN
CASE_BY_ID = {c["id"]: c for c in CASES}
assert len(CASE_BY_ID) == len(CASES)

# the shipped 2D configurations whose slab units are compiled and inspected (test_exact_slab2d.py)
PRESETS = ("c1", "c2", "c3", "c1t2", "c3t2")
# c2 (2d9pt_box, depth 4, deferred scale) as a middle rank of its N = 8 slab (test_exact_slab2d_gpu.py)
C2_MIDDLE = dict(preset="c2", world=8, rank=3, sweeps_per_call=4)


def local_shape(case, g):
    return (g.local_planes, case["N"])


def make_plan(case, g):
    """The rank's plan: the case's operator on the rank's local rows, set_slab to its rows."""
    import drstencil_b200 as drs
    op = X.OPS[case["op"]]
    offs = list(op)
    st = drs.Stencil.from_points(offs, [op[o] for o in offs], local_shape(case, g), 2 * S.step_of(case),
                                 name="exact_" + case["op"])
    p = drs.Plan(st, drs.Knobs(**case["knobs"]))
    p.set_slab(g.g_slow, g.lo, g.hi)
    return p


def impulses(shape, gs, chunks, H):
    """[(index, value)]: +-IMPULSE on exact_slab.impulse_planes() (faces, +-H around them, face_lo_end / face_hi_begin,
    chunk seams, global ring rows) at the first and last interior columns and one hashed column in between."""
    G, N = shape
    out, sign = [], 1
    for z in S.impulse_planes(gs, chunks):
        for x in (H, N - H - 1, H + (z * 104729) % max(1, N - 2 * H), H - 1, N - H):
            if 0 <= x < N:
                out.append(((z, x), sign * X.IMPULSE))
                sign = -sign
    return out


def region(g, zl, x, H, N):
    zg = g.origin + zl
    if not 0 <= zg < g.g_slow:
        r = "out-of-grid ghost"
    elif not g.lo <= zg < g.hi:
        r = "ghost"
    elif zg < H or zg >= g.g_slow - H:
        r = "global ring"
    else:
        r = "owned"
    return r + (", lateral ring" if x < H or x >= N - H else "")


def compare(got, want, g, buf, H, chunk, limit=3):
    """[] or a report: the count of differing points and the first `limit` of them with local and global row, column,
    region and nearest chunk seam (numpy or torch, float64)."""
    diff = got != want
    n = int(diff.sum())
    if n == 0:
        return []
    idxs = np.argwhere(diff)[:limit] if isinstance(diff, np.ndarray) else diff.nonzero()[:limit].tolist()
    seams = list(range(g.out_lo, g.out_hi + 1, chunk))
    out = ["rank %d %s: %d points differ" % (g.rank, buf, n)]
    for zl, x in (tuple(int(v) for v in i) for i in idxs):
        near = min(seams, key=lambda s: abs(s - zl)) if seams else None
        out.append("rank %d %s local row %d (global %d), col %d, %s, chunk seam %s: got %r, exact %r" % (
            g.rank, buf, zl, g.origin + zl, x, region(g, zl, x, H, got.shape[1]), near, float(got[zl, x]),
            float(want[zl, x])))
    return out


def self_check(case, chunks):
    """The frozen-ghost reference, with every rank's ghost rows refreshed from the global reference after every sweep,
    equals the global reference cut into the rank's window (both buffers).  Returns a list of failures."""
    op, step, H = X.OPS[case["op"]], S.step_of(case), S.ghost_of(case)
    gs = S.geoms(case)
    shape = (case["G"], case["N"])
    A0, B0 = S.global_input(shape, impulses(shape, gs, chunks, H))
    fails = []
    for g in gs:
        loc = [S.to_local(A0, g), S.to_local(B0, g)]
        ref = [A0, B0]
        for s in range(case["sweeps"]):
            ref = X.exact_run(op, step, ref[0], ref[1], 1) if s % 2 == 0 else X.exact_run(op, step, ref[1], ref[0], 1)[::-1]
            src, dst = loc[s & 1], loc[(s & 1) ^ 1]
            loc[(s & 1) ^ 1] = S.frozen_run(case["op"], step, g, src, dst, 1)[1]
            for b in (0, 1):
                a, z = max(0, g.origin), min(g.g_slow, g.origin + g.local_planes)
                for zg in list(range(a, g.lo)) + list(range(g.hi, z)):
                    loc[b][zg - g.origin] = ref[b][zg]
        for b in (0, 1):
            fails += compare(loc[b], S.to_local(ref[b], g), g, "AB"[b], H, chunks[g.rank])
    return fails
