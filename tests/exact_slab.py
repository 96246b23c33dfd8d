"""Exact-arithmetic parity of the slab path (drs_plan_set_slab) on one GPU, against the float64 reference of
exact_ops.py.  Shared by test_exact_slab.py (CPU: every case's preconditions) and test_exact_slab_gpu.py.

Two ways to run a slab on one device:
- emulated: every rank of a decomposition is a plan of this process, its neighbours' arrays live on the same device,
  and the ranks' Plan.sweep calls of one step run back to back on one stream (no flags).  The whole local arrays of
  every rank then equal the global reference cut into the rank's window: owned planes and ghost planes, both buffers.
- passive neighbours: ONE rank runs its real entry points (drs_run_slab, drs_run_host_slab, drs_run) while its
  neighbours are plain device arrays filled with SENTINEL.  The rank's own flag words are released in advance (both
  slots hold RELEASED; the waits compare with >=), so no wait spins, and the words it signals are zeroed int64 words
  of the test.  Nothing writes the rank's ghost planes during a call, so its arrays follow the ping-pong schedule on
  the local array with the ghost planes frozen: exact_run with the slab's output range.

Never two ranks' flagged sweeps at once on one GPU: a spinning face unit could starve the other rank."""
import numpy as np

import exact_ops as X

SENTINEL = 5.0          # out-of-grid ghost planes and the passive neighbours' arrays: outside every input's range
RELEASED = 1 << 62      # a flag value every wait accepts
SEED = 5


# ------------------------------------------------------------------------------------------------------------------
# cases
#   runner  "emulated" (all ranks, Plan.sweep), "run_slab", "run_host_slab", "run" (drs_run vs the drs_sweep loop)
#   claims  geometry properties the case exists for, proved on the CPU (test_exact_slab.py):
#           thin          some rank is exactly `ghost` planes thick
#           chunk<ghost   the plan's chunk (sn) is below the ghost depth
#           both-faces    a rank with two neighbours has a chunk that touches both faces
#           ring-ghost    rank 0 is thinner than 2 Halo: rank 1's lower ghost planes are global ring planes
#           hi<nhi        the tested rank's face_hi_chunks < nhi (a chunk counted on both faces keeps its place)
#           hi-fills      the tested rank has a lower-face chunk and every later chunk is an upper-face one: a
#                         face_hi_chunks one too large would run a chunk twice and skip another
# ------------------------------------------------------------------------------------------------------------------

def _k(op, dtype, path, runner, world, G, rank=None, M=20, N=72, sweeps=4, env=None, claims=(), calls=None,
       blocks=(), tag="", **kn):
    step = kn.get("step", 1)
    if path == "fused3d":
        kn.setdefault("fuse", "temporal")
    cid = "%s-%s-%s-%s-w%d" % (runner, op, dtype, path, world)
    if step > 1:
        cid += "-s%d" % step
    if rank is not None:
        cid += "-r%d" % rank
    cid += "-G%d-N%d" % (G, N)
    for k in sorted(kn):
        if k not in ("step", "fuse"):
            cid += "-%s%s" % (k, kn[k])
    if env:
        cid += "-flatmode2"
    if tag:
        cid += "-" + tag
    return dict(id=cid, op=op, dtype=dtype, path=path, runner=runner, world=world, G=G, rank=rank, M=M, N=N,
                sweeps=sweeps, env=env or {}, claims=tuple(claims), calls=calls, blocks=tuple(blocks),
                knobs=dict(kn, dtype=dtype), factored=None)


FLAT2 = X.FLAT2

EMULATED = [
    _k("box27", "f64", "gather3d", "emulated", 2, 40),
    _k("star7asym", "f32", "gather3d", "emulated", 3, 31, sweeps=6),
    _k("aniso", "f64", "gather3d", "emulated", 3, 29, sn=2, claims=("chunk<ghost",)),
    _k("kside", "f64", "gather3d", "emulated", 4, 27),
    _k("star7neg", "f64", "gather3d", "emulated", 4, 5, claims=("thin", "ring-ghost")),
    _k("star7asym", "f64", "gather3d", "emulated", 3, 30, N=71),
    _k("box27", "f64", "gather3d", "emulated", 2, 23, N=71, env=FLAT2),
    _k("star7neg", "f64", "gather3d", "emulated", 3, 12, claims=("both-faces",)),
    _k("box27", "f64", "cta3d", "emulated", 3, 30, share_x=2, share_y=2),
    _k("star7neg", "f32", "cta3d", "emulated", 2, 25, share_x=1, share_y=4),
    _k("aniso", "f64", "cta3d", "emulated", 3, 33, share_x=1, share_y=2),
    _k("box27", "f64", "fused3d", "emulated", 3, 7, step=2, claims=("thin", "ring-ghost")),
    _k("aniso", "f64", "fused3d", "emulated", 2, 30, step=2),
    _k("kside", "f64", "fused3d", "emulated", 4, 37, step=2),
    _k("star7asym", "f64", "fused3d", "emulated", 2, 30, step=3, sn=2, claims=("chunk<ghost",)),
    _k("star7asym", "f64", "fused3d", "emulated", 3, 12, step=2, claims=("both-faces",)),
    _k("diag2k", "f64", "fused3d", "emulated", 3, 40, step=4),
    _k("diag2k", "f32", "fused3d", "emulated", 3, 26, N=70, step=2),
]

# drs_run_slab as one rank: two calls, a Plan.sweep pair, a third call (calls = sweeps per drs_run_slab call)
RUN_SLAB = [
    _k("box27", "f64", "gather3d", "run_slab", 3, 30, rank=0, calls=2, sn=2),
    _k("box27", "f64", "gather3d", "run_slab", 3, 30, rank=1, calls=2, sn=5, claims=("hi-fills",)),
    _k("box27", "f64", "gather3d", "run_slab", 3, 30, rank=2, calls=2, sn=3),
    _k("box27", "f64", "gather3d", "run_slab", 1, 20, rank=0, calls=2),
    _k("star7neg", "f64", "cta3d", "run_slab", 4, 40, rank=2, calls=2, sn=2, share_x=2, share_y=2),
    _k("diag2k", "f64", "fused3d", "run_slab", 3, 30, rank=1, calls=2, step=2, sn=3),
    _k("diag2k", "f64", "fused3d", "run_slab", 3, 36, rank=2, calls=2, step=3, sn=4),
    _k("diag2k", "f32", "gather3d", "run_slab", 3, 30, rank=1, calls=2, sn=4),
    _k("star7asym", "f64", "gather3d", "run_slab", 3, 30, rank=1, N=71, calls=2),
    _k("star7neg", "f64", "gather3d", "run_slab", 4, 12, rank=1, calls=2, claims=("both-faces", "hi<nhi")),
    _k("diag2k", "f64", "fused3d", "run_slab", 3, 12, rank=1, calls=2, step=2, claims=("both-faces", "hi<nhi")),
]

# drs_run_host_slab as one rank: two calls, then one drs_run_slab.  blocks = (host block units, up_skew); 0 units =
# the engine's choice, which needs planes of more than 32 MiB per block
HOST_SLAB = [
    _k("star7neg", "f64", "gather3d", "run_host_slab", 3, 60, rank=1, calls=4, blocks=(2, 0), tag="block2H"),
    _k("star7neg", "f64", "gather3d", "run_host_slab", 3, 60, rank=1, calls=4, blocks=(7, 1), tag="ragged"),
    _k("star7neg", "f64", "gather3d", "run_host_slab", 3, 240, rank=1, M=256, N=264, calls=4, blocks=(0, 0),
       tag="auto"),
    _k("star7neg", "f64", "gather3d", "run_host_slab", 3, 240, rank=2, M=256, N=264, calls=4, blocks=(0, 1),
       tag="auto"),
    _k("diag2k", "f64", "fused3d", "run_host_slab", 3, 60, rank=0, calls=4, step=2, sn=4, blocks=(4, 0), tag="block2H"),
    _k("diag2k", "f64", "fused3d", "run_host_slab", 3, 61, rank=2, calls=4, step=2, sn=5, blocks=(9, 1), tag="ragged"),
]

# drs_run on a slab plan against the loop of drs_sweep on the same plan: a small plan and one of >= 1 GiB per array
# (where the engine has exact pair launches for plain plans), each as an alone rank and as a passive middle rank
RUN = [
    _k("star7neg", "f64", "cta3d", "run", 1, 20, rank=0, M=24, N=72, sweeps=6, share_x=2, share_y=2),
    _k("star7neg", "f64", "cta3d", "run", 3, 60, rank=1, M=24, N=72, sweeps=6, share_x=2, share_y=2),
    _k("star7neg", "f64", "gather3d", "run", 1, 512, rank=0, M=512, N=512, sweeps=6),
    _k("star7neg", "f64", "gather3d", "run", 3, 1536, rank=1, M=512, N=512, sweeps=6),
]

CASES = EMULATED + RUN_SLAB + HOST_SLAB + RUN
CASE_BY_ID = {c["id"]: c for c in CASES}
assert len(CASE_BY_ID) == len(CASES)

# the timed configurations' launch: a middle rank of the N = 8 slab of c5 (and c5t2) at full plane size
PRESET_SLABS = {"c5": dict(preset="c5", world=8, rank=3, sweeps_per_call=4, path="cta3d", hint=True),
                "c5t2": dict(preset="c5t2", world=8, rank=3, sweeps_per_call=2, path="fused3d", hint=True)}


def step_of(case):
    return case["knobs"].get("step", 1)


def ghost_of(case):
    return X.halo_of(X.OPS[case["op"]], step_of(case))


def geoms(case):
    from drstencil_b200.slab import SlabGeometry
    return [SlabGeometry(case["G"], case["world"], r, ghost_of(case)) for r in range(case["world"])]


def local_shape(case, g):
    return (g.local_planes, case["M"], case["N"])


def make_plan(case, g):
    """The rank's plan: the case's operator on the rank's local array, set_slab to its planes."""
    import drstencil_b200 as drs
    op = X.OPS[case["op"]]
    offs = list(op)
    st = drs.Stencil.from_points(offs, [op[o] for o in offs], local_shape(case, g), 2 * step_of(case),
                                 name="exact_" + case["op"])
    p = drs.Plan(st, drs.Knobs(**case["knobs"]))
    p.set_slab(g.g_slow, g.lo, g.hi)
    return p


def total_sweeps(case):
    """Sweeps over the whole schedule of the case (every call)."""
    r = case["runner"]
    if r == "run_slab":
        return 3 * case["calls"] + 2
    if r == "run_host_slab":
        return 3 * case["calls"]
    return case["sweeps"]


def growth_ok(case):
    return X.growth_ok(dict(case, sweeps=total_sweeps(case)), np.array([X.IMPULSE, X.UMAX]))


# ------------------------------------------------------------------------------------------------------------------
# fill_params' face counting, restated (capi.cpp): which chunks of a flagged launch belong to a face
# ------------------------------------------------------------------------------------------------------------------

def faces(g, chunk):
    """dict(nzs, nlo, nhi, face_lo_chunks, face_hi_chunks, both) of rank g's drs_run_slab launch; `both` = some chunk
    touches both faces."""
    ghost, local = g.ghost, g.local_planes
    lo_end, hi_begin = 2 * ghost, local - 2 * ghost
    has_lo, has_hi = g.lower is not None, g.upper is not None
    nzs = max(0, -(-(g.out_hi - g.out_lo) // chunk))
    nlo = nhi = 0
    both = False
    for zc in range(nzs):
        za = g.out_lo + zc * chunk
        zb = min(za + chunk, g.out_hi)
        tl, th = has_lo and za < lo_end, has_hi and zb > hi_begin
        nlo += tl
        nhi += th
        both |= tl and th
    return dict(nzs=nzs, nlo=nlo, nhi=nhi, face_lo_chunks=nlo, face_hi_chunks=min(nhi, nzs - nlo), both=both)


def claim_holds(case, claim, chunks):
    """chunks: {rank: the chunk of its plan} (the engine picks a rank's chunk from its local size)."""
    gs = geoms(case)
    H = ghost_of(case)
    if claim == "thin":
        return any(g.hi - g.lo == H for g in gs)
    if claim == "chunk<ghost":
        return all(c < H for c in chunks.values())
    if claim == "both-faces":
        return any(faces(gs[r], c)["both"] for r, c in chunks.items()
                   if gs[r].lower is not None and gs[r].upper is not None)
    if claim == "ring-ghost":
        return gs[0].hi < 2 * H
    if claim == "hi-fills":
        f = faces(gs[case["rank"]], chunks[case["rank"]])
        return f["nlo"] >= 1 and f["nzs"] > f["nlo"] and f["nlo"] + f["face_hi_chunks"] == f["nzs"]
    if claim == "hi<nhi":
        f = faces(gs[case["rank"]], chunks[case["rank"]])
        return f["face_hi_chunks"] < f["nhi"]
    raise KeyError(claim)


# ------------------------------------------------------------------------------------------------------------------
# inputs and references
# ------------------------------------------------------------------------------------------------------------------

def impulse_planes(gs, chunks):
    """Global planes that get +-IMPULSE: every face lo / hi and +-H around it, the planes face_lo_end and
    face_hi_begin, the local chunk seams of the ranks in `chunks` ({rank: chunk}), and the global ring planes inside
    rank 0 and the last rank."""
    G, H = gs[0].g_slow, gs[0].ghost
    zs = set(range(H)) | set(range(G - H, G))
    for g in gs:
        for f in (g.lo, g.hi):
            zs |= {f - H, f - 1, f, f + H - 1, f + H}
        zs |= {g.origin + 2 * H, g.origin + g.local_planes - 2 * H, g.origin + 2 * H - 1,
               g.origin + g.local_planes - 2 * H - 1}
        for z in (range(g.out_lo, g.out_hi + 1, chunks[g.rank]) if g.rank in chunks else ()):
            zs |= {g.origin + z - 1, g.origin + z}
    return sorted(z for z in zs if 0 <= z < G)


def impulses(shape, gs, chunks, H):
    """[(index, value)]: +-IMPULSE on impulse_planes() at the first and last interior rows / columns and one
    hashed row / column in between."""
    G, M, N = shape
    out, sign = [], 1
    for z in impulse_planes(gs, chunks):
        for y, x in ((H, H), (M - H - 1, N - H - 1), (H + (z * 7919) % max(1, M - 2 * H), H + (z * 104729) % max(1, N - 2 * H)),
                     (H - 1, N // 2), (M // 2, N - H)):
            if 0 <= y < M and 0 <= x < N:
                out.append(((z, y, x), sign * X.IMPULSE))
                sign = -sign
    return out


def global_input(shape, imps, like=None, lo=0, hi=None):
    """(A, B) planes [lo, hi) of the global input: small integers from exact_ops.gen_values, impulses in A."""
    hi = shape[0] if hi is None else hi
    return (X.gen_input(shape, lo, hi, SEED, imps, like=like), X.gen_input(shape, lo, hi, SEED + 1, [], like=like))


def to_local(glob, g, fill=SENTINEL):
    """The rank's local array from a global one (numpy or torch): in-grid planes copied, out-of-grid ghosts `fill`."""
    if isinstance(glob, np.ndarray):
        out = np.full((g.local_planes,) + glob.shape[1:], fill, dtype=glob.dtype)
    else:
        import torch
        out = torch.full((g.local_planes,) + tuple(glob.shape[1:]), fill, dtype=glob.dtype, device=glob.device)
    a, b = max(0, g.origin), min(g.g_slow, g.origin + g.local_planes)
    out[a - g.origin:b - g.origin] = glob[a:b]
    return out


def frozen_run(case_op, step, g, A, B, sweeps):
    """The rank's arrays after `sweeps` sweeps with its ghost planes frozen (passive neighbours)."""
    return X.exact_run(X.OPS[case_op], step, A, B, sweeps, slow=(g.out_lo, g.out_hi))


def region(g, zl, y, x, H, M, N):
    zg = g.origin + zl
    if not 0 <= zg < g.g_slow:
        r = "out-of-grid ghost"
    elif not g.lo <= zg < g.hi:
        r = "ghost"
    elif zg < H or zg >= g.g_slow - H:
        r = "global ring"
    else:
        r = "owned"
    if y < H or y >= M - H or x < H or x >= N - H:
        r += ", lateral ring"
    return r


def describe(g, buf, idx, got, want, H, chunk):
    """One differing point of rank g's buffer `buf`: local and global plane, region, nearest chunk seam."""
    zl, y, x = idx
    M, N = got.shape[1:]
    seams = list(range(g.out_lo, g.out_hi + 1, chunk))
    near = min(seams, key=lambda s: abs(s - zl)) if seams else None
    return "rank %d %s local plane %d (global %d), row %d, col %d, %s, chunk seam %s: got %r, exact %r" % (
        g.rank, buf, zl, g.origin + zl, y, x, region(g, zl, y, x, H, M, N), near, float(got[idx]), float(want[idx]))


def compare(got, want, g, buf, H, chunk, limit=3):
    """[] or a report: count of differing points and the first `limit` of them (numpy or torch, float64)."""
    diff = got != want
    n = int(diff.sum())
    if n == 0:
        return []
    idxs = np.argwhere(diff)[:limit] if isinstance(diff, np.ndarray) else diff.nonzero()[:limit].tolist()
    return ["rank %d %s: %d points differ" % (g.rank, buf, n)] + [
        describe(g, buf, tuple(int(v) for v in i), got, want, H, chunk) for i in idxs]


def self_check(case, chunks):
    """The frozen-ghost reference, with every rank's ghost planes refreshed from the global reference after every
    sweep, equals the global reference cut into the rank's window (both buffers).  Returns a list of failures."""
    op, step, H = X.OPS[case["op"]], step_of(case), ghost_of(case)
    gs = geoms(case)
    shape = (case["G"], case["M"], case["N"])
    A0, B0 = global_input(shape, impulses(shape, gs, chunks, H))
    fails = []
    for g in gs:
        loc = [to_local(A0, g), to_local(B0, g)]
        ref = [A0, B0]
        for s in range(case["sweeps"]):
            ref = X.exact_run(op, step, ref[0], ref[1], 1) if s % 2 == 0 else X.exact_run(op, step, ref[1], ref[0], 1)[::-1]
            src, dst = loc[s & 1], loc[(s & 1) ^ 1]
            nxt = frozen_run(case["op"], step, g, src, dst, 1)
            loc[(s & 1) ^ 1] = nxt[1]
            for b in (0, 1):            # the neighbours' pushes: ghost planes of the level each buffer holds
                a, z = max(0, g.origin), min(g.g_slow, g.origin + g.local_planes)
                for zg in list(range(a, g.lo)) + list(range(g.hi, z)):
                    loc[b][zg - g.origin] = ref[b][zg]
        for b in (0, 1):
            fails += compare(loc[b], to_local(ref[b], g), g, "AB"[b], H, chunks[g.rank])
    return fails
