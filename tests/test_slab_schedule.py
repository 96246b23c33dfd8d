"""Planner for the slab-decomposed host-buffer run (csrc/core/host_schedule.hpp: plan_block_schedule,
reported by drs_plan_slab_schedule) checked on the CPU: the step lists of ALL ranks are executed against
each other -- the CPU oracle stands in for the sweep kernel, ghost planes are pushed into the neighbour's
array exactly where the kernel's fused halo push would store them, flags gate the launches as the slab
flag kernels would -- under random interleavings of the ranks.  Not-yet-uploaded planes and never-filled
ghosts are NaN, so a launch that reads a ghost too early, a push that overwrites a ghost still in use, a
download that comes too late or a deadlock all fail the comparison with the undecomposed schedule
(`for t: sweep(A,B); sweep(B,A)`, /root/reference/codegen.hpp:581-584)."""
import random

import numpy as np
import pytest

from helpers import oracle_terms, stc_path

UPLOAD, SWEEP, DOWNLOAD = 0, 1, 2
WAIT_LO, WAIT_UP, SIG_LO, SIG_UP, INIT_LO, INIT_UP = 1, 2, 4, 8, 16, 32


class Rank:
    def __init__(self, name, gshape, world, rank, block, iters, **kn):
        import drstencil_b200 as drs
        from drstencil_b200.slab import SlabGeometry
        probe = drs.Plan(drs.Stencil.from_file(stc_path(name)).set_size(gshape), drs.Knobs(**kn))
        self.H = probe.halo
        self.geom = SlabGeometry(gshape[0], world, rank, self.H)
        local_shape = (self.geom.local_planes,) + tuple(gshape[1:])
        plan = drs.Plan(drs.Stencil.from_file(stc_path(name)).set_size(local_shape), drs.Knobs(**kn))
        plan.set_slab(gshape[0], self.geom.lo, self.geom.hi)
        plan.set_host_block(block)
        self.steps = plan.slab_schedule(iters, up_skew=rank % 2 == 1)
        self.own_lo, self.own_hi = self.H, self.geom.local_planes - self.H
        self.dev = [np.full(local_shape, np.nan), np.zeros(local_shape)]
        self.flags = [0, 0]          # written by the lower / upper neighbour
        self.pc = 0
        self.host = None

    def enabled(self):
        if self.pc >= len(self.steps):
            return False
        kind, block, sweep, lo, hi, faces = self.steps[self.pc]
        if kind != SWEEP:
            return True
        return (not faces & WAIT_LO or self.flags[0] >= sweep) and (not faces & WAIT_UP or self.flags[1] >= sweep)


def _push(src_rank, dst_rank, buf, planes, to_upper_ghost):
    """Stores src_rank's planes (local indices) into dst_rank's ghost planes of buffer `buf`."""
    for z in planes:
        zg = src_rank.geom.origin + z                         # global plane
        zd = zg - dst_rank.geom.origin                        # neighbour's local index
        assert (zd >= dst_rank.own_hi) if to_upper_ghost else (zd < dst_rank.own_lo)
        dst_rank.dev[buf][zd] = src_rank.dev[buf][z]


def _execute(ranks, r, offs, coefs, halo):
    from oracle import oracle
    me = ranks[r]
    kind, block, sweep, lo, hi, faces = me.steps[me.pc]
    me.pc += 1
    lower = ranks[r - 1] if r > 0 else None
    upper = ranks[r + 1] if r + 1 < len(ranks) else None
    H = me.H
    if kind == UPLOAD:
        me.dev[0][lo:hi] = me.host[lo - me.own_lo:hi - me.own_lo]
        if faces & INIT_LO:
            _push(me, lower, 0, range(me.own_lo, me.own_lo + H), to_upper_ghost=True)
            lower.flags[1] = max(lower.flags[1], 1)
        if faces & INIT_UP:
            _push(me, upper, 0, range(me.own_hi - H, me.own_hi), to_upper_ghost=False)
            upper.flags[0] = max(upper.flags[0], 1)
    elif kind == DOWNLOAD:
        me.host[lo - me.own_lo:hi - me.own_lo] = me.dev[0][lo:hi]
    else:
        src, dst = (me.dev[0], me.dev[1]) if sweep & 1 else (me.dev[1], me.dev[0])
        full = dst.copy()
        oracle.sweep(src, full, offs, coefs, halo)
        dst[lo:hi] = full[lo:hi]
        buf = sweep & 1
        if lower is not None:       # the kernel stores its boundary output planes into the neighbour's ghosts
            _push(me, lower, buf, [z for z in range(lo, hi) if z < me.own_lo + H], to_upper_ghost=True)
        if upper is not None:
            _push(me, upper, buf, [z for z in range(lo, hi) if z >= me.own_hi - H], to_upper_ghost=False)
        if faces & SIG_LO:
            lower.flags[1] = sweep + 1
        if faces & SIG_UP:
            upper.flags[0] = sweep + 1


def _run(name, gshape, world, block, iters, seed, eager_uploads, **kn):
    from oracle import oracle
    step = kn.get("step", 1)
    offs, coefs, halo = oracle_terms(name, step)
    ranks = [Rank(name, gshape, world, r, block, iters, **kn) for r in range(world)]
    assert all(rk.steps for rk in ranks), "expected the streamed slab schedule"
    assert all(rk.H == halo for rk in ranks)
    a0 = oracle.lcg_array(gshape, np.float64, 9)
    for rk in ranks:
        rk.host = a0[rk.geom.lo:rk.geom.hi].copy()
    if eager_uploads:                # the copy engines run ahead: every upload (and ghost init) lands first
        for r, rk in enumerate(ranks):
            ups = [s for s in rk.steps if s[0] == UPLOAD]
            rest = [s for s in rk.steps if s[0] != UPLOAD]
            rk.steps = ups + rest
    rng = random.Random(seed)
    while any(rk.pc < len(rk.steps) for rk in ranks):
        ready = [r for r, rk in enumerate(ranks) if rk.enabled()]
        assert ready, "deadlock: " + str([(rk.pc, len(rk.steps), rk.flags) for rk in ranks])
        _execute(ranks, rng.choice(ready), offs, coefs, halo)
    refA, refB = a0.copy(), np.zeros(gshape)
    oracle.run(refA, refB, offs, coefs, halo, iters, step)
    got = np.concatenate([rk.host for rk in ranks])
    assert np.array_equal(got, refA), (name, gshape, world, block, iters, seed)
    return ranks


CASES = [
    # name, global shape, ranks, block, iterations, knobs
    ("3d7pt_star", (48, 8, 10), 2, 6, 10, dict()),
    ("3d7pt_star", (72, 8, 10), 3, 6, 20, dict()),
    ("3d7pt_star", (80, 8, 10), 4, 8, 30, dict()),             # n * Halo > block and > first blocks
    ("3d7pt_star", (61, 8, 10), 3, 5, 12, dict()),             # uneven slabs
    ("3d7pt_star", (96, 8, 10), 4, 8, 12, dict(step=2, fuse="algebraic")),   # Halo 2: faces split across launches
    ("3d9pt_cross", (60, 8, 10), 3, 4, 8, dict()),
]


@pytest.mark.parametrize("name,gshape,world,block,iters,kn", CASES)
def test_all_ranks_against_each_other(built, name, gshape, world, block, iters, kn):
    for seed in range(4):
        _run(name, gshape, world, block, iters, seed, eager_uploads=bool(seed & 1), **kn)


def _makespan(name, gshape, world, block, iters, alternate, **kn):
    """Ticks needed when every rank that is allowed to run executes one step per tick."""
    offs, coefs, halo = oracle_terms(name, kn.get("step", 1))
    from oracle import oracle
    ranks = [Rank(name, gshape, world, r, block, iters, **kn) for r in range(world)]
    if not alternate:                # every rank skews down: legal, but the faces serialise the ranks
        import drstencil_b200 as drs
        for rk in ranks:
            local_shape = (rk.geom.local_planes,) + tuple(gshape[1:])
            plan = drs.Plan(drs.Stencil.from_file(stc_path(name)).set_size(local_shape), drs.Knobs(**kn))
            plan.set_slab(gshape[0], rk.geom.lo, rk.geom.hi)
            plan.set_host_block(block)
            rk.steps = plan.slab_schedule(iters, up_skew=False)
    a0 = oracle.lcg_array(gshape, np.float64, 9)
    for rk in ranks:
        rk.host = a0[rk.geom.lo:rk.geom.hi].copy()
    ticks = 0
    while any(rk.pc < len(rk.steps) for rk in ranks):
        ready = [r for r, rk in enumerate(ranks) if rk.enabled()]
        assert ready, "deadlock"
        for r in ready:
            _execute(ranks, r, offs, coefs, halo)
        ticks += 1
    return ticks, max(len(rk.steps) for rk in ranks)


def test_alternating_directions_keep_the_ranks_busy(built):
    """With neighbouring ranks skewing in opposite directions the blocks that meet at a face run in
    lockstep and nobody idles; with one direction everywhere the result is the same but every rank
    waits for its lower neighbour's LAST block before it can finish its FIRST one."""
    args = ("3d7pt_star", (96, 8, 10), 4, 6, 16)
    ticks, longest = _makespan(*args, alternate=True)
    assert ticks <= longest + 4, (ticks, longest)
    serial, longest = _makespan(*args, alternate=False)
    assert serial > 1.5 * ticks, (serial, ticks)


def test_faces_and_directions(built):
    """Even ranks skew down (blocks bottom-up), odd ranks are the mirror image; waits and signals
    appear only on launches that touch a face with a neighbour; every level of a face is signalled once."""
    ranks = _run("3d7pt_star", (72, 8, 10), 3, 6, 10, 0, False)
    for r, rk in enumerate(ranks):
        ups = [s for s in rk.steps if s[0] == UPLOAD]
        los = [s[3] for s in ups]
        assert los == sorted(los, reverse=(r % 2 == 1))
        sweeps = [s for s in rk.steps if s[0] == SWEEP]
        n = max(s[2] for s in sweeps)
        for face, sig, has in ((WAIT_LO, SIG_LO, r > 0), (WAIT_UP, SIG_UP, r + 1 < len(ranks))):
            signalled = sorted(s[2] for s in sweeps if s[5] & sig)
            assert signalled == (list(range(1, n + 1)) if has else [])
            assert all(s[5] & face for s in sweeps if s[5] & sig)
        inits = [s[5] for s in ups if s[5]]
        assert sum(bool(f & INIT_LO) for f in inits) == (1 if r > 0 else 0)
        assert sum(bool(f & INIT_UP) for f in inits) == (1 if r + 1 < len(ranks) else 0)


@pytest.mark.parametrize("world", [2, 4, 8])
def test_engine_chosen_blocks_at_the_c5_size(built, world):
    """c5 (1536^3 fp64) over 2 / 4 / 8 ranks with the engine's own block size: every rank gets the same number
    of blocks (the lockstep at the faces relies on it), thin blocks at both ends, 100 signalled levels per face."""
    import drstencil_b200 as drs
    from drstencil_b200.presets import PRESETS
    from drstencil_b200.slab import SlabGeometry
    path, kn = PRESETS["c5"]
    shapes = []
    for rank in range(world):
        geom = SlabGeometry(1536, world, rank, 1)
        st = drs.Stencil.from_file(path).set_size((geom.local_planes, 1536, 1536))
        plan = drs.Plan(st, kn)
        plan.set_slab(1536, geom.lo, geom.hi)
        steps = plan.slab_schedule(100, up_skew=rank % 2 == 1)
        assert steps, (world, rank)
        ups = [s for s in steps if s[0] == UPLOAD]
        sizes = [s[4] - s[3] for s in ups]
        assert sum(sizes) == geom.hi - geom.lo and min(sizes) >= 2
        assert sizes[0] < max(sizes) and sizes[-1] < max(sizes)          # thin first and last block
        shapes.append(len(ups))
        sweeps = [s for s in steps if s[0] == SWEEP]
        for sig, has in ((SIG_LO, rank > 0), (SIG_UP, rank + 1 < world)):
            assert sorted(s[2] for s in sweeps if s[5] & sig) == (list(range(1, 101)) if has else [])
        assert len(sweeps) <= 100 * len(ups)
    assert len(set(shapes)) == 1, shapes
