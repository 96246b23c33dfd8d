"""Exact-arithmetic parity of pair slabs on one GPU (exact_slabpair.py): every rank of a decomposition emulated with
Plan.sweep_pair / Plan.sweep against the global float64 reference, and one rank's drs_run_slab and drs_run against
passive neighbours -- local arrays against the reference restated for pairs, the neighbours' arrays plane by plane, the
flag words the rank signals, the launch counts.  test_exact_slabpair.py proves each case's preconditions on the CPU."""
import time

import numpy as np
import pytest

import exact_ops as X
import exact_slab as S
import exact_slabpair as SP

pytestmark = pytest.mark.gpu


def _dt(case):
    import torch
    return torch.float32 if case["dtype"] == "f32" else torch.float64


def _f64(t):
    import torch
    return t.to(torch.float64)


def _check(fails, cid):
    assert not fails, "%s: %s" % (cid, " | ".join(fails[:8]))


class Passive:
    """Rank g whose neighbours are SENTINEL-filled device arrays of their full local size; the rank's own flag words
    are released in advance, the words it signals are zeroed test memory."""

    def __init__(self, plan, g, gs, bufs, M, N, dtype):
        import torch
        self.g, self.gs = g, gs
        self.nb = {}
        for side, r in (("lower", g.lower), ("upper", g.upper)):
            if r is not None:
                shape = (gs[r].local_planes, M, N)
                self.nb[side] = (gs[r], [torch.full(shape, SP.SENTINEL, dtype=dtype, device="cuda") for _ in range(2)])
        self.my_flags = torch.full((2,), SP.RELEASED, dtype=torch.int64, device="cuda")
        self.words = {side: torch.zeros(2, dtype=torch.int64, device="cuda") for side in self.nb}
        lower = self.nb["lower"][1] if "lower" in self.nb else [0, 0]
        upper = self.nb["upper"][1] if "upper" in self.nb else [0, 0]
        plan.set_peers(bufs, lower, upper, self.nb["lower"][0].lo if "lower" in self.nb else 0,
                       self.nb["upper"][0].lo if "upper" in self.nb else 0)
        if self.nb:
            plan.set_flags(self.my_flags.data_ptr(), self.words["lower"].data_ptr() + 8 if "lower" in self.words else 0,
                           self.words["upper"].data_ptr() if "upper" in self.words else 0)

    def reset(self):
        for _, arrs in self.nb.values():
            for a in arrs:
                a.fill_(SP.SENTINEL)

    def slots(self):
        out = {}
        for side, w in self.words.items():
            v = w.tolist()
            mine, other = (v[1], v[0]) if side == "lower" else (v[0], v[1])
            assert other == 0, "%s neighbour: a slot this rank never writes holds %d" % (side, other)
            out[side] = mine
        return out

    def neighbour_fails(self, own, H):
        """Each neighbour buffer holds, in its deep ghost planes facing this rank, the lateral interior of this rank's
        2H boundary output planes of the matching buffer of `own`; SENTINEL everywhere else."""
        import torch
        g = self.g
        fails = []
        for side, (gn, arrs) in self.nb.items():
            a, b = SP.pushed_planes(g, side)
            shift = g.origin - gn.origin
            lat = (slice(H, own[0].shape[1] - H), slice(H, own[0].shape[2] - H))
            for k in (0, 1):
                want = torch.full_like(arrs[k], SP.SENTINEL, dtype=torch.float64)
                want[(slice(a + shift, b + shift),) + lat] = _f64(own[k][(slice(a, b),) + lat])
                fails += ["%s neighbour: " % side + m for m in S.compare(_f64(arrs[k]), want, gn, "AB"[k], H, 1)]
        return fails


def _inputs(case, gs, chunks, dt):
    import torch
    shape = (case["G"], case["M"], case["N"])
    dev = torch.empty(0, device="cuda")
    return S.global_input(shape, SP.impulses(shape, gs, chunks, SP.halo_of(case)), like=dev)


# ---- every rank emulated, launch by launch, against the global reference ------------------------------------------

@pytest.mark.parametrize("cid", [c["id"] for c in SP.EMULATED])
def test_emulated_ranks_exact(built, cid):
    case = SP.CASE_BY_ID[cid]
    op, H, n = X.OPS[case["op"]], SP.halo_of(case), case["sweeps"]
    gs = SP.geoms(case)
    plans = [SP.make_plan(case, g) for g in gs]
    chunks = {g.rank: p.info.chunk for g, p in zip(gs, plans)}
    assert plans[0].halo == H and SP.growth_ok(case)[0], cid
    assert all(p.slab_split(n) == SP.pair_split(n) for p in plans) and SP.pair_split(n)[0] > 0, cid
    A0, B0 = _inputs(case, gs, chunks, _dt(case))
    arrays = [[S.to_local(A0, g).to(_dt(case)), S.to_local(B0, g).to(_dt(case))] for g in gs]
    for r, (g, p) in enumerate(zip(gs, plans)):
        p.set_peers(arrays[r], arrays[r - 1] if g.lower is not None else [0, 0],
                    arrays[r + 1] if g.upper is not None else [0, 0],
                    gs[g.lower].lo if g.lower is not None else 0, gs[g.upper].lo if g.upper is not None else 0)
    for kind, src in SP.run_launches(n):
        for r, p in enumerate(plans):
            (p.sweep_pair if kind == "pair" else p.sweep)(arrays[r][src], arrays[r][src ^ 1])
    for p in plans:
        p.sync_check()
    ref = X.exact_run(op, 1, A0, B0, n)
    fails = []
    for r, g in enumerate(gs):
        for b in (0, 1):
            fails += S.compare(_f64(arrays[r][b]), S.to_local(ref[b], g), g, "AB"[b], H, chunks[r])
    _check(fails, cid)


# ---- drs_run_slab as one rank with passive neighbours; drs_run on the same plan ------------------------------------

@pytest.mark.parametrize("cid", [c["id"] for c in SP.RUN_SLAB])
def test_run_slab_passive_neighbours(built, cid):
    import torch
    case = SP.CASE_BY_ID[cid]
    op, H, n = X.OPS[case["op"]], SP.halo_of(case), case["sweeps"]
    gs = SP.geoms(case)
    g = gs[case["rank"]]
    plan = SP.make_plan(case, g)
    chunk = plan.info.chunk
    assert plan.halo == H and SP.growth_ok(case)[0], cid
    pairs, singles = plan.slab_split(n)
    assert (pairs, singles) == SP.pair_split(n) and pairs > 0 and plan.pair_split(n) == (0, n), cid
    A0, B0 = _inputs(case, gs, {g.rank: chunk}, _dt(case))
    init = [S.to_local(A0, g), S.to_local(B0, g)]
    bufs = [init[0].to(_dt(case), copy=True), init[1].to(_dt(case), copy=True)]
    P = Passive(plan, g, gs, bufs, case["M"], case["N"], _dt(case))
    ref = [init[0].clone(), init[1].clone()]
    signalled = []
    for call in range(2):
        l0 = plan.launch_count
        assert plan.run_slab(n) == n
        plan.sync_check()
        assert plan.launch_count - l0 == pairs + singles, (call, plan.launch_count - l0, pairs, singles)
        SP.schedule_ref(op, ref, 0, g, H, SP.run_launches(n))
        fails = []
        for b in (0, 1):
            fails += S.compare(_f64(bufs[b]), ref[b], g, "AB"[b], H, chunk)
        _check(fails, "%s after call %d" % (cid, call))
        _check(P.neighbour_fails(bufs, H), "%s after call %d" % (cid, call))
        # flag values count launches: the last launch of call c signals (c + 1) (p + s)
        signalled.append(P.slots())
        assert signalled[-1] == {side: (call + 1) * (pairs + singles) for side in P.words}, (call, signalled)
    # drs_run on the same plan is the loop of single sweeps, each pushing 2H planes, no flags
    for b in (0, 1):
        bufs[b].copy_(init[b])
    P.reset()
    l0 = plan.launch_count
    assert plan.run(bufs[0], bufs[1], n) == n
    plan.sync_check()
    assert plan.launch_count - l0 == n
    got = [b.clone() for b in bufs]
    got_nb = {side: [a.clone() for a in arrs] for side, (_, arrs) in P.nb.items()}
    for b in (0, 1):
        bufs[b].copy_(init[b])
    P.reset()
    for s in range(n):
        plan.sweep(bufs[s & 1], bufs[(s & 1) ^ 1])
    plan.sync_check()
    fails = []
    for b in (0, 1):
        fails += ["drs_run vs the sweep loop: " + m for m in S.compare(_f64(got[b]), _f64(bufs[b]), g, "AB"[b], H, chunk)]
        for side, (gn, arrs) in P.nb.items():
            fails += ["%s neighbour, drs_run vs the sweep loop: " % side + m
                      for m in S.compare(_f64(got_nb[side][b]), _f64(arrs[b]), gn, "AB"[b], H, chunk)]
    ref = X.exact_run(op, 1, init[0], init[1], n, slow=(g.out_lo, g.out_hi))
    for b in (0, 1):
        fails += ["sweep loop: " + m for m in S.compare(_f64(bufs[b]), ref[b], g, "AB"[b], H, chunk)]
    _check(fails + P.neighbour_fails(bufs, H), cid)
    assert P.slots() == signalled[-1], "drs_run signals nothing"
    torch.cuda.synchronize()


# ---- the timed configuration's launches: a middle rank of c5's N = 8 slab at full plane size ------------------------

def test_preset_slab_middle_rank(built):
    import gc
    import torch
    import drstencil_b200 as drs
    from drstencil_b200.presets import PRESETS
    from drstencil_b200.slab import SlabGeometry
    gc.collect()
    torch.cuda.empty_cache()
    t0 = time.time()
    spec = SP.PRESET_SLAB
    shape = X._stc_shape(PRESETS[spec["preset"]][0])
    stname, kn = X._preset_stencil(spec["preset"])
    opname = "star7neg"
    op = X.OPS[opname]
    H = X.halo_of(op, 1)
    gs = [SlabGeometry(shape[0], spec["world"], r, 2 * H, ring=H) for r in range(spec["world"])]
    g = gs[spec["rank"]]
    G, M, N = shape
    lshape = (g.local_planes, M, N)
    assert lshape == (196, 1536, 1536) and g.hi - g.lo == 192
    offs = list(op)
    plan = drs.Plan(drs.Stencil.from_points(offs, [op[o] for o in offs], lshape, 2, name=stname), kn)
    plan.set_slab_pairs(G, g.lo, g.hi)
    assert "drslabpair_" + stname in plan.slab_pair_source and "#define DRS_LD_HINT 1" in plan.slab_pair_source
    n = spec["sweeps_per_call"]
    pairs, singles = plan.slab_split(n)
    assert (pairs, singles) == (2, 2)
    assert X.growth_ok(dict(op=opname, dtype="f64", knobs=dict(step=1), sweeps=2 * n), np.array([X.IMPULSE]))[0]
    dev = torch.empty(0, device="cuda")
    imps = SP.impulses(shape, gs, {g.rank: plan.info.chunk}, H)
    bufs = [torch.empty(lshape, dtype=torch.float64, device="cuda") for _ in range(2)]

    def source(s0, s1):
        return S.global_input(shape, imps, like=dev, lo=g.origin + s0, hi=g.origin + s1)

    for z0, z1 in X.windows(lshape):
        a, b = source(z0, z1)
        bufs[0][z0:z1].copy_(a)
        bufs[1][z0:z1].copy_(b)
        del a, b
    P = Passive(plan, g, gs, bufs, M, N, torch.float64)
    for call in range(2):
        l0 = plan.launch_count
        assert plan.run_slab(n) == n
        plan.sync_check()
        assert plan.launch_count - l0 == pairs + singles
        assert P.slots() == {"lower": (call + 1) * (pairs + singles), "upper": (call + 1) * (pairs + singles)}
    t_run = time.time()
    launches = SP.run_launches(n) * 2
    reach = sum(2 if k == "pair" else 1 for k, _ in launches)
    fails = []
    for z0, z1 in X.windows(lshape):
        s0, s1 = max(0, z0 - reach), min(lshape[0], z1 + reach)
        a, b = source(s0, s1)
        refs = SP.schedule_ref(op, [X._f64(a), X._f64(b)], s0, g, H, launches)
        del a, b
        for k in (0, 1):
            want = refs[k][z0 - s0:z1 - s0]
            if not torch.equal(bufs[k][z0:z1], want):
                fails += S.compare(bufs[k][z0:z1], want, g, "AB"[k] + " planes from %d" % z0, H, plan.info.chunk)
        del refs
    _check(fails, "c5 pair slab middle rank")
    _check(P.neighbour_fails(bufs, H), "c5 pair slab middle rank")
    peak = torch.cuda.max_memory_allocated()
    print("c5 pair slab rank %d of %d, %d planes of %dx%d: %d launches, run %.1f s, check %.1f s, peak allocated %.2f GiB"
          % (g.rank, g.world, g.local_planes, M, N, len(launches), t_run - t0, time.time() - t_run, peak / 2 ** 30))
    del bufs, P, plan
    gc.collect()
    torch.cuda.empty_cache()
