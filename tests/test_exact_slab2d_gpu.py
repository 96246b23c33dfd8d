"""Exact-arithmetic parity of the 2D slab path on one GPU (exact_slab2d.py): every rank of a row decomposition emulated
with Plan.sweep against the global float64 reference, and one rank's drs_run_slab, drs_run_host_slab and drs_run
against passive neighbours -- local arrays against the frozen-ghost reference, the neighbours' arrays row by row, the
flag words the rank signals, the launch counts -- plus c2's shipped kernel as a middle rank against the plain kernel.
test_exact_slab2d.py proves each case's preconditions on the CPU."""
import numpy as np
import pytest

import exact_ops as X
import exact_slab as S
import exact_slab2d as S2

pytestmark = pytest.mark.gpu


def _dt(case):
    import torch
    return torch.float32 if case["dtype"] == "f32" else torch.float64


def _f64(t):
    import torch
    return t.to(torch.float64)


class Passive:
    """Rank g of a row decomposition whose neighbours are plain device arrays of their full local size, filled with
    SENTINEL; the rank's own flag words are released in advance, the words it signals are zeroed test memory."""

    def __init__(self, plan, g, gs, bufs, N, dtype, flags=True):
        import torch
        self.g, self.gs, self.bufs = g, gs, bufs
        self.nb = {}
        for side, r in (("lower", g.lower), ("upper", g.upper)):
            if r is not None:
                self.nb[side] = (gs[r], [torch.full((gs[r].local_planes, N), S.SENTINEL, dtype=dtype, device="cuda")
                                         for _ in range(2)])
        self.my_flags = torch.full((2,), S.RELEASED, dtype=torch.int64, device="cuda")
        self.words = {side: torch.zeros(2, dtype=torch.int64, device="cuda") for side in self.nb}
        lower = self.nb["lower"][1] if "lower" in self.nb else [0, 0]
        upper = self.nb["upper"][1] if "upper" in self.nb else [0, 0]
        plan.set_peers(bufs, lower, upper, self.nb["lower"][0].lo if "lower" in self.nb else 0,
                       self.nb["upper"][0].lo if "upper" in self.nb else 0)
        if flags and self.nb:
            plan.set_flags(self.my_flags.data_ptr(),
                           self.words["lower"].data_ptr() + 8 if "lower" in self.words else 0,
                           self.words["upper"].data_ptr() if "upper" in self.words else 0)

    def reset(self):
        for _, arrs in self.nb.values():
            for a in arrs:
                a.fill_(S.SENTINEL)

    def slots(self):
        out = {}
        for side, w in self.words.items():
            v = w.tolist()
            mine, other = (v[1], v[0]) if side == "lower" else (v[0], v[1])
            assert other == 0, "%s neighbour: a slot this rank never writes holds %d" % (side, other)
            out[side] = mine
        return out

    def neighbour_fails(self, own, H, chunk, init_push=False):
        """Each neighbour buffer holds, in the ghost rows facing this rank, the interior columns of this rank's
        boundary rows of the level in the matching buffer of `own`; SENTINEL everywhere else.  init_push:
        drs_run_host_slab copied the whole level-0 face rows into buffer A's ghosts, lateral ring included."""
        import torch
        g = self.g
        fails = []
        for side, (gn, arrs) in self.nb.items():
            for b in (0, 1):
                want = torch.full_like(arrs[b], S.SENTINEL, dtype=torch.float64)
                if side == "lower":
                    src, dst = slice(H, 2 * H), slice(gn.local_planes - H, gn.local_planes)
                else:
                    src, dst = slice(g.local_planes - 2 * H, g.local_planes - H), slice(0, H)
                lat = slice(None) if init_push and b == 0 else slice(H, own[b].shape[1] - H)
                want[dst, lat] = _f64(own[b][src, lat])
                fails += ["%s neighbour: " % side + m for m in S2.compare(_f64(arrs[b]), want, gn, "AB"[b], H, chunk)]
        return fails


def _local_inputs(case, g, gs, chunk, dt):
    import torch
    shape = (case["G"], case["N"])
    dev = torch.empty(0, device="cuda")
    A0, B0 = S.global_input(shape, S2.impulses(shape, gs, {g.rank: chunk}, S.ghost_of(case)), like=dev)
    la, lb = S.to_local(A0, g), S.to_local(B0, g)
    return [la.to(dt, copy=True), lb.to(dt, copy=True)], [la, lb]


def _check(fails, cid):
    assert not fails, "%s: %s" % (cid, " | ".join(fails[:8]))


# ---- every rank emulated, Plan.sweep with peer stores, against the global reference --------------------------------

@pytest.mark.parametrize("cid", [c["id"] for c in S2.EMULATED])
def test_emulated_ranks_exact(built, cid, monkeypatch):
    import torch
    case = S2.CASE_BY_ID[cid]
    X.set_env(case, monkeypatch)
    op, step, H, sweeps = X.OPS[case["op"]], S.step_of(case), S.ghost_of(case), case["sweeps"]
    gs = S.geoms(case)
    plans = [S2.make_plan(case, g) for g in gs]
    chunks = {g.rank: p.info.chunk for g, p in zip(gs, plans)}
    assert plans[0].halo == H and S.growth_ok(case)[0], cid
    shape = (case["G"], case["N"])
    dev = torch.empty(0, device="cuda")
    A0, B0 = S.global_input(shape, S2.impulses(shape, gs, chunks, H), like=dev)
    arrays = [[S.to_local(A0, g).to(_dt(case)), S.to_local(B0, g).to(_dt(case))] for g in gs]
    for r, (g, p) in enumerate(zip(gs, plans)):
        p.set_peers(arrays[r], arrays[r - 1] if g.lower is not None else [0, 0],
                    arrays[r + 1] if g.upper is not None else [0, 0],
                    gs[g.lower].lo if g.lower is not None else 0, gs[g.upper].lo if g.upper is not None else 0)
    for s in range(sweeps):
        for r, p in enumerate(plans):
            p.sweep(arrays[r][s & 1], arrays[r][(s & 1) ^ 1])
    for p in plans:
        p.sync_check()
    ref = X.exact_run(op, step, A0, B0, sweeps)
    fails = []
    for r, g in enumerate(gs):
        for b in (0, 1):
            fails += S2.compare(_f64(arrays[r][b]), S.to_local(ref[b], g), g, "AB"[b], H, chunks[r])
    _check(fails, cid)


# ---- drs_run_slab as one rank with passive neighbours --------------------------------------------------------------

@pytest.mark.parametrize("cid", [c["id"] for c in S2.RUN_SLAB])
def test_run_slab_passive_neighbours(built, cid):
    case = S2.CASE_BY_ID[cid]
    op, step, H = case["op"], S.step_of(case), S.ghost_of(case)
    gs = S.geoms(case)
    g = gs[case["rank"]]
    plan = S2.make_plan(case, g)
    chunk = plan.info.chunk
    assert plan.halo == H and S.growth_ok(case)[0], cid
    bufs, ref = _local_inputs(case, g, gs, chunk, _dt(case))
    P = Passive(plan, g, gs, bufs, case["N"], _dt(case))
    n, T = case["calls"], case["calls"] * step
    done = 0
    for what in ("run_slab", "run_slab", "sweeps", "run_slab"):
        l0 = plan.launch_count
        if what == "run_slab":
            assert plan.run_slab(T) == n
            k = n
            done += n
        else:
            plan.sweep(bufs[0], bufs[1])
            plan.sweep(bufs[1], bufs[0])
            k = 2
        plan.sync_check()
        assert plan.launch_count - l0 == k, (what, plan.launch_count - l0, k)
        ref = S.frozen_run(op, step, g, ref[0], ref[1], k)
        fails = []
        for b in (0, 1):
            fails += S2.compare(_f64(bufs[b]), ref[b], g, "AB"[b], H, chunk)
        _check(fails, "%s after %s" % (cid, what))
        _check(P.neighbour_fails(bufs, H, chunk), "%s after %s" % (cid, what))
        assert P.slots() == {side: done for side in P.words}, (what, P.slots(), done)


# ---- drs_run_host_slab as one rank with passive neighbours ---------------------------------------------------------

def _expected_slots(recs, sides, base):
    out = {}
    for side in sides:
        sig, init = (4, 16) if side == "lower" else (8, 32)
        vals = [r[2] + 1 for r in recs if r[5] & sig] + [1 for r in recs if r[5] & init]
        out[side] = base + max(vals)
    return out


@pytest.mark.parametrize("cid", [c["id"] for c in S2.HOST_SLAB])
def test_run_host_slab_passive_neighbours(built, cid):
    import torch
    case = S2.CASE_BY_ID[cid]
    op, step, H = case["op"], S.step_of(case), S.ghost_of(case)
    gs = S.geoms(case)
    g = gs[case["rank"]]
    plan = S2.make_plan(case, g)
    chunk = plan.info.chunk
    assert plan.halo == H and S.growth_ok(case)[0], cid
    units, up_skew = case["blocks"]
    plan.set_host_block(units)
    n, T = case["calls"], case["calls"] * step
    recs = plan.slab_schedule(T, bool(up_skew))
    assert recs, cid
    bufs, ref = _local_inputs(case, g, gs, chunk, _dt(case))
    P = Passive(plan, g, gs, bufs, case["N"], _dt(case))
    own = slice(H, g.local_planes - H)
    h_own = torch.empty(tuple(bufs[0][own].shape), dtype=_dt(case), pin_memory=True)
    h_own.copy_(bufs[0][own])
    bufs[0][own].fill_(-S.SENTINEL)         # the call uploads h_own over the device copy of the owned rows
    base = 0
    for call in range(2):
        plan.run_host_slab(h_own, T, bool(up_skew))
        ref = S.frozen_run(op, step, g, ref[0], ref[1], n)
        _check(S2.compare(_f64(h_own.cuda()), ref[0][own], g, "h_own", H, chunk), "%s call %d" % (cid, call))
        _check(P.neighbour_fails(ref, H, chunk, init_push=True), "%s call %d" % (cid, call))
        assert P.slots() == _expected_slots(recs, P.words, base), (call, P.slots(), recs)
        base += n + 1
    l0 = plan.launch_count
    assert plan.run_slab(T) == n
    plan.sync_check()
    assert plan.launch_count - l0 == n
    ref = S.frozen_run(op, step, g, ref[0], ref[1], n)
    fails = []
    for b in (0, 1):
        fails += S2.compare(_f64(bufs[b]), ref[b], g, "AB"[b], H, chunk)
    _check(fails, cid + " run_slab after the host calls")
    _check(P.neighbour_fails(bufs, H, chunk, init_push=True), cid + " run_slab after the host calls")
    assert P.slots() == {side: base + n for side in P.words}


# ---- drs_run on a slab plan equals the loop of drs_sweep on that plan ----------------------------------------------

@pytest.mark.parametrize("cid", [c["id"] for c in S2.RUN])
def test_run_on_slab_plan_is_the_sweep_loop(built, cid):
    case = S2.CASE_BY_ID[cid]
    op, step, H = case["op"], S.step_of(case), S.ghost_of(case)
    gs = S.geoms(case)
    g = gs[case["rank"]]
    plan = S2.make_plan(case, g)
    chunk = plan.info.chunk
    assert plan.halo == H and S.growth_ok(case)[0], cid
    bufs, init = _local_inputs(case, g, gs, chunk, _dt(case))
    P = Passive(plan, g, gs, bufs, case["N"], _dt(case), flags=False)
    T = case["sweeps"] * step
    l0 = plan.launch_count
    assert plan.run(bufs[0], bufs[1], T) == case["sweeps"]
    plan.sync_check()
    launches = plan.launch_count - l0
    got = [b.clone() for b in bufs]
    got_nb = {side: [a.clone() for a in arrs] for side, (_, arrs) in P.nb.items()}
    for b in (0, 1):
        bufs[b].copy_(init[b])
    P.reset()
    for s in range(case["sweeps"]):
        plan.sweep(bufs[s & 1], bufs[(s & 1) ^ 1])
    plan.sync_check()
    fails = []
    for b in (0, 1):
        fails += ["drs_run vs the sweep loop: " + m for m in S2.compare(_f64(got[b]), _f64(bufs[b]), g, "AB"[b], H, chunk)]
        for side, (gn, arrs) in P.nb.items():
            fails += ["%s neighbour, drs_run vs the sweep loop: " % side + m
                      for m in S2.compare(_f64(got_nb[side][b]), _f64(arrs[b]), gn, "AB"[b], H, chunk)]
    _check(fails, cid)
    ref = S.frozen_run(op, step, g, init[0], init[1], case["sweeps"])
    for b in (0, 1):
        fails += S2.compare(_f64(bufs[b]), ref[b], g, "AB"[b], H, chunk)
    _check(fails + P.neighbour_fails(bufs, H, chunk), cid)
    assert launches == case["sweeps"], launches


# ---- c2's shipped kernel as a middle rank: the slab entry against the plain kernel on the same local array ---------

def test_c2_middle_rank_matches_the_plain_kernel(built):
    """c2 (2d9pt_box, depth 4, factored scatter with a deferred scale) is not exact, but the slab entry evaluates every
    output with the same code as dr_: run_slab on a middle rank with frozen ghost rows equals the plain plan's run on
    the same local array bit for bit, both buffers, and the neighbours' ghost rows hold the boundary rows."""
    import torch
    import drstencil_b200 as drs
    from drstencil_b200.presets import PRESETS
    from drstencil_b200.slab import SlabGeometry
    spec = S2.C2_MIDDLE
    path, kn = PRESETS[spec["preset"]]
    st = drs.Stencil.from_file(path)
    M, N = st.shape
    H = drs.Plan(st, kn).halo
    gs = [SlabGeometry(M, spec["world"], r, H) for r in range(spec["world"])]
    g = gs[spec["rank"]]
    st.set_size((g.local_planes, N))
    slab, plain = drs.Plan(st, kn), drs.Plan(st, kn)
    slab.set_slab(M, g.lo, g.hi)
    assert "#define DRS_FACTORED 1" in slab.slab_source and "DRS_OUT_SCALE" in slab.slab_source
    assert (g.out_lo, g.out_hi) == (H, g.local_planes - H)        # the plain plan's output rows
    gen = torch.Generator(device="cuda").manual_seed(7)
    init = [torch.rand((g.local_planes, N), dtype=torch.float64, device="cuda", generator=gen) for _ in range(2)]
    bufs = [t.clone() for t in init]
    P = Passive(slab, g, gs, bufs, N, torch.float64)
    n = spec["sweeps_per_call"]
    for call in range(2):
        l0 = slab.launch_count
        assert slab.run_slab(n * kn.values["step"]) == n
        slab.sync_check()
        assert slab.launch_count - l0 == n and P.slots() == {"lower": (call + 1) * n, "upper": (call + 1) * n}
    ref = [t.clone() for t in init]
    assert plain.run(ref[0], ref[1], 2 * n * kn.values["step"]) == 2 * n
    plain.sync_check()
    fails = []
    for b in (0, 1):
        fails += S2.compare(bufs[b], ref[b], g, "AB"[b] + " vs dr_", H, slab.info.chunk)
    _check(fails, "c2 middle rank")
    _check(P.neighbour_fails(bufs, H, slab.info.chunk), "c2 middle rank")
