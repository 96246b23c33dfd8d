"""The streamed drs_run_host on plans with exact pair launches (csrc/core/host_schedule.hpp with a launch list of depths
1 and 2), checked WITHOUT a GPU: the step list the C ABI reports (Plan.host_schedule, HOST_PAIR records included) is
replayed with the CPU oracle standing in for the kernels, as test_host_schedule.py does for single sweeps.  A pair
launch is emulated as two oracle sweeps with the rings of drs_run's buffers (level 0: A's ring cells, level 1: B's),
storing only its range.  Device planes that were not uploaded yet are poisoned with NaN.  A restatement of the planner
with the naive slide R_k = level_k * Halo makes the replay fail: the test sees the hazard at the pair -> single step."""
import numpy as np
import pytest

import drstencil_b200 as drs
from drstencil_b200.presets import PRESETS
from helpers import oracle_terms, stc_path

UPLOAD, SWEEP, DOWNLOAD, PAIR = drs.HOST_UPLOAD, drs.HOST_SWEEP, drs.HOST_DOWNLOAD, drs.HOST_PAIR


def _plan(name, shape, block, pairs=True, **kn):
    st = drs.Stencil.from_file(stc_path(name)).set_size(shape)
    plan = drs.Plan(st, drs.Knobs(**kn))
    plan.set_host_block(block)
    if pairs:
        plan.set_pairs(True)
    return plan


def _ring_mask(shape, halo):
    m = np.ones(shape, dtype=bool)
    m[tuple(slice(halo, n - halo) for n in shape)] = False
    return m


def _replay(steps, order, host, offs, coefs, halo):
    """Executes the step list in `order` on emulated device buffers; `host` is updated in place."""
    from oracle import oracle
    dev = [np.full(host.shape, np.nan), np.zeros(host.shape)]     # A: nothing uploaded yet; B: cleared
    ring = _ring_mask(host.shape, halo)
    for i in order:
        kind, block, launch, lo, hi = steps[i]
        if kind == UPLOAD:
            dev[0][lo:hi] = host[lo:hi]
        elif kind == DOWNLOAD:
            host[lo:hi] = dev[0][lo:hi]
        else:
            src, dst = (dev[0], dev[1]) if launch & 1 else (dev[1], dev[0])
            if kind == PAIR:
                lv0 = src.copy()
                lv0[ring] = dev[0][ring]             # level 0's ring is A's (NaN where A is not uploaded yet)
                lv1 = dev[1].copy()                  # level 1's ring is B's
                oracle.sweep(lv0, lv1, offs, coefs, halo)
                src = lv1
            full = dst.copy()
            oracle.sweep(src, full, offs, coefs, halo)            # whole interior ...
            dst[lo:hi] = full[lo:hi]                              # ... of which the launch stores [lo, hi)
    return dev


def _orders(steps):
    """The two extreme interleavings the stream/event chain allows:
    lazy uploads + eager downloads (list order), eager uploads + downloads deferred to the end."""
    idx = list(range(len(steps)))
    ups = [i for i in idx if steps[i][0] == UPLOAD]
    dns = [i for i in idx if steps[i][0] == DOWNLOAD]
    mid = [i for i in idx if steps[i][0] in (SWEEP, PAIR)]
    return {"lazy-up/eager-down": idx, "eager-up/late-down": ups + mid + dns}


def _replay_matches(steps, name, shape, iters):
    """Both interleavings end with the plain schedule's host array and device buffers."""
    from oracle import oracle
    offs, coefs, halo = oracle_terms(name, 1)
    a0 = oracle.lcg_array(shape, np.float64, 5)
    refA, refB = a0.copy(), np.zeros(shape)
    oracle.run(refA, refB, offs, coefs, halo, iters, 1)
    for order in _orders(steps).values():
        host = a0.copy()
        dev = _replay(steps, order, host, offs, coefs, halo)
        if not (np.array_equal(host, refA) and np.array_equal(dev[0], refA) and np.array_equal(dev[1], refB)):
            return False
    return True


def _naive(steps, shape, halo, depths):
    """The planner restated with the slide R_k = level_k * Halo (no max term), on the same blocks."""
    slow = shape[0]
    edge = [s[3] for s in steps if s[0] == UPLOAD] + [slow]
    B, K = len(edge) - 1, len(depths)
    R = np.cumsum([0] + list(depths)) * halo

    def cut(b, k):
        if b <= 0:
            return halo
        if b >= B:
            return slow - halo
        return min(max(edge[b] - int(R[k]), halo), slow - halo)

    out = []
    for b in range(B):
        out.append((UPLOAD, b, 0, edge[b], edge[b + 1]))
        for k in range(1, K + 1):
            lo, hi = cut(b, k), cut(b + 1, k)
            if hi > lo:
                out.append((PAIR if depths[k - 1] == 2 else SWEEP, b, k, lo, hi))
        lo = 0 if b == 0 else cut(b, K)
        out.append((DOWNLOAD, b, 0, lo, max(lo, slow if b == B - 1 else cut(b + 1, K))))
    return out


CASES = [
    # name, shape, iterations, block (slow-axis units; 4 * Halo is the least the planner keeps)
    ("2d5pt_star", (60, 24), 6, 4),
    ("2d5pt_star", (61, 24), 8, 7),          # ragged remainder
    ("2d5pt_star", (90, 24), 10, 9),
    ("2d5pt_star", (40, 24), 30, 6),         # n * Halo > block thickness
    ("2d5pt_star", (260, 24), 100, 16),
    ("2d5pt_star", (9, 24), 6, 4),           # slow = 2 * S + 1: a thin remainder joins its predecessor
    ("2d5pt_star", (5, 24), 6, 4),           # slow extent just above one block
    ("2d9pt_star", (70, 20), 6, 8),          # radius 2
    ("2d9pt_star", (97, 20), 10, 8),
    ("2d9pt_star", (17, 20), 8, 8),          # radius 2, slow = 2 * S + 1
    ("2d25pt_box", (80, 24), 8, 11),         # radius 2
    ("3d7pt_star", (40, 10, 12), 8, 5),
    ("3d7pt_star", (33, 10, 12), 10, 4),
    ("3d7pt_star", (7, 10, 12), 6, 4),       # slow = S + 3
    ("3d9pt_cross", (40, 10, 12), 10, 8),    # radius 2
]


def _structure(steps, plan, name, shape, iters):
    halo, slow = plan.halo, shape[0]
    n = plan.pair_split(iters)
    pairs = n[0]
    depths = [2] * pairs + [1] * n[1]
    ups = [s for s in steps if s[0] == UPLOAD]
    assert ups[0][3] == 0 and ups[-1][4] == slow
    assert all(a[4] == b[3] for a, b in zip(ups, ups[1:]))
    assert min(u[4] - u[3] for u in ups) >= (4 if pairs else 2) * halo
    for k in range(1, len(depths) + 1):
        rng = sorted((lo, hi) for kind, b, kk, lo, hi in steps if kind in (SWEEP, PAIR) and kk == k)
        assert rng[0][0] == halo and rng[-1][1] == slow - halo, (k, rng)
        assert all(a[1] == b[0] for a, b in zip(rng, rng[1:])), (k, rng)
        kinds = {kind for kind, b, kk, lo, hi in steps if kind in (SWEEP, PAIR) and kk == k}
        assert kinds == {PAIR if depths[k - 1] == 2 else SWEEP}
    dn = [(lo, hi) for kind, b, kk, lo, hi in steps if kind == DOWNLOAD and hi > lo]
    assert dn[0][0] == 0 and dn[-1][1] == slow and all(a[1] == b[0] for a, b in zip(dn, dn[1:]))
    for b in {s[1] for s in steps}:
        assert sum(1 for s in steps if s[0] == PAIR and s[1] == b) <= pairs
    return depths


@pytest.mark.parametrize("name,shape,iters,block", CASES)
def test_pair_step_list_is_a_legal_order_of_the_plain_schedule(built, name, shape, iters, block):
    plan = _plan(name, shape, block)
    steps = plan.host_schedule(iters)
    assert steps, "expected the streamed path for this case"
    assert oracle_terms(name, 1)[2] == plan.halo
    _structure(steps, plan, name, shape, iters)
    assert _replay_matches(steps, name, shape, iters), (name, shape, iters, block)


@pytest.mark.parametrize("name,shape,block", [("2d5pt_star", (60, 24), 2), ("2d9pt_star", (70, 20), 4),
                                              ("3d7pt_star", (40, 10, 12), 5)])
@pytest.mark.parametrize("iters", [2, 4])
def test_no_pair_launch_below_six_sweeps_keeps_the_single_sweep_list(built, name, shape, block, iters):
    """pair_split(2) and pair_split(4) have no pair launch: the list is the one without set_pairs, record for record."""
    plain = _plan(name, shape, block, pairs=False).host_schedule(iters)
    paired = _plan(name, shape, block)
    assert paired.pair_split(iters)[0] == 0
    assert plain and paired.host_schedule(iters) == plain


def test_minimum_block_is_four_halos_with_pairs(built):
    """set_host_block below 4 * Halo is raised to it once the run has a pair launch; without pairs the floor stays
    2 * Halo."""
    plan = _plan("2d9pt_star", (70, 20), 1)
    ups = [s for s in plan.host_schedule(10) if s[0] == UPLOAD]
    assert min(u[4] - u[3] for u in ups) == 4 * plan.halo
    ups = [s for s in plan.host_schedule(4) if s[0] == UPLOAD]
    assert min(u[4] - u[3] for u in ups) == 2 * plan.halo


def test_naive_slide_fails_the_replay(built):
    """Negative control: the same blocks with R_k = level_k * Halo overwrite planes of B that the next block's last
    pair launch still reads; the replay must see it."""
    name, shape, iters = "2d5pt_star", (90, 24), 10
    plan = _plan(name, shape, 9)
    steps = plan.host_schedule(iters)
    depths = _structure(steps, plan, name, shape, iters)
    assert _replay_matches(steps, name, shape, iters)
    naive = _naive(steps, shape, plan.halo, depths)
    assert naive != steps
    assert not _replay_matches(naive, name, shape, iters)


def test_c5_streamed_run_has_pair_launches(built):
    """c5 at 1536^3 with the engine's own blocks: drs_run pairs by default (>= 1 GiB), so does the streamed run_host.
    Planner only: nothing is allocated."""
    path, kn = PRESETS["c5"]
    plan = drs.Plan(drs.Stencil.from_file(path), kn)
    pairs, singles = plan.pair_split(100)
    assert pairs > 0
    steps = plan.host_schedule(100)
    ups = [s for s in steps if s[0] == UPLOAD]
    assert 8 <= len(ups) <= 20
    assert min(u[4] - u[3] for u in ups) >= 4 * plan.halo
    for b in range(len(ups)):
        assert 0 < sum(1 for s in steps if s[0] == PAIR and s[1] == b) <= pairs
    assert {s[2] for s in steps if s[0] == PAIR} == set(range(1, pairs + 1))
    assert {s[2] for s in steps if s[0] == SWEEP} == set(range(pairs + 1, pairs + singles + 1))
