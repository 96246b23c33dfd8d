"""Second oracle (SURVEY 8c, O2): the original program's OWN emitted kernels.  tests/golden/ref_gold.npz holds, for
every small parity case of oracle/build_ref.py, seeded samples of what its gold_<name> kernel (and, where Dist <= Halo,
its dr_<name> kernel) left in the buffers after the case's schedule (tests/golden/make_ref_gold.py).  Checks, bit for bit:
    reference gold_<name>  ==  CPU oracle  ==  product sweep (algebraic / single step)
and the product's data-reuse mode against the reference's dr_<name> and the reference's own 1e-13 bar."""
import os
import sys

import numpy as np
import pytest

from helpers import ROOT, max_rel, oracle_terms

sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
from make_ref_gold import cases, positions  # noqa: E402

pytestmark = pytest.mark.gpu
CASES = cases()
GOLDEN = np.load(os.path.join(ROOT, "tests", "golden", "ref_gold.npz"))


def test_golden_covers_every_case():
    assert sorted({k.split("/")[0] for k in GOLDEN.files}) == sorted(CASES) and len(CASES) == 13


@pytest.mark.parametrize("case", sorted(CASES))
def test_reference_gold_equals_oracle_equals_product(built, case):
    import torch
    import drstencil_b200 as drs
    from oracle import oracle
    stem, is3d, shape, iters, step, dist_opt = CASES[case]
    offs, coefs, halo = oracle_terms(stem, step)
    s_ = oracle.parse_stc(os.path.join(ROOT, "stc", stem + ".stc"), is3d)
    pts = oracle.compose(s_.points, step)
    _, dist = oracle.order_dist(pts, s_.dim, dist_opt)
    idx = positions(shape)
    at = lambda a: a.reshape(-1)[idx]
    sweeps = oracle.sweep_count(iters, step)
    a0 = oracle.rand_array(shape)
    # CPU oracle == reference gold kernel
    oa, ob = a0.copy(), np.zeros(shape)
    assert oracle.run(oa, ob, offs, coefs, halo, iters, step) == sweeps
    ga, gb = GOLDEN[case + "/gold_A"], GOLDEN[case + "/gold_B"]
    assert np.array_equal(at(oa), ga) and np.array_equal(at(ob), gb), "oracle != reference gold kernel"
    # reference dr_ kernel: the reference's own acceptance bar (common.hpp:53) against its gold.  With `--dist 2` on a
    # radius-1 cross stencil its dr_ kernel disagrees with its own gold by O(1) (Dist > Halo), which is why gold (not
    # dr_) is the canonical oracle; those cases have no dr_ record.
    assert (case + "/dr_A" in GOLDEN.files) == (dist <= halo)
    if dist <= halo:
        da = GOLDEN[case + "/dr_A"]
        assert max_rel(da, ga) <= 1e-12, "reference dr_ vs its own gold"
        # product in `--fuse reuse` mode (drs_reuse.cuh): the reference's own forward/backward evaluation -- against the
        # reference's dr_ kernel itself, bit for bit wherever that kernel is deterministic (no cross-thread forward set),
        # and against the oracle's restatement of the scheme
        st_r = drs.Stencil.from_file(os.path.join(ROOT, "stc", stem + ".stc")).set_size(shape, iters)
        plan_r = drs.Plan(st_r, drs.Knobs(step=step, fuse="reuse", dist=dist))
        A, B = torch.from_numpy(a0).cuda(), torch.zeros(shape, dtype=torch.float64, device="cuda")
        assert plan_r.run(A, B, iters) == sweeps
        plan_r.sync_check()
        got = A.cpu().numpy()
        part = oracle.partition(pts, s_.dim, dist)
        ra, rb = a0.copy(), np.zeros(shape)
        bufs = [ra, rb]
        for sw in range(sweeps):
            assert oracle.sweep_reuse(bufs[sw & 1], bufs[(sw & 1) ^ 1], pts, s_.dim, dist)
        assert np.array_equal(got, ra), "reuse mode != the oracle's restatement of the forward/backward scheme"
        if not part["forward_mid"] and not part["forward_fast"]:
            assert np.array_equal(at(got), da), "reuse mode != the reference's dr_ kernel"
        else:
            assert max_rel(at(got), da) <= 1e-12       # the reference's atomics may land in either order
        assert oracle.check_error(got, oa, halo)[0] <= 1e-12           # and its own acceptance bar against gold
    # product, literal composed operator -> bit-exact against the reference gold
    st = drs.Stencil.from_file(os.path.join(ROOT, "stc", stem + ".stc")).set_size(shape, iters)
    plan = drs.Plan(st, drs.Knobs(step=step, fuse="algebraic"))
    A, B = torch.from_numpy(a0).cuda(), torch.zeros(shape, dtype=torch.float64, device="cuda")
    assert plan.run(A, B, iters) == sweeps
    plan.sync_check()
    assert np.array_equal(A.cpu().numpy(), oa) and np.array_equal(at(A.cpu().numpy()), ga), "product != reference gold kernel"
    # product, temporal blocking (2D, step > 1) -> within 1e-12
    if step > 1 and not is3d:
        plan = drs.Plan(st, drs.Knobs(step=step))
        A, B = torch.from_numpy(a0).cuda(), torch.zeros(shape, dtype=torch.float64, device="cuda")
        plan.run(A, B, iters)
        plan.sync_check()
        assert max_rel(A.cpu().numpy(), oa) <= 1e-12
