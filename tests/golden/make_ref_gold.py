#!/usr/bin/env python
"""Generates tests/golden/ref_gold.npz: for every small parity case of oracle/build_ref.py (the `p*` cases), the values
the original program's kernels left in A and B after the case's schedule, at SAMPLE seeded positions per array:

  <case>/gold_A, <case>/gold_B   its gold_<name> kernel (the canonical oracle)
  <case>/dr_A                    its dr_<name> kernel, for the cases with Dist <= Halo (above that the original's
                                 forward/backward scheme is not self-consistent and there is nothing to pin)

    python tests/golden/make_ref_gold.py

They are computed with the oracle's restatements (oracle.run for gold_, oracle.sweep_reuse for dr_), which the
original's emitted kernels, built by oracle/build_ref.py, matched bit for bit on every one of these cases
(tests/test_ref_gold_gpu.py; dr_ where it is deterministic, within 1e-12 elsewhere).  CPU only.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

SAMPLE = 2048


def cases():
    """{case: (stencil, is3d, shape, iterations, step, --dist option)} of the parity cases."""
    from oracle.build_ref import CASES
    out = {}
    for case, (stem, is3d, (L, M, N), iters, step, opts) in CASES.items():
        if case.startswith("p"):
            dist = int(opts[opts.index("--dist") + 1]) if "--dist" in opts else 0
            out[case] = (stem, is3d, (L, M, N) if is3d else (M, N), iters, step, dist)
    return out


def positions(shape):
    """The sampled flat positions of an array of this shape (sorted, seeded)."""
    n = int(np.prod(shape))
    return np.sort(np.random.default_rng(20251020).choice(n, min(n, SAMPLE), replace=False))


def operator(stem, is3d, step, dist):
    """(points, dim, offs, coefs, halo, Dist) of the composed operator."""
    from oracle import oracle
    s = oracle.parse_stc(os.path.join(ROOT, "stc", stem + ".stc"), is3d)
    pts = oracle.compose(s.points, step)
    offs, coefs = oracle.terms(pts)
    halo, d = oracle.order_dist(pts, s.dim, dist)
    return pts, s.dim, offs, coefs, halo, d


def main():
    from oracle import oracle
    out = {}
    for case, (stem, is3d, shape, iters, step, dist) in sorted(cases().items()):
        pts, dim, offs, coefs, halo, d = operator(stem, is3d, step, dist)
        idx = positions(shape)
        a0 = oracle.rand_array(shape)
        ga, gb = a0.copy(), np.zeros(shape)
        sweeps = oracle.run(ga, gb, offs, coefs, halo, iters, step)
        out[case + "/gold_A"] = ga.reshape(-1)[idx]
        out[case + "/gold_B"] = gb.reshape(-1)[idx]
        if d <= halo:
            bufs = [a0.copy(), np.zeros(shape)]
            for sw in range(sweeps):
                assert oracle.sweep_reuse(bufs[sw & 1], bufs[(sw & 1) ^ 1], pts, dim, d)
            out[case + "/dr_A"] = bufs[0].reshape(-1)[idx]
    path = os.path.join(HERE, "ref_gold.npz")
    np.savez_compressed(path, **out)
    print("wrote %s: %d arrays" % (path, len(out)))


if __name__ == "__main__":
    main()
