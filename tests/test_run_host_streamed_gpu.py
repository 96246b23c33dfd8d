"""drs_run_host with the copy/sweep/copy phases overlapped by time skewing (capi.cpp:
run_blocks) must return exactly what the plain sequence returns: a sweep is a pure function
of its input array, so any block order that honours the dependencies is bit-identical."""
import numpy as np
import pytest

from helpers import oracle_run, stc_path

pytestmark = pytest.mark.gpu


def _plan(name, shape, **kn):
    import drstencil_b200 as drs
    st = drs.Stencil.from_file(stc_path(name)).set_size(shape)
    return drs.Plan(st, drs.Knobs(**kn))


def _host(shape, dtype, seed):
    import torch
    from oracle import oracle
    a = oracle.lcg_array(shape, np.float64, seed).astype(dtype)
    return torch.from_numpy(a).pin_memory()


CASES = [
    # name, shape, knobs, iterations, block thickness (slow-axis units)
    ("2d5pt_star", (300, 264), dict(), 10, 2),            # thinnest legal block (2 * Halo)
    ("2d5pt_star", (300, 264), dict(), 10, 37),           # does not divide the grid
    ("2d5pt_star", (300, 264), dict(), 60, 16),           # n * Halo > block: low blocks run empty
    ("2d9pt_box", (260, 520), dict(step=4), 24, 24),      # temporal depth 4, Halo 4
    ("2d9pt_box", (260, 520), dict(step=4), 24, 8),
    ("2d25pt_box", (190, 264), dict(dtype="f32"), 6, 20),
    ("2d9pt_star", (150, 200), dict(), 4, 5),
    ("3d7pt_star", (48, 40, 72), dict(), 10, 8),
    ("3d7pt_star", (48, 40, 72), dict(), 10, 2),
    ("3d7pt_star", (50, 70, 136), dict(step=2), 12, 10),  # fused 3D temporal kernel, Halo 2
    ("3d9pt_cross", (30, 24, 66), dict(), 4, 7),
]


@pytest.mark.parametrize("name,shape,kn,iters,block", CASES)
def test_streamed_equals_plain(built, name, shape, kn, iters, block):
    import drstencil_b200 as drs
    dtype = np.float32 if kn.get("dtype") == "f32" else np.float64
    plan = _plan(name, shape, **kn)
    assert plan.info.kernel_name.startswith("dr_")
    plain = _host(shape, dtype, 7)
    plan.set_host_block(-1)
    l0 = plan.launch_count
    plan.run_host(plain, None, iters)
    n = drs.sweep_count(iters, kn.get("step", 1))
    assert plan.launch_count - l0 == n
    streamed = _host(shape, dtype, 7)
    plan.set_host_block(block)
    l0 = plan.launch_count
    ms = plan.run_host(streamed, None, iters)
    assert ms > 0
    assert plan.launch_count - l0 > n, "the streamed path did not run"
    assert np.array_equal(streamed.numpy(), plain.numpy()), (name, shape, block)
    # a second call reuses the cleared second buffer
    again = _host(shape, dtype, 7)
    plan.run_host(again, None, iters)
    assert np.array_equal(again.numpy(), plain.numpy())


def test_streamed_against_the_oracle_and_after_an_explicit_b(built):
    """Depth 1 is bit-exact against the CPU oracle; a call with an explicit second buffer (plain
    path, dirties the ring of the device copy of B) must not leak into a later streamed call."""
    import torch
    shape = (200, 264)
    plan = _plan("2d5pt_star", shape)
    from oracle import oracle
    refA, _ = oracle_run("2d5pt_star", 1, shape, 10)
    a = torch.from_numpy(oracle.rand_array(shape)).pin_memory()
    plan.set_host_block(32)
    plan.run_host(a, None, 10)
    assert np.array_equal(a.numpy(), refA)
    a2 = torch.from_numpy(oracle.rand_array(shape)).pin_memory()
    b2 = torch.full(shape, 5.0, dtype=torch.float64).pin_memory()
    plan.run_host(a2, b2, 10)
    assert not np.array_equal(a2.numpy(), refA)       # B's ring of 5s reaches the result
    a3 = torch.from_numpy(oracle.rand_array(shape)).pin_memory()
    plan.run_host(a3, None, 10)
    assert np.array_equal(a3.numpy(), refA)


def test_streamed_auto_block_and_pageable_memory(built):
    """Engine-chosen blocks on a grid big enough to be cut (>= 2 blocks of 32 MiB), from pageable
    host memory (no overlap, same result)."""
    import torch
    shape = (4096, 4096)
    plan = _plan("2d5pt_star", shape)
    g = torch.Generator().manual_seed(3)
    x = torch.rand(shape, dtype=torch.float64, generator=g)
    plain, auto = x.clone(), x.clone()
    plan.set_host_block(-1)
    plan.run_host(plain, None, 10)
    plan.set_host_block(0)
    l0 = plan.launch_count
    plan.run_host(auto, None, 10)
    assert plan.launch_count - l0 > 10
    assert torch.equal(plain, auto)
