"""The streamed drs_run_host on plans with exact pair launches, bit for bit: the time-skewed blocks run drs_run's launch
sequence (pair launches, then two or four single sweeps) and must return exactly what the plain copy-sweep-copy sequence
returns on the same plan, what a loop of single sweeps (Plan.sweep) leaves in A, and -- for exact operators where
growth_ok allows -- the float64 reference exact_run.  test_host_pairs_schedule.py replays the same step lists on the
CPU."""
import numpy as np
import pytest

import drstencil_b200 as drs
import exact_ops as X
from drstencil_b200.presets import PRESETS

pytestmark = pytest.mark.gpu


def _plan(op, shape, dt, knobs=None, pairs=True):
    o = X.OPS[op]
    st = drs.Stencil.from_points(list(o), [o[k] for k in o], shape, len(shape), name="hostpair_" + op)
    plan = drs.Plan(st, drs.Knobs(**dict(knobs or {}, dtype=dt)))
    if pairs:
        plan.set_pairs(True)
    return plan


def _input(shape, dt, seed):
    rng = np.random.default_rng(seed)
    return rng.integers(-X.UMAX, X.UMAX + 1, size=shape).astype(np.float64 if dt == "f64" else np.float32)


def _host(a0, pinned):
    import torch
    t = torch.from_numpy(a0.copy())
    return t.pin_memory() if pinned else t


def _single_sweeps(plan, a0, n):
    """A after n single sweeps on the device from (a0, zeros), the second buffer run_host starts from."""
    import torch
    bufs = [torch.from_numpy(a0).cuda(), torch.zeros(a0.shape, dtype=torch.from_numpy(a0).dtype, device="cuda")]
    for s in range(n):
        plan.sweep(bufs[s % 2], bufs[(s + 1) % 2])
    plan.sync_check()
    return bufs[0].cpu().numpy()


def _check(plan, a0, T, block, op=None, pinned=True, calls=2):
    """Streamed run_host with pair launches against the plain sequence, the single-sweep loop and exact_run."""
    import torch
    n = drs.sweep_count(T, 1)
    pairs, singles = plan.pair_split(T)
    plain = _host(a0, pinned)
    plan.set_host_block(-1)
    assert plan.host_schedule(T) == []
    l0 = plan.launch_count
    plan.run_host(plain, None, T)
    assert plan.launch_count - l0 == pairs + singles
    plan.set_host_block(block)
    steps = plan.host_schedule(T)
    assert steps, "expected the streamed path"
    launches = sum(1 for s in steps if s[0] in (drs.HOST_SWEEP, drs.HOST_PAIR) and s[4] > s[3])
    assert (sum(1 for s in steps if s[0] == drs.HOST_PAIR) > 0) == (pairs > 0)
    for call in range(calls):            # the second call reuses the cleared ring of B
        got = _host(a0, pinned)
        l0 = plan.launch_count
        assert plan.run_host(got, None, T) > 0
        plan.sync_check()
        assert plan.launch_count - l0 == launches
        assert np.array_equal(got.numpy(), plain.numpy()), ("streamed vs plain", call, T, block)
    assert np.array_equal(plain.numpy(), _single_sweeps(plan, a0, n)), ("plain vs single sweeps", T)
    if op is not None and X.growth_ok(dict(op=op, dtype="f64" if a0.dtype == np.float64 else "f32", knobs={},
                                           sweeps=n), a0)[0]:
        ref = X.exact_run(X.OPS[op], 1, torch.from_numpy(a0), torch.zeros(a0.shape, dtype=torch.from_numpy(a0).dtype), n)
        assert np.array_equal(plain.numpy().astype(np.float64), ref[0].numpy()), ("vs exact_run", T)
    return pairs


@pytest.mark.parametrize("T,block", [(6, 4), (8, 4), (10, 37), (16, 16), (60, 16), (100, 24)])
def test_2d_star_f64(built, T, block):
    """2D fp64 star after set_pairs(True): minimum-thickness blocks (4 * Halo), a block that does not divide the grid,
    n * Halo beyond the block thickness."""
    shape = (300, 264)
    plan = _plan("star5", shape, "f64")
    assert _check(plan, _input(shape, "f64", T), T, block, op="star5") > 0


@pytest.mark.parametrize("T,block", [(2, 8), (4, 8), (6, 8), (8, 20), (10, 8)])
def test_2d_box25_f32(built, T, block):
    """2D fp32 box25 (Halo 2) after set_pairs(True); 2 and 4 timesteps make no pair launch."""
    shape = (190, 264)
    plan = _plan("box25", shape, "f32")
    assert (_check(plan, _input(shape, "f32", T), T, block, op="box25") > 0) == (T >= 6)


@pytest.mark.parametrize("T,block", [(6, 4), (8, 9), (10, 5)])
def test_3d_star_opt_in(built, T, block):
    """A 3D star below 1 GiB with set_pairs(True)."""
    shape = (70, 72, 136)
    plan = _plan("star7neg", shape, "f64")
    assert _check(plan, _input(shape, "f64", T), T, block, op="star7neg") > 0


def test_pageable_host_memory(built):
    """Pageable host memory: no overlap, same result."""
    shape = (300, 264)
    plan = _plan("star5", shape, "f64")
    assert _check(plan, _input(shape, "f64", 4), 10, 16, op="star5", pinned=False) > 0
    shape = (70, 72, 136)
    plan = _plan("star7neg", shape, "f64")
    assert _check(plan, _input(shape, "f64", 5), 8, 8, op="star7neg", pinned=False) > 0


@pytest.mark.parametrize("T", [6, 100])
def test_c4_size_default_rule(built, T):
    """c4's size and knobs (768^3 fp64, 3.6 GB per array): the default 1 GiB rule pairs without set_pairs, and so does
    the streamed run_host with the engine's own blocks."""
    path, kn = PRESETS["c4"]
    shape = drs.Plan(drs.Stencil.from_file(path), kn).stencil.shape
    o = X.OPS["star7neg"]
    plan = drs.Plan(drs.Stencil.from_points(list(o), list(o.values()), shape, 3, name="hostpair_c4"), kn)
    assert plan.pair_split(T)[0] > 0
    assert _check(plan, _input(shape, "f64", T), T, 0, calls=1) > 0
