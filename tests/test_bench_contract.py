"""bench.py's driver contract on the CPU: the reference arm (the CPU oracle port; the one leg that needs no
GPU) prints exactly one JSON line with the keys the driver reads, and the GPU arm refuses to run without a
device instead of falling back to anything.  On the GPU: --dump-outputs writes what the timed path computed."""
import json
import os
import subprocess
import sys

import pytest

from helpers import ROOT


def _bench(*args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + list(args), cwd=ROOT, env=e,
                          stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)


def test_reference_arm_line(built):
    r = _bench("--impl", "reference", "--steps", "1", "--warmup", "0", "--workload", "c1")
    assert r.returncode == 0, r.stderr[-800:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "GStencil/s" and d["unit"] == "GStencil/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert d["steps"] == 1 and d["warmup"] == 0 and d["n_gpus"] == 1 and d["gpu_launches"] == 0
    assert d["value"] > 0 and d["ms_per_step"] > 1000          # one step = a sample of about three seconds
    assert d["config"]["workload"].startswith("c1: 2d5pt_star fp64 4096^2")
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sub-grid 4096x4096" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "GStencil/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_uses_every_host_core_under_torchrun_env(built):
    """torch.distributed.run exports OMP_NUM_THREADS=1 to every rank; the CPU legs must not inherit that
    (round 1: the N > 1 reference arm ran on one core and inflated every N > 1 ratio ~15x)."""
    r = _bench("--impl", "reference", "--steps", "1", "--warmup", "0", "--workload", "c1", "--gpus", "2",
               env={"OMP_NUM_THREADS": "1", "RANK": "0", "WORLD_SIZE": "2", "LOCAL_RANK": "0"})
    assert r.returncode == 0, r.stderr[-800:]
    d = json.loads(r.stdout.strip())
    cb = d["cpu_baseline"]
    cores = len(os.sched_getaffinity(0))
    assert cb["host_cores"] == cores and cb["cores"] == cores, cb
    assert "warning" not in cb


def test_reference_arm_other_ranks_stay_silent(built):
    r = _bench("--impl", "reference", "--steps", "1", "--warmup", "0", "--workload", "c1", "--gpus", "2",
               env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_steps_must_be_positive(built):
    r = _bench("--impl", "reference", "--steps", "0", "--warmup", "0", "--workload", "c1")
    assert r.returncode != 0 and "--steps must be at least 1" in r.stderr and r.stdout.strip() == ""


def test_dump_outputs_whole_or_the_same_bounded_sample(tmp_path):
    """--dump-outputs: small arrays whole (shape and dtype kept), large ones as one fixed sample of flat positions."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    small = torch.arange(12, dtype=torch.float64).reshape(3, 4)
    big = torch.rand(bench.DUMP_POINTS + 12345, dtype=torch.float32)
    for d in ("one", "two"):
        bench.dump_outputs(str(tmp_path / d), {"A": small, "B": big})
    a, b = np.load(tmp_path / "one" / "A.npy"), np.load(tmp_path / "one" / "B.npy")
    assert a.dtype == np.float64 and np.array_equal(a, small.numpy())
    assert b.dtype == np.float32 and 0.6 * bench.DUMP_POINTS < b.size <= bench.DUMP_POINTS
    assert np.array_equal(b, np.load(tmp_path / "two" / "B.npy"))
    idx = np.unique(np.random.default_rng(20251020).integers(0, big.numel(), bench.DUMP_POINTS))
    assert np.array_equal(b, big.numpy()[idx])
    bench.dump_outputs(str(tmp_path / "half"), {"B": big}, bench.DUMP_POINTS // 2)
    assert np.load(tmp_path / "half" / "B.npy").size <= bench.DUMP_POINTS // 2


def test_gpu_arm_has_no_cpu_fallback(built):
    import torch
    if torch.cuda.is_available():
        return
    r = _bench("--steps", "1")
    assert r.returncode != 0 and "no CUDA device" in (r.stderr + r.stdout)
    assert r.stdout.strip() == ""


@pytest.mark.gpu
def test_dump_outputs_are_what_the_timed_path_computed(built, tmp_path):
    """bench.py --dump-outputs on c1 (2d5pt_star fp64 4096^2, 10 timesteps per step) == the same schedule run here
    through Plan.run on the same seeded input: W warm-up steps (at least 3) and K timed steps."""
    import numpy as np
    import torch
    import drstencil_b200 as drs
    from drstencil_b200.presets import PRESETS
    sys.path.insert(0, ROOT)
    import bench
    steps, warmup = 2, 3
    r = _bench("--steps", str(steps), "--warmup", str(warmup), "--workload", "c1", "--no-extras", "--no-parity",
               "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-800:]
    path, kn = PRESETS["c1"]
    plan = drs.Plan(drs.Stencil.from_file(path), kn)
    shape, timesteps = (4096, 4096), bench.WORKLOADS["c1"][1]
    A = torch.rand(shape, dtype=torch.float64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(0))
    A.mul_(10.0 ** (-min(290.0, bench.decades_per_step("c1", timesteps) * (steps + warmup) / 2 + 5)))
    B = torch.zeros_like(A)
    for _ in range(steps + warmup):
        plan.run(A, B, timesteps)
    plan.sync_check()
    idx = np.unique(np.random.default_rng(20251020).integers(0, A.numel(), bench.DUMP_POINTS))
    for name, t in (("A", A), ("B", B)):
        assert np.array_equal(np.load(tmp_path / (name + ".npy")), t.reshape(-1).cpu().numpy()[idx]), name
