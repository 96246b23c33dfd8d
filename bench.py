#!/usr/bin/env python
"""bench.py -- the driver's contract benchmark.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cX] [--dump-outputs DIR]

Metric (BASELINE.json): GStencil/s and achieved HBM GB/s (% of roofline) per stencil.
A "step" is one run of the reference's emitted host loop (codegen_2d.hpp:610-613) over one
synthetic grid: `for (t = 0; t < iterations; t += 2*step) { sweep(A,B); sweep(B,A); }`.

  Workload, every N: c5 = 3d7pt_star fp64 1536^3, 100 timesteps per step -- the one BASELINE.json
          configuration defined at 1/2/4/8 GPUs (it fits one B200: 2 x 27 GiB), so that the per-N
          values form one strong-scaling series.  N = 1 sweeps the whole grid on one GPU; N > 1
          slab-decomposes it along k: drs_run_slab, one launch per sweep, halo push and step flags
          fused into the sweep kernel over NVLink.
  N = 1   additionally reports every other configuration (c1-c4) in `per_config`, each timed for
          >= 1 s with its own clocks, roofline fraction and CPU baseline -- c2 (2d9pt_box fp64
          16384^2, temporal depth 4) is the temporally fused one.

`value`     device-resident throughput (inputs already in HBM), CUDA events, max over ranks.
`e2e`       the same step through the host-buffer C-ABI call (drs_run_host; N > 1: drs_run_host_slab)
            on pinned host memory: H2D of the grid, the schedule, D2H of the result inside the
            timed region, overlapped by time-skewed blocks.  `e2e.bound` = the three phases alone.
`parity`    checked in this very run, before timing: N = 1: the sweep kernel against the on-device
            gold kernel (bit for bit at depth 1, relative error at depth 2); N > 1: the slab run
            (same kernels, same protocol) against an undecomposed run of the same grid on each GPU.
`roofline`  dominant kernel: algorithmic bytes (2*sizeof(T) per grid point per launch, SURVEY 8d)
            / mean launch time, against MEASURED_PEAKS.json hbm_gbs (burst copy figure).
`cpu_baseline`  the CPU oracle (a port: the reference has no CPU loop) on ALL host cores (whatever
            OMP_NUM_THREADS says -- torchrun sets it to 1), on a bounded sample of the same workload.
`--impl reference`  the same oracle port, timed as the reference arm (rank 0 only).
`--dump-outputs DIR`  after the timed steps, the buffers the timed call hands back (A, where the result lands, and B)
            as DIR/<name>.npy in their own dtype: whole up to 2^21 / N elements, else the same seeded sample of
            2^21 / N flat positions on every run (N ranks: 32 MiB in all at most).  The inputs depend only on the
            arguments, so two builds can be compared output for output.

The tree is only read: kernels compiled at run time go to a temporary cache seeded with the cubins build() left.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (preset, timesteps per step, description)
    "c1": ("c1", 10, "2d5pt_star fp64 4096^2, 10 timesteps"),
    "c2": ("c2", 128, "2d9pt_box fp64 16384^2, temporal fusion depth 4, 128 timesteps"),
    "c3": ("c3", 8, "2d25pt_box fp32 16384^2, 8 timesteps"),
    "c4": ("c4", 16, "3d7pt_star fp64 768^3, k-streaming, 16 timesteps"),
    "c5": ("c5", 100, "3d7pt_star fp64 1536^3 slab-decomposed along k, 100 timesteps"),
    "c4t2": ("c4t2", 16, "EXTRA (not in BASELINE.json): 3d7pt_star fp64 768^3 with in-kernel temporal depth 2, 16 timesteps"),
    "c5t2": ("c5t2", 20, "EXTRA: c5 (3d7pt_star fp64 1536^3) with in-kernel temporal depth 2, 20 timesteps"),
    "c1t2": ("c1t2", 20, "EXTRA: c1 (2d5pt_star fp64 4096^2) with in-kernel temporal depth 2, 20 timesteps"),
    "c3t2": ("c3t2", 8, "EXTRA: c3 (2d25pt_box fp32 16384^2) with in-kernel temporal depth 2, 8 timesteps"),
}


def host_cores():
    """Cores this process may run on -- NOT the OpenMP default, which torchrun pins to 1."""
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """Samples SM clock and throttle reasons with NVML while the timed region runs."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                 "hw_power_brake_slowdown": 0x80, "sync_boost": 0x10}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop.wait(0.05)

    def start(self):
        if self.nv:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join()
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# sum of the coefficients of each workload's base operator: a field of positive values grows by about this
# factor per timestep (SURVEY.md appendix E), which bounds how many timesteps stay inside the floating range
SUM_COEF = {"c1": 1.1, "c2": 1.5, "c3": 2.38, "c4": 1.5, "c5": 1.5, "c4t2": 1.5, "c5t2": 1.5, "c1t2": 1.1, "c3t2": 2.38}


def decades_per_step(wl, timesteps):
    import math
    return math.log10(SUM_COEF[wl]) * timesteps


def renormalise(A, target, group=False):
    """A *= target / max|A| (the same factor on every rank): keeps long runs finite.  Data-independent kernels:
    only NaN / Inf / all-zero fields would change the timing, and this is what prevents them."""
    import torch
    m = A.abs().max()
    if group:
        torch.distributed.all_reduce(m, op=torch.distributed.ReduceOp.MAX)
    m = float(m)
    if m > 0 and m == m and m != float("inf"):
        A.mul_(target / m)


def interior_points(shape, halo):
    n = 1
    for d in shape:
        n *= max(0, d - 2 * halo)
    return n


def all_points(shape):
    n = 1
    for d in shape:
        n *= d
    return n


def time_steps(plan, A, B, timesteps, steps, warmup):
    """K timed steps of the emitted host loop on device-resident buffers -> (seconds, launches)."""
    import torch
    for _ in range(warmup):
        plan.run(A, B, timesteps)
    plan.sync_check()
    l0 = plan.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        plan.run(A, B, timesteps)
    e1.record()
    plan.sync_check()
    return e0.elapsed_time(e1) * 1e-3, plan.launch_count - l0


DUMP_POINTS = 1 << 21


def dump_outputs(out_dir, arrays, points=DUMP_POINTS):
    """{name: tensor} -> out_dir/<name>.npy: the whole array up to `points` elements, else the values at one fixed,
    seeded set of `points` flat positions (sorted), the same on every run."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        n = t.numel()
        if n <= points:
            host = t.cpu().numpy()
        else:
            idx = np.unique(np.random.default_rng(20251020).integers(0, n, points))
            host = t.reshape(-1)[torch.from_numpy(idx).to(t.device)].cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), host)


def private_jit_cache():
    """Points the engine's kernel cache at a new temporary directory that links the cubins build() left in
    drstencil_b200/_jitcache/, so that kernels compiled during the run are written there and not into the tree."""
    import tempfile
    import drstencil_b200 as drs
    tmp = tempfile.mkdtemp(prefix="drs_bench_jitcache_")
    src = os.path.join(ROOT, "drstencil_b200", "_jitcache")
    if os.path.isdir(src):
        for f in os.listdir(src):
            if f.endswith(".cubin"):
                os.symlink(os.path.join(src, f), os.path.join(tmp, f))
    drs.lib().drs_set_cache_dir(tmp.encode())
    return tmp


# ---------------------------------------------------------------------------------------------
# CPU legs (the only code in this file that touches oracle/)
# ---------------------------------------------------------------------------------------------

class CpuSample:
    """The oracle port on all host cores over a bounded sample of a workload: the composed operator
    of the workload (gold restatement) swept over a sub-grid with the workload's full plane / row
    size, so that the cache behaviour per plane is the real one; only the slow axis is cut."""

    def __init__(self, workload):
        import numpy as np
        from oracle import oracle
        import drstencil_b200 as drs
        from drstencil_b200.presets import PRESETS
        self.oracle = oracle
        self.workload = workload
        path, kn = PRESETS[WORKLOADS[workload][0]]
        is3d = os.path.basename(path)[3:].startswith("3d")
        s = oracle.parse_stc(path, is3d)
        self.step = kn.step
        pts = oracle.compose(s.points, self.step)
        self.offs, self.coefs = oracle.terms(pts)
        self.halo, _ = oracle.order_dist(pts, s.dim)
        dtype = np.float32 if kn.dtype == drs.F32 else np.float64
        # every host core, whatever OMP_NUM_THREADS says (torch.distributed.run exports OMP_NUM_THREADS=1)
        self.host_cores = host_cores()
        oracle.set_threads(self.host_cores)
        # ~3.5 GiB per array at most: 192 planes of c5, 4096 rows of the 16384-wide 2D grids
        self.shape = (min(s.L, 192), s.M, s.N) if is3d else (min(s.M, 4096), s.N)
        self.a = oracle.lcg_array(self.shape, dtype, 1)
        self.b = oracle.lcg_array(self.shape, dtype, 2)
        oracle.sweep(self.a, self.b, self.offs, self.coefs, self.halo)     # warm-up / first touch
        self.cores = oracle.lib().drs_oracle_threads()

    def run(self, budget_s):
        """Sweeps for about budget_s seconds -> (GStencil/s over the sample, seconds, sweeps)."""
        used, sweeps = 0.0, 0
        while used < budget_s or sweeps < 2:
            t0 = time.perf_counter()
            self.oracle.sweep(self.a, self.b, self.offs, self.coefs, self.halo)
            used += time.perf_counter() - t0
            sweeps += 1
            self.a, self.b = self.b, self.a
            if sweeps % 8 == 0:       # sum of coefficients > 1: keep the values finite
                self.a *= 1e-3
        return interior_points(self.shape, self.halo) * self.step * sweeps / used / 1e9, used, sweeps

    def describe(self, sweeps, seconds):
        return ("%s sub-grid %s (full-size planes, slow axis cut), composed %d-point operator (gold restatement, "
                "%d timesteps per sweep), %d sweeps in %.1f s" % (self.workload, "x".join(map(str, self.shape)),
                                                                   len(self.coefs), self.step, sweeps, seconds))


def cpu_baseline(workload, budget_s=12.0):
    """bench.py's cpu_baseline object: about budget_s seconds of CPU work."""
    cs = CpuSample(workload)
    gst, used, sweeps = cs.run(budget_s)
    out = {"value": gst, "unit": "GStencil/s", "cores": cs.cores, "host_cores": cs.host_cores, "kind": "port",
           "sample": cs.describe(sweeps, used), "seconds_per_sweep": used / sweeps}
    if cs.cores < cs.host_cores:
        out["warning"] = "OpenMP used fewer threads than the host has cores"
    return out


def run_reference(args, rank):
    """Reference arm: the CPU oracle port (the reference ships no CPU loop and its emitted CUDA
    is not a CPU implementation), all host threads; each step is a bounded sample (~3 s of sweeps)
    of the workload, W warm-up steps, K timed steps."""
    if rank != 0:
        return None
    wl = args.workload or "c5"
    cs = CpuSample(wl)
    for _ in range(args.warmup):
        cs.run(3.0)
    vals, secs, sweeps = [], 0.0, 0
    for _ in range(args.steps):
        v, t, n = cs.run(3.0)
        vals.append(v)
        secs += t
        sweeps += n
    v = interior_points(cs.shape, cs.halo) * cs.step * sweeps / secs / 1e9
    base = {"value": v, "unit": "GStencil/s", "cores": cs.cores, "host_cores": cs.host_cores, "kind": "port",
            "sample": cs.describe(sweeps, secs), "seconds_per_sweep": secs / sweeps, "per_step": vals}
    if cs.cores < cs.host_cores:
        base["warning"] = "OpenMP used fewer threads than the host has cores"
    preset, timesteps, desc = WORKLOADS[wl]
    return {"impl": "reference", "metric": "GStencil/s", "value": v, "unit": "GStencil/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": secs / max(1, args.steps) * 1e3,
            "higher_is_better": True, "scaling": "strong" if wl == "c5" else "weak", "vs_baseline": None,
            "dtype": "f64" if wl not in ("c3", "c3t2") else "f32", "data": "synthetic",
            "config": {"workload": "%s: %s" % (wl, desc), "note": "CPU port of the reference's gold expression "
                       "(the reference has no CPU implementation); each step = one bounded sample of ~3 s"},
            "cpu_baseline": base, "gpu_launches": 0,
            "e2e": {"value": v, "unit": "GStencil/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


# ---------------------------------------------------------------------------------------------
# the reference's own emitted dr_ kernels (oracle/_ref), for context
# ---------------------------------------------------------------------------------------------

def reference_gpu_kernel(workload):
    """The reference's own emitted dr_ kernel on this GPU: the best configuration its search space produced on
    B200 for this workload (oracle/tune_ref.py, table in profiles/r02_ref_tune.json), re-timed here."""
    import ctypes
    meta_p = os.path.join(ROOT, "oracle", "_ref", "cases.json")
    if not os.path.exists(meta_p):
        return None
    allmeta = json.load(open(meta_p))
    case = None
    for c in ("best_" + workload, "full_" + workload):
        if c in allmeta and os.path.exists(os.path.join(ROOT, "oracle", "_ref", allmeta[c]["so"])):
            case = c
            break
    if case is None:
        return None
    meta = allmeta[case]
    try:
        lib = ctypes.CDLL(os.path.join(ROOT, "oracle", "_ref", meta["so"]))
        lib.drs_ref_time.restype = ctypes.c_float
        lib.drs_ref_time.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int]
        ms = lib.drs_ref_time(1, 20, 3) / 20
        if ms <= 0:
            return None
        halo = meta["step"] * 1
        shape = (meta["L"], meta["M"], meta["N"]) if meta["is3d"] else (meta["M"], meta["N"])
        return {"value": interior_points(shape, halo) * meta["step"] / (ms * 1e-3) / 1e9, "unit": "GStencil/s",
                "ms_per_sweep": ms,
                "tuned": case.startswith("best_"),
                "kernel": "dr_%s emitted by the reference generator (%s), nvcc sm_100a%s"
                          % (meta["stencil"], " ".join(meta["options"]),
                             "; best of the reference's own search space on B200 (profiles/r02_ref_tune.json)"
                             if case.startswith("best_") else "; hand-picked options, NOT tuned")}
    except Exception as e:   # context only
        return {"error": str(e)[:200]}


# ---------------------------------------------------------------------------------------------
# parity, checked in the bench run itself
# ---------------------------------------------------------------------------------------------

def _rel_errors(x, ref, floor_frac=1e-6):
    """(max |x - ref| / max |ref|, max pointwise |x - ref| / max(|ref|, floor)), floor = floor_frac * max |ref|."""
    import torch
    d = (x - ref).abs()
    scale = float(ref.abs().max())
    if scale == 0.0:
        return float(d.max()), float(d.max())
    pw = d / torch.clamp(ref.abs(), min=floor_frac * scale)
    return float(d.max()) / scale, float(pw.max())


def parity_single():
    """N = 1: the shipped c5 kernel configuration (and the fused temporal one) against the on-device gold
    kernel -- the naive one-thread-per-point evaluation of the composed operator (K5's stand-in) -- over the
    reference's schedule on a grid of several waves."""
    import torch
    import drstencil_b200 as drs
    from drstencil_b200.presets import PRESETS
    out = {"against": "gold_<name> on the device (one thread per point, composed operator, gold term order)", "cases": []}
    ok = True
    shape, timesteps = (96, 384, 512), 8
    for label, kn, exact in (("c5 preset, depth 1", PRESETS["c5"][1], True), ("depth 2 (fused temporal kernel)", drs.Knobs(step=2), False)):
        st = drs.Stencil.from_file(PRESETS["c5"][0]).set_size(shape)
        plan = drs.Plan(st, kn)
        g = torch.Generator(device="cuda").manual_seed(7)
        A0 = torch.rand(shape, dtype=torch.float64, device="cuda", generator=g)
        A, B = A0.clone(), torch.zeros_like(A0)
        n = plan.run(A, B, timesteps)
        Ag, Bg = A0.clone(), torch.zeros_like(A0)
        plan.gold_run(Ag, Bg, timesteps)
        plan.sync_check()
        rel, pw = _rel_errors(A, Ag)
        same = bool(torch.equal(A, Ag))
        good = same if exact else (rel <= 1e-12 and pw <= 1e-11)
        ok = ok and good
        out["cases"].append({"case": label, "grid": list(shape), "sweeps": n, "bit_exact": same, "max_rel": rel,
                             "max_pointwise_rel": pw, "bar": "bit-exact" if exact else "max_rel <= 1e-12", "ok": good})
    out["ok"] = ok
    return out


def parity_slab(rank, world, halo):
    """N > 1: the slab-decomposed run (same kernel knobs, same exchange protocol as the timed run) against the
    undecomposed run of the same global grid on this rank's own GPU; every rank compares its owned planes."""
    import torch
    import torch.distributed as dist
    import drstencil_b200 as drs
    from drstencil_b200.presets import PRESETS
    from drstencil_b200.slab import GpuSlab
    path = PRESETS["c5"][0]
    out = {"against": "the undecomposed single-GPU run of the same global grid (each rank, its own planes)", "cases": []}
    ok = True
    shape, timesteps = (40 * world, 384, 512), 24
    L, M, N = shape
    g = torch.Generator(device="cuda")

    def plane(zg):
        g.manual_seed(4321 + zg)
        return torch.rand((M, N), dtype=torch.float64, device="cuda", generator=g)

    for label, kn in (("c5 preset, depth 1", PRESETS["c5"][1]), ("depth 2 (fused temporal kernel)", drs.Knobs(step=2))):
        st = drs.Stencil.from_file(path).set_size(shape)
        plan = drs.Plan(st, kn)
        A = torch.stack([plane(z) for z in range(L)])
        B = torch.zeros_like(A)
        n = plan.run(A, B, timesteps)
        plan.sync_check()
        slab = GpuSlab(path, kn, rank, world, halo=halo, global_shape=shape)
        slab.fill(plane)
        slab.run(timesteps // 2 if (timesteps // 2) % (2 * kn.step) == 0 else timesteps)
        if (timesteps // 2) % (2 * kn.step) == 0:
            slab.run(timesteps // 2)            # two calls: the flag values carry over
        slab.plan.sync_check()
        mine, ref = slab.owned(0), A[slab.geom.lo:slab.geom.hi]
        same = bool(torch.equal(mine, ref))
        rel, pw = _rel_errors(mine, ref)
        res = {"device": (same, rel, pw)}
        # the host-buffer path (drs_run_host_slab) on the same grid
        if halo == "p2p":
            try:
                h = torch.stack([plane(z) for z in range(slab.geom.lo, slab.geom.hi)]).cpu().pin_memory()
                slab.fill(plane)                 # B's ring back to zeros, flags untouched
                slab.plan.set_host_block(8)      # several blocks even on this small grid
                slab.run_host(h, timesteps)
                hd = h.cuda()
                r2, p2 = _rel_errors(hd, ref)
                res["host"] = (bool(torch.equal(hd, ref)), r2, p2)
            except Exception as e:
                res["host"] = (False, float("inf"), float("inf"))
                res["host_error"] = str(e)[:200]
        flat = []
        for key in ("device", "host"):
            s_, r_, p_ = res.get(key, (True, 0.0, 0.0))
            flat += [1.0 if s_ else 0.0, r_, p_]
        t = torch.tensor(flat, device="cuda", dtype=torch.float64)
        tmin, tmax = t.clone(), t.clone()
        dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        case = {"case": label, "grid": list(shape), "sweeps": n, "ranks": world,
                "slab_vs_single": "bit-exact" if tmin[0] > 0 else "MISMATCH", "max_rel": float(tmax[1]),
                "max_pointwise_rel": float(tmax[2]), "ok": bool(tmin[0] > 0)}
        if "host" in res:
            case["host_path_vs_single"] = "bit-exact" if tmin[3] > 0 else "MISMATCH"
            case["host_path_max_rel"] = float(tmax[4])
            case["host_ok"] = bool(tmin[3] > 0)
            if "host_error" in res:
                case["host_error"] = res["host_error"]
        ok = ok and case["ok"]
        out["cases"].append(case)
        slab.close()
        del A, B, plan
        torch.cuda.empty_cache()
    out["ok"] = ok
    out["slab_vs_single"] = "bit-exact" if ok else "MISMATCH"
    out["max_rel"] = max(c["max_rel"] for c in out["cases"])
    out["host_path_ok"] = all(c.get("host_ok", False) for c in out["cases"])
    return out


# ---------------------------------------------------------------------------------------------
# GPU legs
# ---------------------------------------------------------------------------------------------

def run_single(args, rank, world):
    import torch
    import drstencil_b200 as drs
    from drstencil_b200.presets import PRESETS
    wl = args.workload or "c5"
    preset, timesteps, desc = WORKLOADS[wl]
    path, kn = PRESETS[preset]
    if wl == "c5" and args.depth > 1:
        kn = drs.Knobs(step=args.depth)
        desc += " [temporal depth %d]" % args.depth
    parity = parity_single() if not args.no_parity else None
    st = drs.Stencil.from_file(path)
    plan = drs.Plan(st, kn)
    shape = st.shape
    dtype = torch.float32 if kn.dtype == drs.F32 else torch.float64
    esize = 4 if kn.dtype == drs.F32 else 8
    g = torch.Generator(device="cuda").manual_seed(rank)
    A = torch.rand(shape, dtype=dtype, device="cuda", generator=g)
    # sum of coefficients > 1: start low enough that (K + W) * timesteps updates stay inside the floating range
    total_decades = decades_per_step(wl, timesteps) * (args.steps + args.warmup)
    limit = 290.0 if dtype == torch.float64 else 36.0
    if total_decades > 2 * limit:
        sys.exit("bench.py: %d steps of %d timesteps overflow %s (growth 10^%.0f): use fewer --steps"
                 % (args.steps + args.warmup, timesteps, "fp64" if esize == 8 else "fp32", total_decades))
    A.mul_(10.0 ** (-min(limit, total_decades / 2 + 5)))
    B = torch.zeros_like(A)
    sampler = ClockSampler(torch.cuda.current_device())
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()
    sampler.start()
    secs, launches = time_steps(plan, A, B, timesteps, args.steps, args.warmup)
    clocks = sampler.stop()
    if args.dump_outputs:
        suffix = "_rank%d" % rank if world > 1 else ""
        dump_outputs(args.dump_outputs, {"A" + suffix: A, "B" + suffix: B}, DUMP_POINTS // world)
    data_finite = bool(torch.isfinite(A).all()) and float(A.abs().max()) > 0
    info = plan.info
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([secs], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        secs = float(t)
    sweeps_per_step = drs.sweep_count(timesteps, kn.step)
    upd = interior_points(shape, info.halo) * sweeps_per_step * kn.step   # stencil updates per step
    value = world * upd * args.steps / secs / 1e9
    peak, peak_src = measured_peak()
    alg_bytes = all_points(shape) * 2 * esize
    ach = alg_bytes / (secs / launches) / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        # keyed by workload (tools/make_profiles.py); --depth n swaps the kernel, for which there is no capture
        traffic = json.load(open(tp)).get(wl if kn.step == PRESETS[preset][1].step else "")
    line = {
        "metric": "GStencil/s", "value": value, "unit": "GStencil/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": secs / args.steps * 1e3, "higher_is_better": True,
        "scaling": "strong" if wl == "c5" else "weak", "vs_baseline": None,
        "dtype": "f32" if kn.dtype == drs.F32 else "f64", "data": "synthetic",
        "config": {"workload": "%s: %s" % (wl, desc), "grid": list(shape), "timesteps_per_step": timesteps,
                   "sweeps_per_step": sweeps_per_step, "temporal_depth": kn.step, "kernel": info.kernel_name,
                   "knobs": repr(kn),
                   "tile": {"warps_per_cta": info.warps_per_cta, "tile_x": info.tile_x, "chunk": info.chunk,
                            "stages": info.stages, "regs": info.regs_per_thread, "smem": info.smem_bytes},
                   "l2": "inputs larger than L2 (2 x %.2f GiB per sweep vs 126 MB)" % (alg_bytes / 2 / 2 ** 30),
                   "replicas": world if world > 1 else None},
        "gpu_launches": launches,
        "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                     "traffic": traffic, "peak_source": peak_src, "kernel": info.kernel_name,
                     "algorithmic_bytes_per_launch": alg_bytes, "launch_ms": secs / launches * 1e3,
                     "gstencil_roofline": peak / (2 * esize) * kn.step},
        "clocks": clocks,
        "data_finite": data_finite,
        "parity": parity,
    }
    # ---- e2e: the host-buffer entry point (H2D + schedule + D2H in the timed region) ----
    if rank == 0 or world > 1:
        del A, B
        torch.cuda.empty_cache()
        pinned = True
        try:
            hA = torch.empty(shape, dtype=dtype, pin_memory=True)
        except RuntimeError:
            pinned = False
            hA = torch.empty(shape, dtype=dtype)
        hA.fill_(0.5e-100)
        e2e_steps = 2 if all_points(shape) * esize > 8 * 2 ** 30 else max(2, min(args.steps, 5))
        plan.run_host(hA, None, timesteps)               # warm (allocates the device pair)
        dev_ms = 0.0
        for _ in range(e2e_steps):
            dev_ms += plan.run_host(hA, None, timesteps)
        e_secs = dev_ms * 1e-3
        if world > 1:
            import torch.distributed as dist
            t = torch.tensor([e_secs], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e_secs = float(t)
        nbytes = all_points(shape) * esize
        # the same call with the overlap switched off (copy, sweep, copy in sequence), for reference
        plan.set_host_block(-1)
        plain_ms = plan.run_host(hA, None, timesteps)
        plan.set_host_block(0)
        # the three phases alone: what bounds the overlapped run
        d = torch.empty(shape, dtype=dtype, device="cuda")
        bound = _copy_bounds(hA, d)
        bound["sweeps_ms"] = secs / args.steps * 1e3
        bound["limit"] = max(("h2d_ms", "d2h_ms", "sweeps_ms"), key=lambda k: bound[k])
        del d
        line["e2e"] = {"value": world * upd * e2e_steps / e_secs / 1e9, "unit": "GStencil/s",
                       "h2d_bytes_per_step": nbytes, "d2h_bytes_per_step": nbytes, "steps": e2e_steps,
                       "ms_per_step": e_secs / e2e_steps * 1e3,
                       "api": "drs_run_host (C ABI): %s host grid -> H2D, schedule, D2H of the result; the three phases "
                              "overlapped by time-skewed blocks along the slow axis (bit-identical to the plain sequence)"
                              % ("pinned" if pinned else "pageable"),
                       "plain_sequence_ms_per_step": plain_ms, "bound": bound}
        del hA
    return line, plan


def _copy_bounds(h, d):
    """Host link alone: H2D and D2H of the step's bytes, ms (all ranks at once when run under torchrun)."""
    import torch
    out = {}
    for key, fn in (("h2d_ms", lambda: d.copy_(h, non_blocking=True)), ("d2h_ms", lambda: h.copy_(d, non_blocking=True))):
        torch.cuda.synchronize()
        if torch.distributed.is_available() and torch.distributed.is_initialized():
            torch.distributed.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if torch.distributed.is_available() and torch.distributed.is_initialized():
            t = torch.tensor([ms], device="cuda", dtype=torch.float64)
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
            ms = float(t)
        out[key] = ms
    return out


def run_slab(args, rank, world):
    """N > 1: c5 (3d7pt_star fp64 1536^3) over `world` GPUs, strong scaling."""
    import torch
    import torch.distributed as dist
    import drstencil_b200 as drs
    from drstencil_b200.presets import PRESETS
    from drstencil_b200.slab import GpuSlab, halo_exchange
    preset, timesteps, desc = WORKLOADS["c5"]
    path, kn = PRESETS[preset]
    if args.depth > 1:
        kn = drs.Knobs(step=args.depth)
        desc += " [temporal depth %d]" % args.depth
    parity = parity_slab(rank, world, args.halo) if not args.no_parity else None
    slab = GpuSlab(path, kn, rank, world, halo=args.halo)
    L, M, N = slab.global_shape
    g = torch.Generator(device="cuda")
    dtype = slab.dtype

    warm = max(3, args.warmup)
    total_decades = decades_per_step("c5", timesteps) * (args.steps + warm)
    if total_decades > 580:
        sys.exit("bench.py: %d steps of %d timesteps overflow fp64 (growth 10^%.0f): use fewer --steps"
                 % (args.steps + warm, timesteps, total_decades))
    start = 10.0 ** (-min(290.0, total_decades / 2 + 5))

    def plane(zg):
        g.manual_seed(1234 + zg)
        return torch.rand((M, N), dtype=dtype, device="cuda", generator=g) * start

    slab.fill(plane)
    info = slab.plan.info
    for _ in range(warm):
        slab.run(timesteps)
    slab.plan.sync_check()
    sampler = ClockSampler(torch.cuda.current_device())
    dist.barrier()
    torch.cuda.synchronize()
    l0 = slab.plan.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.start()
    e0.record()
    for _ in range(args.steps):
        slab.run(timesteps)
    e1.record()
    slab.plan.sync_check()
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"A_rank%d" % rank: slab.owned(0), "B_rank%d" % rank: slab.owned(1)},
                     DUMP_POINTS // world)
    secs = e0.elapsed_time(e1) * 1e-3
    t = torch.tensor([secs], device="cuda", dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    secs = float(t)
    data_finite = bool(torch.isfinite(slab.owned(0)).all()) and float(slab.owned(0).abs().max()) > 0
    launches = slab.plan.launch_count - l0
    H = info.halo
    sweeps = drs.sweep_count(timesteps, kn.step)
    upd = (L - 2 * H) * (M - 2 * H) * (N - 2 * H) * sweeps * kn.step
    value = upd * args.steps / secs / 1e9
    peak, peak_src = measured_peak()
    esize = 8 if slab.dtype == torch.float64 else 4
    geom = slab.geom
    local_bytes = (geom.hi - geom.lo) * M * N * 2 * esize        # algorithmic bytes of this rank's launch
    sweep_launches = sweeps * args.steps
    ach = local_bytes / (secs / sweep_launches) / 1e9
    halo_bytes = 2 * geom.ghost * M * N * esize                  # pushed per sweep by an interior rank
    exchange = {"p2p": "fused into the sweep kernel (drs_run_slab): NVLink peer stores of the boundary planes + in-kernel "
                       "acquire/release step flags, boundary tiles first; one launch per sweep, CUDA-graph replay",
                "p2p-flags": "NVLink peer stores from the sweep kernel + separate one-thread flag kernels (3 launches per sweep)",
                "nccl": "NCCL isend/irecv after each sweep"}[args.halo]
    line = {
        "metric": "GStencil/s", "value": value, "unit": "GStencil/s", "n_gpus": world, "steps": args.steps,
        "warmup": warm, "ms_per_step": secs / args.steps * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64" if esize == 8 else "f32", "data": "synthetic",
        "config": {"workload": "%s: %s" % (preset, desc), "grid": [L, M, N], "timesteps_per_step": timesteps,
                   "decomposition": "k-slabs, %d planes per GPU + %d ghost planes per side" % (geom.hi - geom.lo, geom.ghost),
                   "halo_exchange": exchange, "knobs": repr(kn),
                   "halo_bytes_per_sweep_per_gpu": halo_bytes, "kernel": info.kernel_name,
                   "l2": "inputs larger than L2 (%.1f GiB per rank per sweep)" % (local_bytes / 2 ** 30)},
        "gpu_launches": launches,
        "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": None,
                     "peak_source": peak_src, "kernel": info.kernel_name, "per": "GPU (rank 0's slab)",
                     "algorithmic_bytes_per_launch": local_bytes, "launch_ms": secs / sweep_launches * 1e3},
        "clocks": clocks,
        "data_finite": data_finite,
        "parity": parity,
    }
    # ---- e2e: pinned host slab -> device, the schedule, result back (every step) ----
    own = slab.owned(0)
    h = torch.empty(own.shape, dtype=own.dtype, pin_memory=True)
    h.fill_(0.5e-100)
    streamed = args.halo == "p2p" and parity is not None and parity.get("host_path_ok", False) and not args.e2e_plain

    def e2e_step():
        if streamed:
            slab.run_host(h, timesteps)
            return
        own.copy_(h, non_blocking=True)
        halo_exchange(slab.bufs[0], geom, None)
        slab.run(timesteps)
        h.copy_(own, non_blocking=True)

    e2e_steps = 2
    slab.bufs[1].zero_()        # the streamed path relies on B's frozen ring holding the reference's zeros
    e2e_step()                  # untimed warm-up
    h.fill_(0.5e-100)
    slab.plan.sync_check()
    dist.barrier()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(e2e_steps):
        e2e_step()
    e1.record()
    slab.plan.sync_check()
    es = e0.elapsed_time(e1) * 1e-3
    t = torch.tensor([es], device="cuda", dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    es = float(t)
    bound = _copy_bounds(h, own)
    bound["sweeps_ms"] = secs / args.steps * 1e3
    bound["limit"] = max(("h2d_ms", "d2h_ms", "sweeps_ms"), key=lambda k: bound[k])
    bound["note"] = "each phase alone, all ranks at once, max over ranks: the overlapped run cannot beat the largest"
    line["e2e"] = {"value": upd * e2e_steps / es / 1e9, "unit": "GStencil/s", "h2d_bytes_per_step": own.numel() * esize * world,
                   "d2h_bytes_per_step": own.numel() * esize * world, "steps": e2e_steps, "ms_per_step": es / e2e_steps * 1e3,
                   "api": ("drs_run_host_slab (C ABI; one process per GPU): pinned host slab -> H2D, schedule, D2H, the "
                           "three phases overlapped by time-skewed blocks, faces in lockstep with the neighbours"
                           if streamed else "copy, GpuSlab.run, copy in sequence on pinned host slabs (one process per GPU)"),
                   "bound": bound}
    slab.close()
    del slab, own
    torch.cuda.empty_cache()
    # extra evidence in the same run: the same grid with in-kernel temporal depth 2 (fused halo push of
    # two ghost planes per side); the contract value above stays the bit-exact depth-1 sweep
    if args.depth == 1 and not args.no_extras:
        try:
            kn2 = drs.Knobs(step=2)
            s2 = GpuSlab(path, kn2, rank, world, halo=args.halo)
            s2.fill(plane)
            s2.run(timesteps)
            s2.plan.sync_check()
            dist.barrier()
            torch.cuda.synchronize()
            e0.record()
            for _ in range(3):
                s2.run(timesteps)
            e1.record()
            s2.plan.sync_check()
            t = torch.tensor([e0.elapsed_time(e1) * 1e-3], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            H2 = s2.plan.info.halo
            upd2 = (L - 2 * H2) * (M - 2 * H2) * (N - 2 * H2) * drs.sweep_count(timesteps, 2) * 2
            line["temporal_fused"] = {"depth": 2, "value": upd2 * 3 / float(t) / 1e9, "unit": "GStencil/s",
                                      "ms_per_step": float(t) / 3 * 1e3, "kernel": s2.plan.info.kernel_name,
                                      "parity": "see parity.cases (depth 2)"}
            s2.close()
        except Exception as e:   # extra only
            line["temporal_fused"] = {"error": str(e)[:200]}
    return line


def per_config(args):
    """The other single-GPU BASELINE configs, device-resident: each timed for >= 1 s after warm-up, with its own
    clock samples and (BASELINE configs) its own CPU baseline."""
    import torch
    import drstencil_b200 as drs
    from drstencil_b200.presets import PRESETS
    peak, _ = measured_peak()
    out = []
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    traffic = json.load(open(tp)) if os.path.exists(tp) else {}
    for wl in ("c1", "c2", "c3", "c4", "c1t2", "c3t2", "c4t2", "c5t2"):
        preset, timesteps, desc = WORKLOADS[wl]
        path, kn = PRESETS[preset]
        st = drs.Stencil.from_file(path)
        shape = st.shape
        esize = 4 if kn.dtype == drs.F32 else 8
        if 2 * all_points(shape) * esize > 0.8 * torch.cuda.get_device_properties(0).total_memory:
            continue
        try:
            plan = drs.Plan(st, kn)
            dtype = torch.float32 if kn.dtype == drs.F32 else torch.float64
            A = torch.rand(shape, dtype=dtype, device="cuda")
            B = torch.zeros_like(A)
            # values grow like (sum of coefficients)^timesteps: the >= 1 s of sweeps run in segments, the field is
            # renormalised between segments (outside the event-timed regions; NaN / Inf fields would run faster)
            low = 1e-30 if dtype == torch.float32 else 1e-200
            A.mul_(low)
            probe_s, _ = time_steps(plan, A, B, timesteps, 1, 1)
            k = max(2, int(1.05 / max(probe_s, 1e-6)) + 1)
            seg = max(1, int((50.0 if dtype == torch.float32 else 400.0) / decades_per_step(wl, timesteps)))
            sampler = ClockSampler(torch.cuda.current_device())
            renormalise(A, low)
            for _ in range(min(3, seg)):
                plan.run(A, B, timesteps)
            plan.sync_check()
            renormalise(A, low)
            l0 = plan.launch_count
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            sampler.start()
            secs = 0.0
            done = 0
            while done < k:
                m = min(seg, k - done)
                e0.record()
                for _ in range(m):
                    plan.run(A, B, timesteps)
                e1.record()
                plan.sync_check()
                secs += e0.elapsed_time(e1) * 1e-3
                done += m
                if done < k:
                    renormalise(A, low)
            clocks = sampler.stop()
            launches = plan.launch_count - l0
            finite = bool(torch.isfinite(A).all())
            info = plan.info
            upd = interior_points(shape, info.halo) * drs.sweep_count(timesteps, kn.step) * kn.step * k
            ach = all_points(shape) * 2 * esize / (secs / launches) / 1e9
            # what a plain device copy of the same array reaches (small grids cannot reach the big-copy peak)
            for _ in range(3):
                B.copy_(A)
            e0.record()
            for _ in range(10):
                B.copy_(A)
            e1.record()
            torch.cuda.synchronize()
            copy_gbs = all_points(shape) * 2 * esize / (e0.elapsed_time(e1) * 1e-4) / 1e9
            entry = {"workload": "%s: %s" % (wl, desc), "value": upd / secs / 1e9, "unit": "GStencil/s",
                     "temporal_depth": kn.step, "kernel": info.kernel_name, "knobs": repr(kn), "launch_ms": secs / launches * 1e3,
                     "gpu_launches": launches, "n_gpus": 1, "steps": k, "timesteps_per_step": timesteps,
                     "timed_seconds": secs, "segments_of_steps": seg, "data_finite": finite, "clocks": clocks,
                     "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                                  "gstencil_roofline": peak / (2 * esize) * kn.step,
                                  "frac_of_single_step_gstencil_roofline": (upd / secs / 1e9) / (peak / (2 * esize)),
                                  "torch_copy_same_array_gbs": copy_gbs, "traffic": traffic.get(wl)}}
            del A, B, plan
            torch.cuda.empty_cache()
            if wl in ("c1", "c2", "c3", "c4"):
                entry["cpu_baseline"] = cpu_baseline(wl, budget_s=4.0)
                ref = reference_gpu_kernel(wl)
                if ref:
                    entry["reference_gpu_kernel"] = ref
            out.append(entry)
        except Exception as e:
            out.append({"workload": wl, "error": str(e)[:200]})
    return out


def main():
    sys.dont_write_bytecode = True       # the tree may be read-only; nothing is cached in it
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS))
    ap.add_argument("--no-extras", action="store_true", help="skip per_config / cpu_baseline (profiling runs)")
    ap.add_argument("--no-parity", action="store_true", help="skip the in-run parity check (profiling runs)")
    ap.add_argument("--e2e-plain", action="store_true", help="N > 1: copy-sweep-copy e2e instead of drs_run_host_slab")
    ap.add_argument("--halo", default="p2p", choices=["p2p", "p2p-flags", "nccl"], help="N > 1: halo exchange path")
    ap.add_argument("--depth", type=int, default=1, help="c5 only: in-kernel temporal depth (extra evidence; "
                    "the contract line is depth 1, bit-exact)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the buffers of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm sweeps for a fixed time, so its outputs differ from run to run")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly ONE line (the JSON): libraries that write to fd 1 from C (NCCL prints its
    # version there) are sent to stderr instead
    sys.stdout.flush()
    json_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)

    if args.impl == "reference":
        line = run_reference(args, rank)
        if line is not None:
            print(json.dumps(line), file=json_out, flush=True)
        return

    import torch
    if not torch.cuda.is_available():
        sys.exit("bench.py: no CUDA device -- the engine has no CPU path (use --impl reference for the CPU oracle)")
    torch.cuda.set_device(local)
    import atexit
    import shutil
    atexit.register(shutil.rmtree, private_jit_cache(), True)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if world > 1 and (args.workload in (None, "c5")):   # world == 1 sweeps the whole grid on one GPU
        line = run_slab(args, rank, world)
    else:
        line, plan = run_single(args, rank, world)
        del plan                     # frees the device pair drs_run_host allocated
        torch.cuda.empty_cache()
    if rank == 0 and not args.no_extras:
        # the CPU baseline beside every GPU number (the other ranks wait at the barrier below)
        line["cpu_baseline"] = cpu_baseline(args.workload or "c5")
        if world == 1:
            line["per_config"] = per_config(args)
            refs = {w: reference_gpu_kernel(w) for w in ("c1", "c2", "c4")}
            line["reference_gpu_kernels"] = {w: r for w, r in refs.items() if r}
    if rank == 0:
        print(json.dumps(line), file=json_out, flush=True)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
