"""Slab decomposition of a grid along its slowest axis (planes, k, of a 3D grid; rows, j, of a 2D one) over the GPUs
of one box, one process per GPU (torchrun), with nearest-neighbour halo exchange after every sweep.

The reference is single-GPU (SURVEY.md F5); this is the engine's extension for BASELINE.json
config c5 and the 2D configs.  Semantics are those of ONE global grid swept by the reference's schedule: the global
Halo-wide ring stays frozen, every rank owns planes (rows) [lo, hi) and keeps `ghost` = Halo copies of
its neighbours' boundary planes (rows) on each side.  Below, "plane" stands for a row of a 2D grid.

Exchange paths (`halo=`):
  "p2p"        drs_run_slab: ONE launch per sweep.  The sweep kernel stores its boundary planes a second
               time, straight into the neighbour's ghost planes over NVLink (buffers mapped with CUDA IPC),
               and handles the step flags itself: tiles next to a neighbour wait (ld.acquire.sys) for that
               neighbour's previous sweep, the last boundary tile of a face releases the next flag value;
               boundary tiles run first.  No collective, no extra kernel, the whole schedule is one CUDA graph.
  "p2p-flags"  the same push, but the flags as separate one-thread kernels around every sweep (three launches
               per sweep, driven from Python) -- round 1's protocol, kept for A/B measurements.
  "nccl"       plain torch.distributed isend/irecv of the boundary planes after each sweep (NCCL on GPUs,
               gloo on CPU -- the path the CPU tests drive with a stand-in sweep).

Pair slabs (`GpuSlab(..., pairs=True)`, 3D step-1 plans, "p2p" only): the ghost regions are 2 * Halo planes deep and
drs_run_slab runs the sweeps as exact pair launches (two sweeps per launch, one double-depth halo exchange) plus two or
four single sweeps (drs_plan_set_slab_pairs).
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass
from typing import Callable, List, Optional


def split(n: int, parts: int):
    """[(lo, hi)] -- contiguous, as even as possible."""
    return [(r * n // parts, (r + 1) * n // parts) for r in range(parts)]


@dataclass
class SlabGeometry:
    """Where one rank's slab sits in the global grid (all plane indices)."""
    g_slow: int      # global planes
    world: int
    rank: int
    ghost: int       # Halo = step * order: ghost planes per side (2 * Halo on pair slabs)
    ring: Optional[int] = None   # width of the global frozen ring (default: ghost)

    def __post_init__(self):
        if self.ring is None:
            self.ring = self.ghost
        b = split(self.g_slow, self.world)
        self.bounds = b
        self.lo, self.hi = b[self.rank]
        if min(h - l for l, h in b) < self.ghost:
            raise ValueError("slab thinner than the halo: %d planes over %d ranks with Halo %d"
                             % (self.g_slow, self.world, self.ghost))
        self.origin = self.lo - self.ghost                 # global index of local plane 0
        self.local_planes = self.hi - self.lo + 2 * self.ghost
        self.lower = self.rank - 1 if self.rank > 0 else None
        self.upper = self.rank + 1 if self.rank + 1 < self.world else None
        # output range in local indices (the global ring stays frozen)
        self.out_lo = max(self.lo, self.ring) - self.origin
        self.out_hi = min(self.hi, self.g_slow - self.ring) - self.origin

    def local(self, g: int) -> int:
        return g - self.origin

    # planes (local indices) this rank sends to / receives from each neighbour after a sweep
    def send_lower(self):
        return (self.local(self.lo), self.local(self.lo + self.ghost))

    def send_upper(self):
        return (self.local(self.hi - self.ghost), self.local(self.hi))

    def recv_lower(self):
        return (self.local(self.lo - self.ghost), self.local(self.lo))

    def recv_upper(self):
        return (self.local(self.hi), self.local(self.hi + self.ghost))


def halo_exchange(buf, geom: SlabGeometry, group=None) -> None:
    """Refreshes the ghost planes of `buf` (a [local_planes, M, N] or [local_planes, N] tensor) from the
    neighbours' boundary planes with point-to-point sends/receives."""
    import torch.distributed as dist
    ops = []
    if geom.lower is not None:
        a, b = geom.send_lower()
        ops.append(dist.P2POp(dist.isend, buf[a:b], geom.lower, group))
        a, b = geom.recv_lower()
        ops.append(dist.P2POp(dist.irecv, buf[a:b], geom.lower, group))
    if geom.upper is not None:
        a, b = geom.send_upper()
        ops.append(dist.P2POp(dist.isend, buf[a:b], geom.upper, group))
        a, b = geom.recv_upper()
        ops.append(dist.P2POp(dist.irecv, buf[a:b], geom.upper, group))
    if ops:
        for r in dist.batch_isend_irecv(ops):
            r.wait()


class SlabRunner:
    """The reference's ping-pong schedule over a slab.  `sweep(src, dst)` advances the local
    output range of `dst` from `src`; `after(dst, s)` makes the neighbours' ghosts current."""

    def __init__(self, geom: SlabGeometry, bufs, sweep: Callable, after: Callable, before: Optional[Callable] = None):
        self.geom, self.bufs, self.sweep, self.after, self.before = geom, bufs, sweep, after, before
        self.sweeps_done = 0

    def run(self, timesteps: int, step: int) -> int:
        n = 0
        t = 0
        while t < timesteps:
            for _ in range(2):
                s = self.sweeps_done
                src, dst = self.bufs[s & 1], self.bufs[(s & 1) ^ 1]
                if self.before:
                    self.before(s)
                self.sweep(src, dst)
                self.after(dst, s)
                self.sweeps_done += 1
                n += 1
            t += 2 * step
        return n


# ---------------------------------------------------------------------------------------------
# GPU wiring
# ---------------------------------------------------------------------------------------------

class _DevArray:
    """A cudaMalloc allocation (whole allocation, so it can be exported with CUDA IPC) viewed as a
    torch tensor through __cuda_array_interface__."""

    def __init__(self, shape, np_typestr: str, itemsize: int):
        from . import lib, _check
        n = 1
        for d in shape:
            n *= d
        p = ctypes.c_void_p()
        _check(lib().drs_device_malloc(n * itemsize, ctypes.byref(p)))
        self.ptr = p.value
        self.nbytes = n * itemsize
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": np_typestr, "data": (self.ptr, False),
                                         "version": 2, "strides": None}

    def tensor(self):
        import torch
        return torch.as_tensor(self, device="cuda")

    def free(self):
        from . import lib
        if self.ptr:
            lib().drs_device_free(self.ptr)
            self.ptr = 0


def _ipc_export(ptr: int) -> bytes:
    from . import lib, _check
    h = ctypes.create_string_buffer(64)
    _check(lib().drs_ipc_export(ptr, h))
    return h.raw


def _ipc_import(handle: bytes) -> int:
    from . import lib, _check
    p = ctypes.c_void_p()
    _check(lib().drs_ipc_import(handle, ctypes.byref(p)))
    return p.value


class GpuSlab:
    """One rank's share of a slab-decomposed run on its GPU."""

    def __init__(self, stc_path: str, knobs, rank: int, world: int, halo: str = "p2p", group=None,
                 global_shape=None, pairs: bool = False):
        import torch
        import torch.distributed as dist
        from . import Plan, Stencil, F32
        if pairs and halo != "p2p":
            raise ValueError("pair slabs need the p2p halo mode (drs_run_slab), not %r" % halo)
        self.rank, self.world, self.mode, self.group, self.pairs = rank, world, halo, group, pairs
        st = Stencil.from_file(stc_path)
        if global_shape is not None:
            st.set_size(global_shape)
        self.global_shape = tuple(st.shape)
        slow, rest = self.global_shape[0], self.global_shape[1:]     # (L, (M, N)) or (M, (N,))
        probe = Plan(st, knobs)                      # halo of the (possibly multi-step) sweep
        ghost = probe.halo
        self.step = knobs.step
        self.geom = SlabGeometry(slow, world, rank, 2 * ghost if pairs else ghost, ring=ghost)
        shape = (self.geom.local_planes,) + rest
        st.set_size(shape)
        self.plan = Plan(st, knobs)
        if pairs:
            self.plan.set_slab_pairs(slow, self.geom.lo, self.geom.hi)
        else:
            self.plan.set_slab(slow, self.geom.lo, self.geom.hi)
        self.dtype = torch.float32 if knobs.dtype == F32 else torch.float64
        typestr, isz = ("<f4", 4) if knobs.dtype == F32 else ("<f8", 8)
        self._raw = [_DevArray(shape, typestr, isz), _DevArray(shape, typestr, isz)]
        self.bufs = [r.tensor() for r in self._raw]
        for b in self.bufs:
            b.zero_()
        self._peer_ptrs: List[int] = []
        self._flags = None
        if halo in ("p2p", "p2p-flags") and world > 1:
            self._flags = _DevArray((2,), "<i8", 8)
            self._flags.tensor().zero_()
            mine = [_ipc_export(r.ptr) for r in self._raw] + [_ipc_export(self._flags.ptr)]
            everyone = [None] * world
            dist.all_gather_object(everyone, mine, group=group)
            lower = upper = None
            g = self.geom
            if g.lower is not None:
                lower = [_ipc_import(h) for h in everyone[g.lower]]
                self._peer_ptrs += lower
            if g.upper is not None:
                upper = [_ipc_import(h) for h in everyone[g.upper]]
                self._peer_ptrs += upper
            self.plan.set_peers([r.ptr for r in self._raw], lower[:2] if lower else [0, 0],
                                upper[:2] if upper else [0, 0],
                                g.bounds[g.lower][0] if lower else 0, g.bounds[g.upper][0] if upper else 0)
            # a rank writes slot 1 of its lower neighbour's flags and slot 0 of its upper neighbour's
            self._lower_flag = lower[2] + 8 if lower else 0
            self._upper_flag = upper[2] if upper else 0
            self.plan.set_flags(self._flags.ptr, self._lower_flag, self._upper_flag)
            torch.cuda.synchronize()
            dist.barrier(group=group)
        elif halo == "p2p":
            self.plan.set_peers([r.ptr for r in self._raw], [0, 0], [0, 0], 0, 0)
        # flag values are monotone over the life of the object (sweeps run so far): never reset
        self._seq = 0
        self.runner = SlabRunner(self.geom, self.bufs, self._sweep, self._after, self._before)

    # -- schedule hooks --
    def _before(self, s: int) -> None:
        if self.mode == "p2p-flags" and self.world > 1:
            g = self.geom
            self.plan.wait_flags(self._flags.ptr, g.lower is not None, g.upper is not None, self._seq)

    def _sweep(self, src, dst) -> None:
        self.plan.sweep(src, dst)

    def _after(self, dst, s: int) -> None:
        if self.world == 1:
            return
        if self.mode == "p2p-flags":
            self._seq += 1
            self.plan.signal_peers(self._lower_flag, self._upper_flag, self._seq)
        else:
            halo_exchange(dst, self.geom, self.group)

    # -- data --
    def fill(self, plane_fn: Callable) -> None:
        """A[local plane] = plane_fn(global plane index) for every in-grid plane (row of a 2D grid) this rank
        holds (owned and ghost); B = 0.  Restarts the schedule at sweep(A, B).  Collective: every rank calls it."""
        import torch
        import torch.distributed as dist
        g = self.geom
        if self.world > 1:
            # nobody may still be pushing into these arrays: all ranks drain their streams first
            self.plan.sync_check()
            torch.cuda.synchronize()
            dist.barrier(group=self.group)
        self.bufs[0].zero_()
        self.bufs[1].zero_()
        for zl in range(g.local_planes):
            zg = g.origin + zl
            if 0 <= zg < g.g_slow:
                self.bufs[0][zl].copy_(plane_fn(zg))
        if self.world > 1:
            torch.cuda.synchronize()
            dist.barrier(group=self.group)
        self.runner.sweeps_done = 0

    def run(self, timesteps: int) -> int:
        if self.mode == "p2p":
            return self.plan.run_slab(timesteps)
        return self.runner.run(timesteps, self.step)

    def run_host(self, h_own, timesteps: int) -> float:
        """The reference schedule on this rank's HOST slab `h_own` (own planes only, pinned), uploads / sweeps /
        downloads overlapped by time-skewed blocks, faces in lockstep with the neighbours (drs_run_host_slab).
        Needs the "p2p" halo mode.  Collective (contains the barrier that separates calls).  Returns device ms.
        The device copy of B must hold zeros in its frozen ring (true after construction or fill())."""
        import torch
        import torch.distributed as dist
        if self.mode != "p2p" or self.world < 2:
            raise ValueError("run_host needs the p2p halo mode and at least two ranks (one GPU: Plan.run_host)")
        if self.pairs:
            raise ValueError("run_host has no pair schedule: use a GpuSlab with pairs=False")
        self.plan.sync_check()
        torch.cuda.synchronize()
        dist.barrier(group=self.group)               # nobody still reads ghosts of the previous call
        return self.plan.run_host_slab(h_own, timesteps, self.rank % 2 == 1)

    def owned(self, which: int = 0):
        """The rank's owned planes of buffer `which` (0 = A, where the result lands)."""
        g = self.geom
        return self.bufs[which][g.ghost:g.ghost + (g.hi - g.lo)]

    def close(self) -> None:
        """Collective: unmaps the neighbours' arrays and frees this rank's."""
        from . import lib
        import torch
        torch.cuda.synchronize()
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier(group=self.group)           # no neighbour still pushes into / reads from these arrays
        for p in self._peer_ptrs:
            lib().drs_ipc_close(p)
        self._peer_ptrs = []
        self.bufs = []
        self.runner = None
        self.plan = None
        for r in self._raw:
            r.free()
        self._raw = []
        if self._flags is not None:
            self._flags.free()
            self._flags = None
