"""drstencil_b200 -- host-side mirror of the DRStencil generator flow over the C ABI in
include/drstencil.h (libdrstencil.so).

The reference's "API" is `drstencil [options] x.stc` (/root/reference/main.cpp:10-280) followed by
nvcc and the emitted program.  The same steps here:

    st   = Stencil.from_file("2d9pt_box.stc")            # DRStencil_2d::get_stencil
    plan = Plan(st, Knobs(step=4))                       # fusing + codeGen_2d::output + nvcc
    plan.run(a, b, iterations=st.iterations)             # the emitted main()'s ping-pong loop

Device memory comes from the caller (torch tensors or raw pointers); torch is only plumbing.
There is no CPU fallback: every compute call needs a B200 and raises DrsError otherwise.
"""
from __future__ import annotations

import ctypes
import os
from dataclasses import dataclass, field, fields
from typing import Optional, Sequence

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIBPATH = os.path.join(_HERE, "libdrstencil.so")

F64, F32 = 0, 1
FUSE_TEMPORAL, FUSE_ALGEBRAIC, FUSE_REUSE = 0, 1, 2
E_ARG, E_IO, E_NOREUSE, E_CONFIG, E_COMPILE, E_CUDA, E_NOGPU, E_KERNEL = -1, -2, -3, -4, -5, -6, -7, -8
HOST_UPLOAD, HOST_SWEEP, HOST_DOWNLOAD, HOST_PAIR = 0, 1, 2, 3     # record kinds of Plan.host_schedule


class DrsError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("drstencil error %d: %s" % (code, msg))
        self.code = code


class _CKnobs(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int) for n in (
        "step", "dist", "streaming", "bx", "by", "sn", "stream_unroll", "block_merge_x", "block_merge_y",
        "cyclic_merge_x", "cyclic_merge_y", "prefetch", "merge_forward", "check", "dtype", "fuse",
        "explicit_mask")] + [("reserved", ctypes.c_int * 7)]


class _CInfo(ctypes.Structure):
    _fields_ = [("dim", ctypes.c_int), ("dtype", ctypes.c_int), ("step", ctypes.c_int), ("fuse", ctypes.c_int),
                ("L", ctypes.c_longlong), ("M", ctypes.c_longlong), ("N", ctypes.c_longlong),
                ("halo", ctypes.c_int), ("npoints", ctypes.c_int), ("timesteps_per_sweep", ctypes.c_int),
                ("warps_per_cta", ctypes.c_int), ("tile_x", ctypes.c_int), ("tile_y", ctypes.c_int),
                ("chunk", ctypes.c_int), ("stages", ctypes.c_int), ("rows_per_stage", ctypes.c_int),
                ("grid_x", ctypes.c_int), ("grid_y", ctypes.c_int), ("grid_z", ctypes.c_int), ("block", ctypes.c_int),
                ("smem_bytes", ctypes.c_int), ("regs_per_thread", ctypes.c_int), ("spill_bytes", ctypes.c_int),
                ("redundancy", ctypes.c_double), ("kernel_name", ctypes.c_char * 96)]


_lib = None


def build(verbose: bool = False) -> str:
    from . import _build as _b
    return _b.build(verbose=verbose)


def lib():
    """The loaded C ABI.  Fails loudly when the native library is missing (no Python fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIBPATH):
        raise ImportError("%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(or drstencil_b200.build())" % _LIBPATH)
    # The library dlopen()s ONE pinned NVRTC by absolute path (csrc/capi/capi.cpp, _build.pinned_nvrtc), so the
    # cubins no longer depend on whether torch was imported first (round 1: two compilers, two sets of cubins).
    L = ctypes.CDLL(_LIBPATH)
    vp, i32, ll = ctypes.c_void_p, ctypes.c_int, ctypes.c_longlong
    P = ctypes.POINTER
    sig = {
        "drs_knobs_default": (None, [P(_CKnobs)]),
        "drs_stencil_from_file": (i32, [ctypes.c_char_p, i32, P(vp)]),
        "drs_stencil_from_points": (i32, [i32, P(i32), P(ctypes.c_double), i32, ll, ll, ll, i32, P(vp)]),
        "drs_stencil_destroy": (None, [vp]),
        "drs_stencil_set_name": (i32, [vp, ctypes.c_char_p]),
        "drs_stencil_set_size": (i32, [vp, ll, ll, ll, i32]),
        "drs_stencil_compose": (i32, [vp, i32]),
        "drs_stencil_size": (i32, [vp, P(ll), P(i32)]),
        "drs_stencil_terms": (i32, [vp, P(i32), P(ctypes.c_double), i32]),
        "drs_stencil_term_text": (i32, [vp, i32, ctypes.c_char_p, ctypes.c_size_t]),
        "drs_stencil_analyze": (i32, [vp, i32, i32, P(i32), P(i32), P(i32), P(i32)]),
        "drs_plan_create": (i32, [vp, P(_CKnobs), P(vp)]),
        "drs_plan_warm_cache": (i32, [vp, P(_CKnobs)]),
        "drs_plan_destroy": (None, [vp]),
        "drs_plan_get_info": (i32, [vp, P(_CInfo)]),
        "drs_plan_source": (ctypes.c_char_p, [vp]),
        "drs_plan_note": (ctypes.c_char_p, [vp]),
        "drs_plan_cache_key": (ctypes.c_char_p, [vp]),
        "drs_plan_pair_source": (ctypes.c_char_p, [vp]),
        "drs_plan_pair_cache_key": (ctypes.c_char_p, [vp]),
        "drs_plan_slab_source": (ctypes.c_char_p, [vp]),
        "drs_plan_slab_cache_key": (ctypes.c_char_p, [vp]),
        "drs_plan_slab_pair_source": (ctypes.c_char_p, [vp]),
        "drs_plan_slab_pair_cache_key": (ctypes.c_char_p, [vp]),
        "drs_plan_slab_split": (i32, [vp, i32, P(i32), P(i32)]),
        "drs_sweep_pair": (i32, [vp, vp, vp, vp]),
        "drs_plan_set_slab_pairs": (i32, [vp, ll, ll, ll]),
        "drs_plan_pair_split": (i32, [vp, i32, P(i32), P(i32)]),
        "drs_plan_set_pairs": (i32, [vp, i32]),
        "drs_sweep": (i32, [vp, vp, vp, vp]),
        "drs_gold_sweep": (i32, [vp, vp, vp, vp]),
        "drs_run": (i32, [vp, vp, vp, i32, vp, P(i32)]),
        "drs_gold_run": (i32, [vp, vp, vp, i32, vp, P(i32)]),
        "drs_run_host": (i32, [vp, vp, vp, i32, P(ctypes.c_float)]),
        "drs_plan_set_host_block": (i32, [vp, ll]),
        "drs_plan_set_graph": (i32, [vp, i32]),
        "drs_plan_host_schedule": (i32, [vp, i32, P(ll), i32]),
        "drs_plan_slab_schedule": (i32, [vp, i32, i32, P(ll), i32]),
        "drs_run_host_slab": (i32, [vp, vp, i32, i32, P(ctypes.c_float)]),
        "drs_plan_set_flags": (i32, [vp, vp, vp, vp]),
        "drs_run_slab": (i32, [vp, i32, vp, P(i32)]),
        "drs_check_error": (i32, [vp, vp, vp, P(ctypes.c_double)]),
        "drs_plan_sync_check": (i32, [vp, vp]),
        "drs_plan_launch_count": (ll, [vp]),
        "drs_plan_set_slab": (i32, [vp, ll, ll, ll]),
        "drs_plan_set_peers": (i32, [vp, P(vp), P(vp), P(vp), ll, ll]),
        "drs_signal_peers": (i32, [vp, vp, vp, ll, vp]),
        "drs_wait_flags": (i32, [vp, vp, i32, i32, ll, vp]),
        "drs_device_malloc": (i32, [ctypes.c_size_t, P(vp)]),
        "drs_device_free": (i32, [vp]),
        "drs_device_upload": (i32, [vp, vp, ctypes.c_size_t]),
        "drs_device_download": (i32, [vp, vp, ctypes.c_size_t]),
        "drs_ipc_export": (i32, [vp, ctypes.c_char_p]),
        "drs_ipc_import": (i32, [ctypes.c_char_p, P(vp)]),
        "drs_ipc_close": (i32, [vp]),
        "drs_emit_program": (i32, [vp, P(_CKnobs), ctypes.c_char_p, ctypes.c_char_p]),
        "drs_last_error": (ctypes.c_char_p, []),
        "drs_version": (ctypes.c_char_p, []),
        "drs_compiler": (ctypes.c_char_p, []),
        "drs_device_count": (i32, []),
        "drs_set_device": (i32, [i32]),
        "drs_set_cache_dir": (None, [ctypes.c_char_p]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def _check(rc: int) -> int:
    if rc < 0:
        raise DrsError(rc, lib().drs_last_error().decode(errors="replace"))
    return rc


def _ptr(x) -> int:
    """Device/host address of a torch tensor, numpy array or int."""
    if x is None:
        return 0
    if isinstance(x, int):
        return x
    if hasattr(x, "data_ptr"):
        return x.data_ptr()
    if hasattr(x, "ctypes"):
        return x.ctypes.data
    raise TypeError("expected a tensor, array or address, got %r" % type(x))


def _stream(s) -> int:
    if s is None:
        try:
            import torch
            if torch.cuda.is_available():
                return torch.cuda.current_stream().cuda_stream
        except Exception:
            pass
        return 0
    return s if isinstance(s, int) else s.cuda_stream


# knob order == bit positions of drs_knobs.explicit_mask
_KNOB_ORDER = ("step", "dist", "streaming", "bx", "by", "sn", "stream_unroll", "block_merge_x", "block_merge_y",
               "cyclic_merge_x", "cyclic_merge_y", "prefetch", "merge_forward", "check", "dtype", "fuse")
_KNOB_DEFAULTS = dict(step=1, dist=0, streaming=0, bx=16, by=16, sn=16, stream_unroll=4, block_merge_x=1,
                      block_merge_y=1, cyclic_merge_x=1, cyclic_merge_y=1, prefetch=0, merge_forward=5, check=0,
                      dtype=F64, fuse=FUSE_TEMPORAL)


class Knobs:
    """The generator's options (main.cpp:12-56), same names, same defaults.  Only options passed
    explicitly constrain the engine; the rest are chosen for B200.  Engine-only tuning overrides:
    stages, min_blocks, warps, rows_3d (RY), rows_per_stage, vectors (128-bit vectors per thread, 2D),
    share_x / share_y (warps of a CTA that share one input ring in the single-step 3D sweep: the c4 / c5 presets)."""

    def __init__(self, **kw):
        self.values = dict(_KNOB_DEFAULTS)
        self.explicit = set()
        self.extra = dict(stages=0, min_blocks=0, warps=0, rows_3d=0, rows_per_stage=0, vectors=0, no_factor=0, no_fused3d=0,
                          share_x=0, share_y=0)
        for k, v in kw.items():
            self.set(k, v)

    def set(self, name: str, value) -> "Knobs":
        name = name.replace("-", "_")
        if name == "dtype" and isinstance(value, str):
            value = {"f64": F64, "fp64": F64, "double": F64, "f32": F32, "fp32": F32, "float": F32}[value]
        if name == "fuse" and isinstance(value, str):
            value = {"temporal": FUSE_TEMPORAL, "algebraic": FUSE_ALGEBRAIC, "reuse": FUSE_REUSE}[value]
        if name in self.extra:
            self.extra[name] = int(value)
        elif name in self.values:
            self.values[name] = int(value)
            self.explicit.add(name)
        else:
            raise KeyError("unknown knob %r" % name)
        return self

    def __getattr__(self, name):
        v = self.__dict__.get("values", {})
        if name in v:
            return v[name]
        raise AttributeError(name)

    def to_c(self) -> _CKnobs:
        k = _CKnobs()
        lib().drs_knobs_default(ctypes.byref(k))
        mask = 0
        for bit, name in enumerate(_KNOB_ORDER):
            setattr(k, name, self.values[name])
            if name in self.explicit:
                mask |= 1 << bit
        k.explicit_mask = mask
        k.reserved[0] = self.extra["stages"]
        k.reserved[1] = self.extra["min_blocks"]
        k.reserved[2] = self.extra["warps"]
        k.reserved[3] = self.extra["rows_3d"]
        k.reserved[4] = self.extra["rows_per_stage"]
        k.reserved[5] = self.extra["vectors"]
        k.reserved[6] = (1 if self.extra["no_factor"] else 0) | (2 if self.extra["no_fused3d"] else 0)
        if self.extra["share_x"] > 1 or self.extra["share_y"] > 1:      # CTA-shared 3D ring (drs_sweep3d_cta.cuh)
            k.reserved[6] |= ((max(1, self.extra["share_x"]) - 1) & 3) << 2 | ((max(1, self.extra["share_y"]) - 1) & 3) << 4
        return k

    def __repr__(self):
        parts = ["%s=%s" % (n, self.values[n]) for n in _KNOB_ORDER if n in self.explicit]
        parts += ["%s=%s" % (n, v) for n, v in self.extra.items() if v]
        return "Knobs(%s)" % ", ".join(parts)


class Stencil:
    """DRStencil_2d / DRStencil: a parsed stencil description (drstencil_2d.hpp:14-45)."""

    def __init__(self, handle: int, dim: int):
        self._h = ctypes.c_void_p(handle)
        self.dim = dim

    @classmethod
    def from_file(cls, path: str, is3d: Optional[bool] = None) -> "Stencil":
        if is3d is None:
            import re
            is3d = re.match(r"(c\d+_)?3d", os.path.basename(path)) is not None
        h = ctypes.c_void_p()
        _check(lib().drs_stencil_from_file(os.fsencode(path), 1 if is3d else 0, ctypes.byref(h)))
        return cls(h.value, 3 if is3d else 2)

    @classmethod
    def from_points(cls, offsets: Sequence[Sequence[int]], coefs: Sequence[float], shape: Sequence[int],
                    iterations: int = 0, name: Optional[str] = None) -> "Stencil":
        dim = len(shape)
        flat = [int(v) for p in offsets for v in p]
        assert len(flat) == dim * len(coefs)
        co = (ctypes.c_int * len(flat))(*flat)
        cc = (ctypes.c_double * len(coefs))(*[float(c) for c in coefs])
        L, M, N = (1, shape[0], shape[1]) if dim == 2 else shape
        h = ctypes.c_void_p()
        _check(lib().drs_stencil_from_points(dim, co, cc, len(coefs), L, M, N, iterations, ctypes.byref(h)))
        s = cls(h.value, dim)
        if name:
            s.set_name(name)
        return s

    def __del__(self):
        try:
            if self._h:
                lib().drs_stencil_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def set_name(self, name: str) -> "Stencil":
        _check(lib().drs_stencil_set_name(self._h, name.encode()))
        return self

    def set_size(self, shape: Sequence[int], iterations: Optional[int] = None) -> "Stencil":
        L, M, N = (1, shape[0], shape[1]) if len(shape) == 2 else shape
        it = self.iterations if iterations is None else iterations
        _check(lib().drs_stencil_set_size(self._h, L, M, N, it))
        return self

    def compose(self, step: int) -> "Stencil":
        """fusing() -- in place; only for inspection: Plan wants the un-composed stencil."""
        _check(lib().drs_stencil_compose(self._h, step))
        return self

    def _size(self):
        d = (ctypes.c_longlong * 3)()
        it = ctypes.c_int()
        _check(lib().drs_stencil_size(self._h, d, ctypes.byref(it)))
        return (d[0], d[1], d[2]), it.value

    @property
    def shape(self):
        (L, M, N), _ = self._size()
        return (M, N) if self.dim == 2 else (L, M, N)

    @property
    def iterations(self) -> int:
        return self._size()[1]

    def terms(self):
        """[(dk, dj, di, coef)] of the current operator in evaluation order; coef = literal value."""
        n = _check(lib().drs_stencil_terms(self._h, None, None, 0))
        offs = (ctypes.c_int * (3 * n))()
        co = (ctypes.c_double * n)()
        _check(lib().drs_stencil_terms(self._h, offs, co, n))
        return [(offs[3 * q], offs[3 * q + 1], offs[3 * q + 2], co[q]) for q in range(n)]

    def term_texts(self):
        n = _check(lib().drs_stencil_terms(self._h, None, None, 0))
        out = []
        buf = ctypes.create_string_buffer(64)
        for q in range(n):
            _check(lib().drs_stencil_term_text(self._h, q, buf, 64))
            out.append(buf.value.decode())
        return out

    def analyze(self, dist: int = 0, merge_forward: int = 5):
        """dict(halo, dist, range, forward_slow, forward_mid, forward_fast, backward);
        raises DrsError(E_NOREUSE) where the reference exits with "No data to reuse"."""
        halo, d, rng = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
        sizes = (ctypes.c_int * 4)()
        _check(lib().drs_stencil_analyze(self._h, dist, merge_forward, ctypes.byref(halo), ctypes.byref(d),
                                         ctypes.byref(rng), sizes))
        return dict(halo=halo.value, dist=d.value, range=rng.value, forward_slow=sizes[0], forward_mid=sizes[1],
                    forward_fast=sizes[2], backward=sizes[3])


@dataclass
class PlanInfo:
    dim: int = 0
    dtype: int = 0
    step: int = 0
    fuse: int = 0
    L: int = 0
    M: int = 0
    N: int = 0
    halo: int = 0
    npoints: int = 0
    timesteps_per_sweep: int = 0
    warps_per_cta: int = 0
    tile_x: int = 0
    tile_y: int = 0
    chunk: int = 0
    stages: int = 0
    rows_per_stage: int = 0
    grid_x: int = 0
    grid_y: int = 0
    grid_z: int = 0
    block: int = 0
    smem_bytes: int = 0
    regs_per_thread: int = 0
    spill_bytes: int = 0
    redundancy: float = 0.0
    kernel_name: str = ""


class Plan:
    """One specialised, compiled sweep: what `drstencil [options] x.stc` + nvcc produce."""

    def __init__(self, stencil: Stencil, knobs: Optional[Knobs] = None):
        self.stencil = stencil
        self.knobs = knobs or Knobs()
        h = ctypes.c_void_p()
        ck = self.knobs.to_c()
        _check(lib().drs_plan_create(stencil._h, ctypes.byref(ck), ctypes.byref(h)))
        self._h = h

    def __del__(self):
        try:
            if self._h:
                lib().drs_plan_destroy(self._h)
                self._h = None
        except Exception:
            pass

    @property
    def info(self) -> PlanInfo:
        ci = _CInfo()
        _check(lib().drs_plan_get_info(self._h, ctypes.byref(ci)))
        out = PlanInfo()
        for f in fields(PlanInfo):
            v = getattr(ci, f.name)
            setattr(out, f.name, v.decode() if isinstance(v, bytes) else v)
        return out

    @property
    def source(self) -> str:
        return lib().drs_plan_source(self._h).decode()

    @property
    def note(self) -> str:
        return lib().drs_plan_note(self._h).decode()

    @property
    def cache_key(self) -> str:
        return lib().drs_plan_cache_key(self._h).decode()

    @property
    def pair_source(self) -> str:
        """Translation unit of the exact pair kernel run() uses on this plan ("" = none: one launch per sweep)."""
        return lib().drs_plan_pair_source(self._h).decode()

    @property
    def pair_cache_key(self) -> str:
        return lib().drs_plan_pair_cache_key(self._h).decode()

    @property
    def slab_source(self) -> str:
        """Translation unit of the 2D slab entry drslab_<name>, made by set_slab ("" on 3D plans, whose main unit has
        it, and on plans without a slab kernel)."""
        return lib().drs_plan_slab_source(self._h).decode()

    @property
    def slab_cache_key(self) -> str:
        return lib().drs_plan_slab_cache_key(self._h).decode()

    @property
    def slab_pair_source(self) -> str:
        """Translation unit of the slab pair entry drslabpair_<name>, made by set_slab_pairs ("" on every other plan)."""
        return lib().drs_plan_slab_pair_source(self._h).decode()

    @property
    def slab_pair_cache_key(self) -> str:
        return lib().drs_plan_slab_pair_cache_key(self._h).decode()

    def slab_split(self, iterations: int):
        """(pairs, singles): run_slab() performs `pairs` pair launches, then `singles` single sweeps (pairs = 0
        except after set_slab_pairs)."""
        p, s = ctypes.c_int(), ctypes.c_int()
        _check(lib().drs_plan_slab_split(self._h, iterations, ctypes.byref(p), ctypes.byref(s)))
        return p.value, s.value

    def pair_split(self, iterations: int):
        """(pairs, singles): run() performs `pairs` exact pair launches, then `singles` single sweeps."""
        p, s = ctypes.c_int(), ctypes.c_int()
        _check(lib().drs_plan_pair_split(self._h, iterations, ctypes.byref(p), ctypes.byref(s)))
        return p.value, s.value

    def set_pairs(self, enable: bool) -> None:
        """Opt-in exact pair launches for run() and run_host(), streamed or plain: on 2D plans the 2D pair unit, on 3D
        plans the pair unit without its 1 GiB rule (see drs_plan_set_pairs in drstencil.h).  False restores the default rule.
        Raises DrsError (E_ARG, with the reason) for plans that have no pair kernel and for slab plans."""
        _check(lib().drs_plan_set_pairs(self._h, 1 if enable else 0))

    @property
    def halo(self) -> int:
        return self.info.halo

    def sweep(self, d_in, d_out, stream=None) -> None:
        _check(lib().drs_sweep(self._h, _ptr(d_in), _ptr(d_out), _stream(stream)))

    def sweep_pair(self, d_in, d_out, stream=None) -> None:
        """One pair launch on a pair slab with peers set (two sweeps, pushes, no flags): the counterpart of sweep()."""
        _check(lib().drs_sweep_pair(self._h, _ptr(d_in), _ptr(d_out), _stream(stream)))

    def gold_sweep(self, d_in, d_out, stream=None) -> None:
        _check(lib().drs_gold_sweep(self._h, _ptr(d_in), _ptr(d_out), _stream(stream)))

    def run(self, d_a, d_b, iterations: int, stream=None) -> int:
        n = ctypes.c_int()
        _check(lib().drs_run(self._h, _ptr(d_a), _ptr(d_b), iterations, _stream(stream), ctypes.byref(n)))
        return n.value

    def gold_run(self, d_a, d_b, iterations: int, stream=None) -> int:
        n = ctypes.c_int()
        _check(lib().drs_gold_run(self._h, _ptr(d_a), _ptr(d_b), iterations, _stream(stream), ctypes.byref(n)))
        return n.value

    def run_host(self, h_a, h_b, iterations: int) -> float:
        """The emitted main()'s data path on host arrays (H2D, schedule, D2H of A); returns device ms."""
        ms = ctypes.c_float()
        _check(lib().drs_run_host(self._h, _ptr(h_a), _ptr(h_b) or None, iterations, ctypes.byref(ms)))
        return ms.value

    def set_graph(self, enable: bool) -> None:
        """run() as one CUDA graph per (A, B, sweep count) (default) or as plain launches."""
        _check(lib().drs_plan_set_graph(self._h, int(bool(enable))))

    def host_schedule(self, iterations: int):
        """[(kind, block, launch, lo, hi)] the streamed run_host would execute ([] = plain sequence); no GPU needed.
        kind: HOST_UPLOAD, HOST_SWEEP (one single sweep), HOST_PAIR (one exact pair launch, on plans where run() pairs)
        or HOST_DOWNLOAD.  launch: 1-based index in run()'s launch sequence (odd: A -> B; the sweep number on plans
        without pair launches), 0 for copies.  [lo, hi): the slow-axis planes (rows in 2D) copied or stored."""
        n = _check(lib().drs_plan_host_schedule(self._h, iterations, None, 0))
        if n == 0:
            return []
        buf = (ctypes.c_longlong * (5 * n))()
        _check(lib().drs_plan_host_schedule(self._h, iterations, buf, n))
        return [tuple(buf[5 * i:5 * i + 5]) for i in range(n)]

    def slab_schedule(self, iterations: int, up_skew: bool):
        """[(kind, block, sweep, lo, hi, faces)] for this rank of a slab run (planner only; see drstencil.h)."""
        n = _check(lib().drs_plan_slab_schedule(self._h, iterations, int(up_skew), None, 0))
        if n == 0:
            return []
        buf = (ctypes.c_longlong * (6 * n))()
        _check(lib().drs_plan_slab_schedule(self._h, iterations, int(up_skew), buf, n))
        return [tuple(buf[6 * i:6 * i + 6]) for i in range(n)]

    def set_flags(self, my_flags: int, lower_flag: int, upper_flag: int) -> None:
        _check(lib().drs_plan_set_flags(self._h, my_flags, lower_flag or None, upper_flag or None))

    def run_slab(self, iterations: int, stream=None) -> int:
        """This rank's share of the emitted host loop on a slab-decomposed grid: one launch per sweep, the
        halo exchange and the step flags fused into the sweep kernel (drs_run_slab)."""
        n = ctypes.c_int()
        _check(lib().drs_run_slab(self._h, iterations, _stream(stream), ctypes.byref(n)))
        return n.value

    def run_host_slab(self, h_own, iterations: int, up_skew: bool) -> float:
        """This rank's share of a slab-decomposed host-buffer run (see drstencil.h); device ms."""
        ms = ctypes.c_float()
        _check(lib().drs_run_host_slab(self._h, _ptr(h_own), iterations, int(up_skew), ctypes.byref(ms)))
        return ms.value

    def set_host_block(self, units: int) -> None:
        """Block thickness (slow-axis units) of the streamed run_host: 0 = auto, < 0 = plain sequence."""
        _check(lib().drs_plan_set_host_block(self._h, units))

    def check_error(self, d_out, d_ref):
        res = (ctypes.c_double * 2)()
        _check(lib().drs_check_error(self._h, _ptr(d_out), _ptr(d_ref), res))
        return res[0], res[1]

    def sync_check(self, stream=None) -> None:
        _check(lib().drs_plan_sync_check(self._h, _stream(stream)))

    @property
    def launch_count(self) -> int:
        return lib().drs_plan_launch_count(self._h)

    def set_slab(self, global_slow: int, lo: int, hi: int) -> None:
        _check(lib().drs_plan_set_slab(self._h, global_slow, lo, hi))

    def set_slab_pairs(self, global_slow: int, lo: int, hi: int) -> None:
        """set_slab with ghost regions of 2 * Halo planes: run_slab() then runs exact pair launches (see drstencil.h)."""
        _check(lib().drs_plan_set_slab_pairs(self._h, global_slow, lo, hi))

    def set_peers(self, my_bases, lower_bases, upper_bases, lower_lo: int, upper_lo: int) -> None:
        arr = lambda xs: (ctypes.c_void_p * 2)(*[_ptr(x) or None for x in xs])
        _check(lib().drs_plan_set_peers(self._h, arr(my_bases), arr(lower_bases), arr(upper_bases), lower_lo, upper_lo))

    def signal_peers(self, lower_flag: int, upper_flag: int, value: int, stream=None) -> None:
        _check(lib().drs_signal_peers(self._h, lower_flag or None, upper_flag or None, value, _stream(stream)))

    def wait_flags(self, my_flags: int, wait_lower: bool, wait_upper: bool, value: int, stream=None) -> None:
        _check(lib().drs_wait_flags(self._h, my_flags, int(wait_lower), int(wait_upper), value, _stream(stream)))

    def emit_program(self, path: str, kernel_name: Optional[str] = None) -> None:
        ck = self.knobs.to_c()
        _check(lib().drs_emit_program(self.stencil._h, ctypes.byref(ck), (kernel_name or "").encode(), os.fsencode(path)))


def sweep_count(iterations: int, step: int) -> int:
    """Launches the emitted loop `for (t = 0; t < Iterations; t += 2*step)` performs (codegen_2d.hpp:610-613)."""
    n, t = 0, 0
    while t < iterations:
        n += 2
        t += 2 * step
    return n


def warm_cache(verbose: bool = False) -> int:
    """Pre-compiles (NVRTC, no GPU needed) the kernels of the shipped stencils and the BASELINE
    configurations into drstencil_b200/_jitcache/ so that they travel to the GPU box."""
    from .presets import PRESETS
    n = 0
    for name, (path, kn) in PRESETS.items():
        st = Stencil.from_file(path)
        ck = kn.to_c()
        _check(lib().drs_plan_warm_cache(st._h, ctypes.byref(ck)))
        n += 1
        if verbose:
            print("warm_cache:", name)
    return n
