"""Host-side mirror of the reference's accelerator interface over the C-ABI.

`NKA` follows the F08 type-bound API (src-F08/nka_type.F90:169-181): init,
set_vec_tol, accel_update, relax, restart, num_vec, max_vec, vec_len, vec_tol,
defined -- plus delete (src-F95/nka_type.F90:266-275).  The module-level
nka_* functions follow the C header (src-C/nonlinear_krylov_accelerator.h:3-12).

Vectors are torch CUDA tensors (float64, contiguous; zero copy) or numpy /
CPU-tensor host arrays (staged through the device inside the call).  Python is
only the binding: every number is produced by the CUDA kernels in
libnka_b200.so, and nothing here computes on the CPU.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib


class NKAError(RuntimeError):
    pass


def _is_torch(x) -> bool:
    return type(x).__module__.startswith("torch")


class NKA:
    """type(nka) of the reference, device resident."""

    def __init__(self, vlen: int | None = None, mvec: int | None = None, vtol: float = 0.01,
                 device: int = -1, stream: int | None = None):
        self._h = None
        self._lib = _lib.load()
        if vlen is not None:
            self.init(vlen, mvec, vtol=vtol, device=device, stream=stream)

    # -- life cycle -------------------------------------------------------
    def init(self, vlen: int, mvec: int, vtol: float = 0.01, device: int = -1, stream: int | None = None):
        """init(vlen, mvec): src-F08/nka_type.F90:185-200.  Re-initialising frees
        the previous storage (the Fortran dummy is intent(out))."""
        # the reference ASSERTs these (src-F08/nka_type.F90:190-191,205); the C
        # library aborts on them, so the binding raises first
        if mvec is None or mvec <= 0:
            raise ValueError("mvec must be > 0")
        if mvec > _lib.MAX_MVEC:
            raise ValueError("mvec > %d is not supported by this build" % _lib.MAX_MVEC)
        if vlen < 0:
            raise ValueError("vlen must be >= 0")
        if not vtol > 0.0:
            raise ValueError("vtol must be > 0")
        self.delete()
        self._h = self._lib.nka_init_ex(vlen, mvec, vtol, device, stream)
        if not self._h:
            raise NKAError("nka_init_ex returned NULL")
        self._vlen = vlen
        return self

    def delete(self):
        if self._h:
            self._lib.nka_delete(self._h)
            self._h = None

    def __del__(self):
        try:
            self.delete()
        except Exception:
            pass

    def _handle(self):
        if not self._h:
            raise NKAError("accelerator is not initialised")
        return self._h

    def _uncaptured(self, call: str, why: str):
        """The handle, or NKAError while its stream is capturing: `call` cannot be part of a CUDA
        graph, and the library would abort on it."""
        h = self._handle()
        if self._lib.nka_stream_capturing(h) != 0:
            raise NKAError("%s cannot be captured in a CUDA graph: %s" % (call, why))
        return h

    # -- the hot path -----------------------------------------------------
    def accel_update(self, f) -> None:
        """accel_update(f): f is overwritten with the accelerated correction
        (src-F08/nka_type.F90:249-419).  A CUDA tensor f can be captured in a CUDA graph
        (INTEGRATION.md, "CUDA graphs"); a host f cannot."""
        h = self._handle()
        if _is_torch(f):
            import torch
            if f.dtype != torch.float64 or not f.is_contiguous() or f.numel() != self._vlen:
                raise ValueError("f must be a contiguous float64 tensor of length vlen")   # ASSERT(size(f) == vlen) :258
            if f.is_cuda:
                if getattr(self, "_dp_keepalive", None) is not None:
                    self._uncaptured("accel_update", "the handle sums its dot products through a host callback")
                self._lib.nka_accel_update_dev(h, f.data_ptr())
            else:
                self._uncaptured("accel_update of a host f", "it is staged through the device and synchronises")
                self._lib.nka_accel_update_host(h, f.data_ptr())
        else:
            if not isinstance(f, np.ndarray) or f.dtype != np.float64 or not f.flags["C_CONTIGUOUS"] \
                    or f.size != self._vlen:
                raise ValueError("f must be a contiguous float64 array of length vlen")
            self._uncaptured("accel_update of a host f", "it is staged through the device and synchronises")
            self._lib.nka_accel_update_host(h, f.ctypes.data)

    def relax(self): self._lib.nka_relax(self._handle())
    def restart(self): self._lib.nka_restart(self._handle())

    def set_dot_prod(self, dp) -> None:
        """set_dot_prod(dot_prod): src-F08/nka_type.F90:209-219.  dp(n, x, y) is a ctypes callback of the
        C header's type (double (*)(int, double*, double*)) or None; the library calls it with n = 1 to
        make each of this process's partial dot products global (include/nonlinear_krylov_accelerator.h)."""
        h = self._uncaptured("set_dot_prod", "it changes the launch shape of later updates")
        self._dp_keepalive = dp
        self._lib.nka_set_dot_prod(h, C.cast(dp, C.c_void_p) if dp is not None else None)

    def set_vec_tol(self, vtol: float):
        if not vtol > 0.0:
            raise ValueError("vtol must be > 0")
        self._lib.nka_set_vec_tol(self._handle(), vtol)

    # -- queries ----------------------------------------------------------
    def num_vec(self) -> int: return self._lib.nka_num_vec(self._uncaptured("num_vec", "it copies the device state to the host and synchronises"))
    def max_vec(self) -> int: return self._lib.nka_max_vec(self._handle())
    def vec_len(self) -> int: return self._lib.nka_vec_len64(self._handle())
    def vec_tol(self) -> float: return self._lib.nka_vec_tol(self._handle())
    def defined(self) -> bool:
        return bool(self._h) and bool(self._lib.nka_defined(self._uncaptured("defined", "it copies the device state to the host and synchronises")))

    # -- additive: streams, distributed, introspection --------------------
    def set_stream(self, stream: int | None):
        """The stream every later call is queued on.  To capture calls in a CUDA graph, set the capture
        stream here before the capture begins."""
        self._lib.nka_set_stream(self._uncaptured("set_stream", "it synchronises the handle's stream"), stream)

    def synchronize(self): self._lib.nka_synchronize(self._uncaptured("synchronize", "it synchronises the handle's stream"))

    def stream_capturing(self) -> int:
        """1 while the handle's stream is capturing a CUDA graph, 0 when not, -1 when the handle is on
        the legacy default stream while a blocking stream captures (include/nka_b200.h)."""
        return self._lib.nka_stream_capturing(self._handle())

    def comm_init(self, nranks: int, rank: int, unique_id: bytes):
        buf = C.create_string_buffer(unique_id, 128)
        rc = self._lib.nka_comm_init(self._uncaptured("comm_init", "it is a collective that synchronises"),
                                     nranks, rank, buf)
        if rc != 0:
            raise NKAError("nka_comm_init failed with NCCL code %d" % rc)

    def comm_mode(self) -> str:
        """How the partial dot products are summed across ranks (include/nka_b200.h: nka_comm_mode)."""
        return ("single", "nccl", "peer")[self._lib.nka_comm_mode(self._handle())]

    def state(self) -> dict:
        v = _lib.StateView()
        self._lib.nka_get_state(self._uncaptured("state", "it copies the device state to the host and synchronises"), C.byref(v))
        n = v.mvec + 1
        return {
            "subspace": v.subspace, "pending": v.pending, "first": v.first, "last": v.last,
            "free": v.free_slot, "next": list(v.next[:n]), "prev": list(v.prev[:n]),
            "chained": list(v.chained[:n]), "ndrop_last": v.ndrop_last, "evicted_last": v.evicted_last,
            "relaxed_last": v.relaxed_last, "error": v.error, "vtol": v.vtol, "min_margin": v.min_margin,
            "s_last": v.s_last, "c": np.array(v.c[:n]), "s": np.array(v.s[:n]),
            "h": np.array(v.h[: n * n]).reshape(n, n), "ncalls": v.ncalls,
        }

    def launch_count(self) -> int: return self._lib.nka_launch_count(self._handle())
    def timing_enable(self, on: bool = True):
        self._lib.nka_timing_enable(self._uncaptured("timing_enable", "it synchronises the handle's stream"), int(on))

    def timing_reset(self): self._lib.nka_timing_reset(self._uncaptured("timing_reset", "it synchronises the handle's stream"))

    def timing_read(self) -> dict:
        ms = (C.c_double * 5)()
        cnt = (C.c_ulonglong * 5)()
        self._lib.nka_timing_read(self._uncaptured("timing_read", "it synchronises the handle's stream"), ms, cnt)
        names = ("pass_a", "state", "materialise", "pass_b", "allreduce")
        return {k: {"ms": ms[i], "count": cnt[i]} for i, k in enumerate(names)}

    def launch_geometry(self) -> dict:
        ga, gb, th = C.c_int(), C.c_int(), C.c_int()
        self._lib.nka_launch_geometry(self._handle(), C.byref(ga), C.byref(gb), C.byref(th))
        return {"grid_a": ga.value, "grid_b": gb.value, "threads": th.value}


def comm_unique_id() -> bytes:
    buf = C.create_string_buffer(128)
    rc = _lib.load().nka_comm_unique_id(buf)
    if rc != 0:
        raise NKAError("nka_comm_unique_id failed (%d): is libnccl.so.2 loadable?" % rc)
    return buf.raw


# ---- the C header's call shapes (src-C/nonlinear_krylov_accelerator.h:3-12) ----
DP_FUNC = C.CFUNCTYPE(C.c_double, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double))


def nka_init(vlen: int, mvec: int, vtol: float, dp=None) -> NKA:
    """dp: None, or a DP_FUNC callback (the reference's parallel dot-product hook, used for its global sum)."""
    acc = NKA(vlen, mvec, vtol)
    if dp is not None:
        acc.set_dot_prod(dp)
    return acc


def nka_delete(state: NKA): state.delete()
def nka_accel_update(state: NKA, f): state.accel_update(f)
def nka_restart(state: NKA): state.restart()
def nka_relax(state: NKA): state.relax()
def nka_num_vec(state: NKA) -> int: return state.num_vec()
def nka_max_vec(state: NKA) -> int: return state.max_vec()
def nka_vec_len(state: NKA) -> int: return state.vec_len()
def nka_vec_tol(state: NKA) -> float: return state.vec_tol()
