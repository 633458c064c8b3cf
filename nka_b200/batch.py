"""Batched accelerators: `nbatch` independent NKA instances of one length in one handle.

Each member has its own subspace, list, Gram factor, vtol decisions, relax and restart, and gives bit for
bit what a single `NKA` handle in the capacity shape (INTEGRATION.md section 6) gives when fed that
member's calls.  One batched update is a fixed number of kernel launches whatever `nbatch` is.
Device-only and single-GPU: rows of f are CUDA float64 tensor rows (INTEGRATION.md section 7).
"""
from __future__ import annotations

import ctypes as C
import weakref

import numpy as np

from . import _lib
from .nka import NKAError, _is_torch

MAX_BATCH = 65535


class BatchNKA:
    """`nbatch` accelerators sharing vlen, mvec and vtol, updated together."""

    def __init__(self, nbatch: int | None = None, vlen: int | None = None, mvec: int | None = None,
                 vtol: float = 0.01, device: int = -1, stream: int | None = None):
        self._h = None
        self._loops = weakref.WeakSet()
        self._lib = _lib.load()
        if nbatch is not None:
            self.init(nbatch, vlen, mvec, vtol=vtol, device=device, stream=stream)

    # -- life cycle -------------------------------------------------------
    def init(self, nbatch: int, vlen: int, mvec: int, vtol: float = 0.01, device: int = -1,
             stream: int | None = None):
        """Re-initialising frees the previous storage.  Bad arguments raise ValueError before any CUDA call."""
        if nbatch is None or not 1 <= nbatch <= MAX_BATCH:
            raise ValueError("nbatch must be in 1..%d" % MAX_BATCH)
        if vlen is None or vlen < 1:
            raise ValueError("vlen must be >= 1")
        if mvec is None or mvec <= 0:
            raise ValueError("mvec must be > 0")
        if mvec > _lib.MAX_MVEC:
            raise ValueError("mvec > %d is not supported by this build" % _lib.MAX_MVEC)
        if not vtol > 0.0:
            raise ValueError("vtol must be > 0")
        self.delete()
        self._h = self._lib.nka_batch_init(nbatch, vlen, mvec, vtol, device, stream)
        if not self._h:
            raise NKAError("nka_batch_init returned NULL")
        self.nbatch, self.vlen, self.mvec = nbatch, vlen, mvec
        return self

    def delete(self):
        for loop in list(self._loops):
            loop.destroy()
        if self._h:
            self._lib.nka_batch_delete(self._h)
            self._h = None

    def __del__(self):
        try:
            self.delete()
        except Exception:
            pass

    def _handle(self):
        if not self._h:
            raise NKAError("batched accelerator is not initialised")
        return self._h

    def _uncaptured(self, call: str, why: str):
        h = self._handle()
        if self._lib.nka_batch_stream_capturing(h) != 0:
            raise NKAError("%s cannot be captured in a CUDA graph: %s" % (call, why))
        return h

    def _mask(self, mask, what: str):
        """The device address of a length-nbatch CUDA bool / uint8 tensor, or None for every member."""
        if mask is None:
            return None
        if not _is_torch(mask):
            raise ValueError("%s must be a CUDA bool or uint8 tensor of length nbatch" % what)
        import torch
        if mask.dtype not in (torch.bool, torch.uint8) or not mask.is_cuda or mask.dim() != 1 \
                or mask.numel() != self.nbatch or (self.nbatch > 1 and mask.stride(0) != 1):
            raise ValueError("%s must be a contiguous CUDA bool or uint8 tensor of length nbatch" % what)
        return mask.data_ptr()

    def _rows(self, T, name: str) -> int:
        """The row stride of T, a CUDA float64 tensor [nbatch, vlen] with unit column stride."""
        if not _is_torch(T):
            raise ValueError("%s must be a CUDA float64 tensor of shape [nbatch, vlen]" % name)
        import torch
        if T.dtype != torch.float64 or T.dim() != 2 or tuple(T.shape) != (self.nbatch, self.vlen):
            raise ValueError("%s must be a CUDA float64 tensor of shape [nbatch, vlen] = [%d, %d]"
                             % (name, self.nbatch, self.vlen))
        if T.stride(1) != 1 and self.vlen > 1:
            raise ValueError("%s must have unit column stride (%s.stride(1) == 1)" % (name, name))
        ld = T.stride(0)
        if ld < self.vlen:
            if self.nbatch > 1:
                raise ValueError("%s's row stride must be >= vlen" % name)
            ld = self.vlen                      # one row: its stride is never used to address anything
        if not T.is_cuda:
            raise ValueError("%s must be a CUDA tensor: the batched accelerator is device-only" % name)
        return ld

    # -- the hot path -----------------------------------------------------
    def accel_update(self, F, active=None) -> None:
        """F: CUDA float64 tensor [nbatch, vlen] with unit column stride; row b is member b's f and is
        overwritten with its accelerated correction.  active: optional length-nbatch CUDA bool / uint8
        tensor; an inactive member's row and state are left exactly as they are.  Capturable."""
        ldf = self._rows(F, "F")
        a = self._mask(active, "active")
        self._lib.nka_batch_accel_update(self._handle(), F.data_ptr(), ldf, a)

    def relax(self, mask=None) -> None:
        m = self._mask(mask, "mask")
        self._lib.nka_batch_relax(self._handle(), m)

    def restart(self, mask=None) -> None:
        m = self._mask(mask, "mask")
        self._lib.nka_batch_restart(self._handle(), m)

    def set_vec_tol(self, vtol: float) -> None:
        if not vtol > 0.0:
            raise ValueError("vtol must be > 0")
        self._lib.nka_batch_set_vec_tol(self._handle(), vtol)

    # -- queries ----------------------------------------------------------
    def num_vec(self) -> np.ndarray:
        out = np.zeros(self.nbatch, dtype=np.int32)
        self._lib.nka_batch_num_vec(self._uncaptured("num_vec", "it copies the device state to the host and synchronises"),
                                    out.ctypes.data_as(C.POINTER(C.c_int)))
        return out

    def defined(self) -> bool:
        return bool(self._h) and bool(self._lib.nka_batch_defined(
            self._uncaptured("defined", "it copies the device state to the host and synchronises")))

    def state(self, b: int) -> dict:
        """Member b's state, with the keys and layout of NKA.state()."""
        if not 0 <= b < self.nbatch:
            raise ValueError("member index out of range")
        v = _lib.StateView()
        self._lib.nka_batch_get_state(self._uncaptured("state", "it copies the device state to the host and synchronises"),
                                      b, C.byref(v))
        n = v.mvec + 1
        return {
            "subspace": v.subspace, "pending": v.pending, "first": v.first, "last": v.last,
            "free": v.free_slot, "next": list(v.next[:n]), "prev": list(v.prev[:n]),
            "chained": list(v.chained[:n]), "ndrop_last": v.ndrop_last, "evicted_last": v.evicted_last,
            "relaxed_last": v.relaxed_last, "error": v.error, "vtol": v.vtol, "min_margin": v.min_margin,
            "s_last": v.s_last, "c": np.array(v.c[:n]), "s": np.array(v.s[:n]),
            "h": np.array(v.h[: n * n]).reshape(n, n), "ncalls": v.ncalls,
        }

    def set_stream(self, stream: int | None):
        """The stream every later call is queued on; set the capture stream here before a capture begins."""
        self._lib.nka_batch_set_stream(self._uncaptured("set_stream", "it synchronises the handle's stream"), stream)

    def synchronize(self):
        self._lib.nka_batch_synchronize(self._uncaptured("synchronize", "it synchronises the handle's stream"))

    def stream_capturing(self) -> int:
        return self._lib.nka_batch_stream_capturing(self._handle())

    def launch_count(self) -> int:
        return self._lib.nka_batch_launch_count(self._handle())

    # -- device-side fixed-point loops --------------------------------------
    def fixed_point_loop(self, residual, X, F, atol: float = 0.0, rtol: float = 1e-8,
                         maxit: int = 100) -> "FixedPointLoop":
        """A solve of x_b = G(x_b) for every member that runs to its end in one graph launch
        (INTEGRATION.md section 8).  residual: a zero-argument callable writing F = G(X) - X in place with
        torch ops; it is run once to warm up, then captured.  X, F: CUDA float64 tensors [nbatch, vlen]
        with unit column stride.  A member stops when ||F_b|| is not finite, when ||F_b|| <
        max(atol, rtol * (its norm at the launch's first check)), or after maxit steps."""
        if isinstance(atol, bool) or not isinstance(atol, (int, float)) or not atol >= 0.0:
            raise ValueError("atol must be a number >= 0")
        if isinstance(rtol, bool) or not isinstance(rtol, (int, float)) or not rtol >= 0.0:
            raise ValueError("rtol must be a number >= 0")
        if isinstance(maxit, bool) or not isinstance(maxit, (int, np.integer)) or maxit < 0 or maxit > 2**31 - 2:
            raise ValueError("maxit must be an integer >= 0")
        ldx = self._rows(X, "X")
        ldf = self._rows(F, "F")
        h = self._uncaptured("fixed_point_loop", "it captures the residual and synchronises")
        import torch
        side = torch.cuda.Stream(device=F.device)
        side.wait_stream(torch.cuda.current_stream(F.device))
        with torch.cuda.stream(side):
            residual()
        torch.cuda.current_stream(F.device).wait_stream(side)
        graph = torch.cuda.CUDAGraph(keep_graph=True)
        with torch.cuda.graph(graph):
            residual()
        torch.cuda.synchronize(F.device)
        loop = FixedPointLoop(self, graph, X, F, int(maxit))
        loop._h = self._lib.nka_batch_loop_create(h, graph.raw_cuda_graph(), X.data_ptr(), ldx, F.data_ptr(), ldf,
                                                  float(atol), float(rtol), int(maxit))
        if not loop._h:
            raise NKAError("nka_batch_loop_create returned NULL: CUDA refused the residual graph or the driver "
                           "has no conditional graph nodes (the reason is printed on stderr)")
        self._loops.add(loop)
        return loop


class FixedPointLoop:
    """A device-side fixed-point loop over a BatchNKA (BatchNKA.fixed_point_loop).  Keeps the captured
    residual graph (and its memory pool), X, F and the batch alive."""

    def __init__(self, batch: BatchNKA, graph, X, F, maxit: int):
        self._h = None
        self._batch, self._graph, self._X, self._F = batch, graph, X, F
        self._lib = batch._lib
        self.maxit = maxit

    def _handle(self, call: str, why: str | None = None):
        if not self._h:
            raise NKAError("fixed-point loop is destroyed")
        if why is not None:
            self._batch._uncaptured(call, why)
        return self._h

    def run(self) -> None:
        """One graph launch on the batch's stream: the whole solve.  Returns at once."""
        self._lib.nka_batch_loop_launch(self._handle(
            "run", "a graph with conditional nodes cannot become a child of another graph"))

    def results(self):
        """(steps, status, norm) per member as numpy arrays; status is one of RUNNING, CONVERGED, MAXIT,
        NONFINITE.  Synchronises."""
        h = self._handle("results", "it copies the loop's results to the host and synchronises")
        nb = self._batch.nbatch
        it = np.zeros(nb, dtype=np.int32)
        st = np.zeros(nb, dtype=np.int32)
        norm = np.zeros(nb, dtype=np.float64)
        self._lib.nka_batch_loop_results(h, it.ctypes.data_as(C.POINTER(C.c_int)), st.ctypes.data_as(C.POINTER(C.c_int)),
                                         norm.ctypes.data_as(C.POINTER(C.c_double)))
        return it, st, norm

    def history(self) -> np.ndarray:
        """[(maxit+1), nbatch]: row k holds each member's norm at check k, NaN where it made none.  Synchronises."""
        h = self._handle("history", "it copies the loop's history to the host and synchronises")
        out = np.zeros((self.maxit + 1, self._batch.nbatch), dtype=np.float64)
        self._lib.nka_batch_loop_history(h, out.ctypes.data_as(C.POINTER(C.c_double)))
        return out

    def destroy(self) -> None:
        if self._h:
            self._lib.nka_batch_loop_destroy(self._h)
            self._h = None
        self._batch._loops.discard(self)

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass


RUNNING, CONVERGED, MAXIT, NONFINITE = 0, 1, 2, 3
