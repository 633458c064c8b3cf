"""Interleaved batched accelerators: `nbatch` independent NKA instances of one length whose vectors are
stored component-major, one thread per member.

Element i of member b sits at f[i*ldf + b], the layout of a Fortran array f(ncell, nvar) with one member
per cell.  Each member gives bit for bit what the reference's C accelerator gives when fed that member's
calls (INTEGRATION.md section 10).  Device-only and single-GPU.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from .batch import _mask_address, _state_dict
from .nka import NKAError, _is_torch

MAX_BATCH = 2**31 - 1


class InterleavedBatchNKA:
    """`nbatch` accelerators sharing vlen, mvec and vtol, stored interleaved and updated together."""

    def __init__(self, nbatch: int | None = None, vlen: int | None = None, mvec: int | None = None,
                 vtol: float = 0.01, device: int = -1, stream: int | None = None):
        self._h = None
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
        self._h = self._lib.nka_ibatch_init(nbatch, vlen, mvec, vtol, device, stream)
        if not self._h:
            raise NKAError("nka_ibatch_init returned NULL")
        self.nbatch, self.vlen, self.mvec = nbatch, vlen, mvec
        return self

    def delete(self):
        if self._h:
            self._lib.nka_ibatch_delete(self._h)
            self._h = None

    def __del__(self):
        try:
            self.delete()
        except Exception:
            pass

    def _handle(self):
        if not self._h:
            raise NKAError("interleaved batched accelerator is not initialised")
        return self._h

    def _uncaptured(self, call: str, why: str):
        h = self._handle()
        if self._lib.nka_ibatch_stream_capturing(h) != 0:
            raise NKAError("%s cannot be captured in a CUDA graph: %s" % (call, why))
        return h

    def _ldf(self, F) -> int:
        """The column stride of F, a CUDA float64 tensor [nbatch, vlen] with unit row stride."""
        if not _is_torch(F):
            raise ValueError("F must be a CUDA float64 tensor of shape [nbatch, vlen]")
        import torch
        if F.dtype != torch.float64 or F.dim() != 2 or tuple(F.shape) != (self.nbatch, self.vlen):
            raise ValueError("F must be a CUDA float64 tensor of shape [nbatch, vlen] = [%d, %d]"
                             % (self.nbatch, self.vlen))
        if F.stride(0) != 1 and self.nbatch > 1:
            raise ValueError("F must be interleaved: unit member stride (F.stride(0) == 1), "
                             "e.g. torch.empty(vlen, nbatch).t()")
        ldf = F.stride(1)
        if ldf < self.nbatch:
            if self.vlen > 1:
                raise ValueError("F's component stride (F.stride(1)) must be >= nbatch")
            ldf = self.nbatch                   # one component: its stride is never used to address anything
        if not F.is_cuda:
            raise ValueError("F must be a CUDA tensor: the interleaved batched accelerator is device-only")
        return ldf

    # -- the hot path -----------------------------------------------------
    def accel_update(self, F, active=None) -> None:
        """F: CUDA float64 tensor [nbatch, vlen] with F.stride(0) == 1 and F.stride(1) = ldf >= nbatch
        (torch.empty(vlen, nbatch).t(), or a Fortran f(ncell, nvar)); row b is member b's f and is
        overwritten with its accelerated correction.  active: optional length-nbatch CUDA bool / uint8
        tensor; an inactive member's elements of F and its state are left exactly as they are.  Capturable."""
        ldf = self._ldf(F)
        a = _mask_address(active, self.nbatch, "active")
        self._lib.nka_ibatch_accel_update(self._handle(), F.data_ptr(), ldf, a)

    def relax(self, mask=None) -> None:
        m = _mask_address(mask, self.nbatch, "mask")
        self._lib.nka_ibatch_relax(self._handle(), m)

    def restart(self, mask=None) -> None:
        m = _mask_address(mask, self.nbatch, "mask")
        self._lib.nka_ibatch_restart(self._handle(), m)

    def set_vec_tol(self, vtol: float) -> None:
        if not vtol > 0.0:
            raise ValueError("vtol must be > 0")
        self._lib.nka_ibatch_set_vec_tol(self._handle(), vtol)

    # -- queries ----------------------------------------------------------
    def num_vec(self) -> np.ndarray:
        out = np.zeros(self.nbatch, dtype=np.int32)
        self._lib.nka_ibatch_num_vec(self._uncaptured("num_vec", "it copies the device state to the host and synchronises"),
                                     out.ctypes.data_as(C.POINTER(C.c_int)))
        return out

    def defined(self) -> bool:
        return bool(self._h) and bool(self._lib.nka_ibatch_defined(
            self._uncaptured("defined", "it copies the device state to the host and synchronises")))

    def state(self, b: int) -> dict:
        """Member b's state, with the keys and layout of NKA.state().  Filled: subspace, pending, first, last,
        free, next, prev, c, h, vtol, min_margin, ndrop_last, evicted_last, relaxed_last; the rest are zero."""
        if not 0 <= b < self.nbatch:
            raise ValueError("member index out of range")
        v = _lib.StateView()
        self._lib.nka_ibatch_get_state(self._uncaptured("state", "it copies the device state to the host and synchronises"),
                                       b, C.byref(v))
        return _state_dict(v)

    def set_stream(self, stream: int | None):
        """The stream every later call is queued on; set the capture stream here before a capture begins."""
        self._lib.nka_ibatch_set_stream(self._uncaptured("set_stream", "it synchronises the handle's stream"), stream)

    def synchronize(self):
        self._lib.nka_ibatch_synchronize(self._uncaptured("synchronize", "it synchronises the handle's stream"))

    def stream_capturing(self) -> int:
        return self._lib.nka_ibatch_stream_capturing(self._handle())

    def launch_count(self) -> int:
        return self._lib.nka_ibatch_launch_count(self._handle())
