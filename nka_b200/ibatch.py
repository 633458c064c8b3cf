"""Interleaved batched accelerators: `nbatch` independent NKA instances of one length whose vectors are
stored component-major, one thread per member.

Element i of member b sits at f[i*ldf + b], the layout of a Fortran array f(ncell, nvar) with one member
per cell.  Each member gives bit for bit what the reference's C accelerator gives when fed that member's
calls (INTEGRATION.md section 10).  Device-only and single-GPU.
"""
from __future__ import annotations

from .batch import _Batch
from .nka import NKAError, _is_torch

MAX_BATCH = 2**31 - 1


class InterleavedBatchNKA(_Batch):
    """`nbatch` accelerators sharing vlen, mvec and vtol, stored interleaved and updated together.  state(b)
    fills subspace, pending, first, last, free, next, prev, c, h, vtol, min_margin, ndrop_last, evicted_last
    and relaxed_last; the rest are zero."""
    _prefix = "nka_ibatch"
    _max_batch = MAX_BATCH
    _name = "interleaved batched accelerator"

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
        a = self._mask(active, "active")
        self._lib.nka_ibatch_accel_update(self._handle(), F.data_ptr(), ldf, a)
