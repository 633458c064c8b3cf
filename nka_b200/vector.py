"""gpu_vector: the reference's abstract `vector` interface (src-F08-vector/vector_class.F90:90-109)
over device memory, and the vector flavour of the accelerator
(src-F08-vector/nka_type.F90:148-171).  Python is the binding only; every operation is a CUDA
kernel in libnka_b200.so (nka_vec.cu).

The non-virtual wrappers of the base class keep their zero-coefficient short cuts
(vector_class.F90:176,189,203-206,219-222) and their "incompatible arguments" errors."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from .nka import NKAError


class GpuVector:
    def __init__(self, n: int | None = None, device: int = -1, stream: int | None = None, _handle=None):
        self._lib = _lib.load()
        self._h = _handle
        if _handle is None:
            if n is None or n < 0:
                raise ValueError("n must be >= 0")
            self._h = self._lib.nka_vec_create(n, device, stream)

    # -- clone / copy ------------------------------------------------------
    def clone(self, n: int | None = None):
        """clone1 (a copy) or clone2 (a list of n copies): vector_class.F90:92-93."""
        if n is None:
            return GpuVector(_handle=self._lib.nka_vec_clone(self._h))
        return [GpuVector(_handle=self._lib.nka_vec_clone(self._h)) for _ in range(n)]

    def _same(self, other, what):
        if not isinstance(other, GpuVector) or len(other) != len(self):
            raise TypeError("incompatible arguments to VECTOR%%%s" % what)   # error stop in the reference

    def copy(self, src):
        self._same(src, "COPY")
        self._lib.nka_vec_copy(self._h, src._h)

    def setval(self, val: float): self._lib.nka_vec_setval(self._h, val)
    def scale(self, a: float): self._lib.nka_vec_scale(self._h, a)

    def update(self, a, x, b=None, y=None, c=None):
        """The generic `update` (update1..update4 by argument count), vector_class.F90:171-228."""
        if b is None:                                   # update1: this += a*x
            if a == 0.0:
                return
            self._same(x, "UPDATE")
            self._lib.nka_vec_update1(self._h, a, x._h)
        elif y is None:                                 # update2: this = a*x + b*this
            if a == 0.0:
                return self.scale(b)
            self._same(x, "UPDATE")
            self._lib.nka_vec_update2(self._h, a, x._h, b)
        elif c is None:                                 # update3: this = a*x + b*y + this
            if a == 0.0:
                return self.update(b, y)
            if b == 0.0:
                return self.update(a, x)
            self._same(x, "UPDATE"); self._same(y, "UPDATE")
            self._lib.nka_vec_update3(self._h, a, x._h, b, y._h)
        else:                                           # update4: this = a*x + b*y + c*this
            if a == 0.0:
                return self.update(b, y, c)
            if b == 0.0:
                return self.update(a, x, c)
            self._same(x, "UPDATE"); self._same(y, "UPDATE")
            self._lib.nka_vec_update4(self._h, a, x._h, b, y._h, c)

    def dot(self, y) -> float:
        self._same(y, "DOT")
        return self._lib.nka_vec_dot(self._h, y._h)

    def norm2(self) -> float: return self._lib.nka_vec_norm2(self._h)

    # -- data movement -------------------------------------------------------
    def __len__(self): return self._lib.nka_vec_size(self._h)
    def data_ptr(self) -> int: return self._lib.nka_vec_data(self._h)

    def set(self, host: np.ndarray):
        host = np.ascontiguousarray(host, dtype=np.float64)
        if host.size != len(self):
            raise ValueError("length mismatch")
        self._lib.nka_vec_set_host(self._h, host.ctypes.data)

    def get(self) -> np.ndarray:
        out = np.empty(len(self))
        self._lib.nka_vec_get_host(self._h, out.ctypes.data)
        return out

    def comm_init(self, nranks: int, rank: int, unique_id: bytes):
        buf = C.create_string_buffer(unique_id, 128)
        rc = self._lib.nka_vec_comm_init(self._h, nranks, rank, buf)
        if rc != 0:
            raise NKAError("nka_vec_comm_init failed with NCCL code %d" % rc)

    def __del__(self):
        try:
            if self._h:
                self._lib.nka_vec_destroy(self._h)
                self._h = None
        except Exception:
            pass


class VectorNKA:
    """type(nka) of src-F08-vector/nka_type.F90: init(vec, mvec), accel_update(f) on gpu_vectors."""

    def __init__(self):
        self._lib = _lib.load()
        self._h = None

    def init(self, vec: GpuVector, mvec: int, vtol: float = 0.01):
        if mvec <= 0:
            raise ValueError("mvec must be > 0")      # ASSERT(mvec > 0) :180
        if not isinstance(vec, GpuVector):
            raise TypeError("this build accelerates gpu_vector objects only")
        self.delete()
        self._h = self._lib.nka_init_like(vec._h, mvec, vtol)
        return self

    def accel_update(self, f: GpuVector):
        """Can be captured in a CUDA graph on the vectors' stream (INTEGRATION.md, "CUDA graphs")."""
        if not isinstance(f, GpuVector):
            raise TypeError("incompatible arguments to NKA%ACCEL_UPDATE")
        self._lib.nka_accel_update_vec(self._h, f._h)

    def set_vec_tol(self, vtol: float):
        if not vtol > 0.0:
            raise ValueError("vtol must be > 0")
        self._lib.nka_set_vec_tol(self._h, vtol)

    def relax(self): self._lib.nka_relax(self._h)
    def restart(self): self._lib.nka_restart(self._h)
    def max_vec(self): return self._lib.nka_max_vec(self._h)
    def vec_tol(self): return self._lib.nka_vec_tol(self._h)

    def _uncaptured(self, call: str):
        if self._lib.nka_stream_capturing(self._h) != 0:
            raise NKAError("%s cannot be captured in a CUDA graph: it copies the device state to the host "
                           "and synchronises" % call)
        return self._h

    def num_vec(self): return self._lib.nka_num_vec(self._uncaptured("num_vec"))
    def defined(self): return bool(self._h) and bool(self._lib.nka_defined(self._uncaptured("defined")))

    def delete(self):
        if self._h:
            self._lib.nka_delete(self._h)
            self._h = None

    def __del__(self):
        try:
            self.delete()
        except Exception:
            pass
