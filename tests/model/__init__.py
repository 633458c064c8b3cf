"""TEST-ONLY host model of the device algorithm (see nka_model.cpp)."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
_SO = os.path.join(HERE, "_build", "libnka_model.so")
_lib = None


def lib():
    global _lib
    if _lib is None:
        src = os.path.join(HERE, "nka_model.cpp")
        hdr = os.path.join(ROOT, "nka_b200", "csrc", "nka_state.h")
        stale = (not os.path.exists(_SO)) or any(os.path.getmtime(p) > os.path.getmtime(_SO) for p in (src, hdr))
        if stale:
            os.makedirs(os.path.dirname(_SO), exist_ok=True)
            subprocess.run(["g++", "-O2", "-ffp-contract=off", "-std=c++17", "-fPIC", "-shared", "-Wall",
                            "-o", _SO, src], check=True)
        L = C.CDLL(_SO)
        L.model_init.restype = C.c_void_p
        L.model_init.argtypes = [C.c_size_t, C.c_int, C.c_double]
        L.model_accel_update.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
        L.model_accel_update.restype = None
        for nm in ("model_delete", "model_restart", "model_relax"):
            getattr(L, nm).argtypes = [C.c_void_p]
            getattr(L, nm).restype = None
        for nm in ("model_num_vec", "model_defined", "model_bound_violations", "model_error", "model_ndrop_last",
                   "model_relaxed_last", "model_evicted_last", "model_host_pending", "model_dev_pending",
                   "model_list_len", "model_ub_len", "model_plan_a_ncol", "model_plan_a_skip_last",
                   "model_plan_b_nz", "model_plan_b_has_pair", "model_plan_b_write_f", "model_plan_m_n"):
            getattr(L, nm).argtypes = [C.c_void_p]
            getattr(L, nm).restype = C.c_int
        L.model_mat_entries.argtypes = [C.c_void_p]
        L.model_mat_entries.restype = C.c_ulonglong
        L.model_fixups.argtypes = [C.c_void_p]
        L.model_fixups.restype = C.c_ulonglong
        L.model_plan_a_submask.argtypes = [C.c_void_p]
        L.model_plan_a_submask.restype = C.c_ulonglong
        L.model_set_lazy.argtypes = [C.c_void_p, C.c_int]
        L.model_set_lazy.restype = None
        L.model_min_margin.argtypes = [C.c_void_p]
        L.model_min_margin.restype = C.c_double
        _lib = L
    return _lib


class ModelNKA:
    def __init__(self, vlen, mvec, vtol=0.01, lazy=True):
        self._lib = lib()
        self._h = self._lib.model_init(vlen, mvec, vtol)
        if not self._h:
            raise ValueError("bad arguments")
        self.vlen = vlen
        if not lazy:
            self._lib.model_set_lazy(self._h, 0)

    def fixups(self): return self._lib.model_fixups(self._h)

    def accel_update(self, f: np.ndarray):
        assert f.dtype == np.float64 and f.shape == (self.vlen,)
        self._lib.model_accel_update(self._h, f.ctypes.data_as(C.POINTER(C.c_double)))

    def relax(self): self._lib.model_relax(self._h)
    def restart(self): self._lib.model_restart(self._h)
    def num_vec(self): return self._lib.model_num_vec(self._h)
    def defined(self): return bool(self._lib.model_defined(self._h))
    def bound_violations(self): return self._lib.model_bound_violations(self._h)
    def mat_entries(self): return self._lib.model_mat_entries(self._h)
    def error(self): return self._lib.model_error(self._h)
    def ndrop_last(self): return self._lib.model_ndrop_last(self._h)
    def relaxed_last(self): return self._lib.model_relaxed_last(self._h)
    def evicted_last(self): return self._lib.model_evicted_last(self._h)
    def min_margin(self): return self._lib.model_min_margin(self._h)
    def host_pending(self): return self._lib.model_host_pending(self._h)
    def dev_pending(self): return self._lib.model_dev_pending(self._h)
    def list_len(self): return self._lib.model_list_len(self._h)
    def ub_len(self): return self._lib.model_ub_len(self._h)

    def plan_a(self):
        """Plan A as the next pass A reads it: (ncol, skip_last, submask)."""
        L = self._lib
        return L.model_plan_a_ncol(self._h), L.model_plan_a_skip_last(self._h), L.model_plan_a_submask(self._h)

    def plan_b(self):
        """Plans B and M as the last update left them: (nz, has_pair, write_f, planM.n)."""
        L = self._lib
        return (L.model_plan_b_nz(self._h), L.model_plan_b_has_pair(self._h), L.model_plan_b_write_f(self._h),
                L.model_plan_m_n(self._h))

    def __del__(self):
        try:
            if self._h:
                self._lib.model_delete(self._h)
                self._h = None
        except Exception:
            pass
