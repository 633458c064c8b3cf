"""ctypes bindings for the parity checker (TEST INFRASTRUCTURE ONLY).

``OracleNKA``  -- our C restatement (oracle/nka_oracle.c).
``RefNKA``     -- the reference's own C library compiled into oracle/_ref/
                  (None-able: absent if it was never built in this tree).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
``--impl reference`` legs may import this module.  nka_b200/ never does.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import build as _build

_dbl_p = C.POINTER(C.c_double)
_int_p = C.POINTER(C.c_int)
# the reference's dp hook: double dp(int n, double *x, double *y)
DP_FUNC = C.CFUNCTYPE(C.c_double, C.c_int, _dbl_p, _dbl_p)


def _dp(a: np.ndarray):
    assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(_dbl_p)


_oracle_lib = None


def oracle_lib() -> C.CDLL:
    global _oracle_lib
    if _oracle_lib is None:
        lib = C.CDLL(_build.build_oracle())
        lib.orc_nka_init.restype = C.c_void_p
        lib.orc_nka_init.argtypes = [C.c_size_t, C.c_int, C.c_double, C.c_int, C.c_int]
        for name in ("orc_nka_delete", "orc_nka_restart", "orc_nka_relax"):
            getattr(lib, name).restype = None
            getattr(lib, name).argtypes = [C.c_void_p]
        lib.orc_nka_accel_update.restype = None
        lib.orc_nka_accel_update.argtypes = [C.c_void_p, _dbl_p]
        lib.orc_nka_set_dp.restype = None
        lib.orc_nka_set_dp.argtypes = [C.c_void_p, C.c_void_p]
        lib.orc_nka_set_vec_tol.restype = None
        lib.orc_nka_set_vec_tol.argtypes = [C.c_void_p, C.c_double]
        for name in ("orc_nka_num_vec", "orc_nka_max_vec", "orc_nka_defined", "orc_nka_ndrop_last",
                     "orc_nka_evicted_last", "orc_nka_relaxed_last"):
            getattr(lib, name).restype = C.c_int
            getattr(lib, name).argtypes = [C.c_void_p]
        lib.orc_nka_vec_len.restype = C.c_size_t
        lib.orc_nka_vec_len.argtypes = [C.c_void_p]
        lib.orc_nka_vec_tol.restype = C.c_double
        lib.orc_nka_vec_tol.argtypes = [C.c_void_p]
        lib.orc_nka_min_margin.restype = C.c_double
        lib.orc_nka_min_margin.argtypes = [C.c_void_p]
        lib.orc_nka_get_lists.restype = None
        lib.orc_nka_get_lists.argtypes = [C.c_void_p, _int_p, _int_p, _int_p]
        lib.orc_nka_get_h.restype = None
        lib.orc_nka_get_h.argtypes = [C.c_void_p, _dbl_p]
        lib.orc_nka_get_coeffs.restype = C.c_int
        lib.orc_nka_get_coeffs.argtypes = [C.c_void_p, _dbl_p]
        lib.orc_system_init.restype = C.c_void_p
        lib.orc_system_init.argtypes = [C.c_int, C.c_int, C.c_double, C.c_int]
        lib.orc_system_delete.restype = None
        lib.orc_system_delete.argtypes = [C.c_void_p]
        lib.orc_residual.restype = None
        lib.orc_residual.argtypes = [C.c_void_p, _dbl_p, _dbl_p]
        lib.orc_ssor.restype = None
        lib.orc_ssor.argtypes = [C.c_void_p, C.c_int, C.c_double, _dbl_p]
        lib.orc_l2norm.restype = C.c_double
        lib.orc_l2norm.argtypes = [_dbl_p, C.c_size_t]
        lib.orc_example_solve.restype = C.c_int
        lib.orc_example_solve.argtypes = [C.c_int, C.c_int, C.c_double, C.c_int, C.c_double, C.c_int,
                                          C.c_double, C.c_int, C.c_int, C.c_int, C.c_double,
                                          _dbl_p, _dbl_p, _dbl_p, _dbl_p, _int_p]
        lib.orc_format_line.restype = C.c_int
        lib.orc_format_line.argtypes = [C.c_char_p, C.c_size_t, C.c_int, C.c_double, C.c_double]
        _oracle_lib = lib
    return _oracle_lib


class OracleNKA:
    """The restatement, with the reference C header's call shapes.

    dotmode 0 = the reference's serial sum, 1 = long double accumulation.
    flavour 0 = C correction statement, 1 = Fortran association.
    dp = a dot product with the signature of the reference's `dp` hook (a ctypes function
    pointer, e.g. DP_FUNC(callable)); it replaces every dot product, as in the reference."""

    def __init__(self, vlen: int, mvec: int, vtol: float = 0.01, dotmode: int = 0, flavour: int = 0, dp=None):
        self._lib = oracle_lib()
        self._h = self._lib.orc_nka_init(vlen, mvec, vtol, dotmode, flavour)
        if not self._h:
            raise ValueError("orc_nka_init rejected its arguments")
        self._dp = dp                      # keeps a Python callback alive as long as the handle
        if dp is not None:
            self._lib.orc_nka_set_dp(self._h, C.cast(dp, C.c_void_p))
        self.vlen, self.mvec = vlen, mvec

    def accel_update(self, f: np.ndarray) -> None:
        assert f.shape == (self.vlen,)
        self._lib.orc_nka_accel_update(self._h, _dp(f))

    def restart(self): self._lib.orc_nka_restart(self._h)
    def relax(self): self._lib.orc_nka_relax(self._h)
    def set_vec_tol(self, vtol: float): self._lib.orc_nka_set_vec_tol(self._h, vtol)
    def num_vec(self) -> int: return self._lib.orc_nka_num_vec(self._h)
    def max_vec(self) -> int: return self._lib.orc_nka_max_vec(self._h)
    def vec_len(self) -> int: return self._lib.orc_nka_vec_len(self._h)
    def vec_tol(self) -> float: return self._lib.orc_nka_vec_tol(self._h)
    def defined(self) -> bool: return bool(self._lib.orc_nka_defined(self._h))
    def min_margin(self) -> float: return self._lib.orc_nka_min_margin(self._h)
    def ndrop_last(self) -> int: return self._lib.orc_nka_ndrop_last(self._h)
    def evicted_last(self) -> bool: return bool(self._lib.orc_nka_evicted_last(self._h))
    def relaxed_last(self) -> bool: return bool(self._lib.orc_nka_relaxed_last(self._h))

    def lists(self) -> dict:
        n = self.mvec + 1
        out = (C.c_int * 5)()
        nxt = (C.c_int * n)()
        prv = (C.c_int * n)()
        self._lib.orc_nka_get_lists(self._h, out, nxt, prv)
        return {"subspace": out[0], "pending": out[1], "first": out[2], "last": out[3], "free": out[4],
                "next": list(nxt), "prev": list(prv)}

    def h(self) -> np.ndarray:
        n = self.mvec + 1
        a = np.zeros((n, n))
        self._lib.orc_nka_get_h(self._h, _dp(a))
        return a

    def coeffs(self) -> np.ndarray:
        a = np.zeros(self.mvec + 1)
        m = self._lib.orc_nka_get_coeffs(self._h, _dp(a))
        return a[:m].copy()

    def close(self):
        if self._h:
            self._lib.orc_nka_delete(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_ref_lib = None


def ref_lib() -> C.CDLL | None:
    """The compiled reference (oracle/_ref/libnka_ref.so), or None."""
    global _ref_lib
    if _ref_lib is None:
        path, _ = _build.build_reference()
        if path is None:
            return None
        lib = C.CDLL(path)
        # src-C/nonlinear_krylov_accelerator.h:3-12
        lib.nka_init.restype = C.c_void_p
        lib.nka_init.argtypes = [C.c_int, C.c_int, C.c_double, C.c_void_p]
        for name in ("nka_delete", "nka_restart", "nka_relax"):
            getattr(lib, name).restype = None
            getattr(lib, name).argtypes = [C.c_void_p]
        lib.nka_accel_update.restype = None
        lib.nka_accel_update.argtypes = [C.c_void_p, _dbl_p]
        for name in ("nka_num_vec", "nka_max_vec", "nka_vec_len"):
            getattr(lib, name).restype = C.c_int
            getattr(lib, name).argtypes = [C.c_void_p]
        lib.nka_vec_tol.restype = C.c_double
        lib.nka_vec_tol.argtypes = [C.c_void_p]
        _ref_lib = lib
    return _ref_lib


class RefNKA:
    """The reference's own C accelerator (unmodified source, compiled here).

    long_double_dp=True injects a long-double dot product through the
    reference's documented `dp` hook (src-C/...c:227-231)."""

    def __init__(self, vlen: int, mvec: int, vtol: float = 0.01, long_double_dp: bool = False):
        lib = ref_lib()
        if lib is None:
            raise RuntimeError("oracle/_ref/libnka_ref.so is not built (no /root/reference here)")
        if (mvec + 1) * vlen >= 2 ** 31:
            raise OverflowError("reference nka_init overflows int for (mvec+1)*vlen >= 2^31")
        self._lib = lib
        dp = None
        if long_double_dp:
            dp = C.cast(oracle_lib().orc_dp_long_double, C.c_void_p)
        self._h = lib.nka_init(vlen, mvec, vtol, dp)
        self.vlen, self.mvec = vlen, mvec

    def accel_update(self, f: np.ndarray) -> None:
        assert f.shape == (self.vlen,)
        self._lib.nka_accel_update(self._h, _dp(f))

    def restart(self): self._lib.nka_restart(self._h)
    def relax(self): self._lib.nka_relax(self._h)
    def num_vec(self) -> int: return self._lib.nka_num_vec(self._h)
    def max_vec(self) -> int: return self._lib.nka_max_vec(self._h)
    def vec_len(self) -> int: return self._lib.nka_vec_len(self._h)
    def vec_tol(self) -> float: return self._lib.nka_vec_tol(self._h)

    def close(self):
        if self._h:
            self._lib.nka_delete(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass



class _OrcSystemStruct(C.Structure):
    """oracle/nka_oracle.c: struct orc_system"""
    _fields_ = [("nx", C.c_int), ("ny", C.c_int), ("scaling", C.c_int),
                ("a", C.c_double), ("hx", C.c_double), ("hy", C.c_double),
                ("ax", _dbl_p), ("ay", _dbl_p), ("ac", _dbl_p), ("q", _dbl_p)]


class OracleSystem:
    """The restated example system (system_type: src-F08/nka_example.F90:67-181), one call at a
    time, natural order: r[k*nx + j]; u is padded (ny+2, nx+2) with the boundary values."""

    def __init__(self, nx: int, ny: int, a: float = 0.02, scaling: int = 1):
        self._lib = oracle_lib()
        self.nx, self.ny = nx, ny
        self._h = self._lib.orc_system_init(nx, ny, a, scaling)

    def residual(self, upad: np.ndarray) -> np.ndarray:
        r = np.zeros(self.nx * self.ny)
        self._lib.orc_residual(self._h, _dp(np.ascontiguousarray(upad, dtype=np.float64).ravel()), _dp(r))
        return r

    def pc_ssor(self, nsweep: int, omega: float, r: np.ndarray) -> np.ndarray:
        z = np.array(r, dtype=np.float64).ravel().copy()
        self._lib.orc_ssor(self._h, nsweep, omega, _dp(z))
        return z

    def coefficients(self):
        """(ax[(ny, nx+1)], ay[(ny+1, nx)], ac[(ny, nx)]) of the last residual call."""
        st = C.cast(self._h, C.POINTER(_OrcSystemStruct)).contents
        nx, ny = self.nx, self.ny
        ax = np.ctypeslib.as_array(st.ax, shape=(ny * (nx + 1),)).reshape(ny, nx + 1).copy()
        ay = np.ctypeslib.as_array(st.ay, shape=((ny + 1) * nx,)).reshape(ny + 1, nx).copy()
        ac = np.ctypeslib.as_array(st.ac, shape=(ny * nx,)).reshape(ny, nx).copy()
        return ax, ay, ac

    @staticmethod
    def norm2(x: np.ndarray) -> float:
        x = np.ascontiguousarray(x, dtype=np.float64).ravel()
        return oracle_lib().orc_l2norm(_dp(x), x.size)

    def close(self):
        if self._h:
            self._lib.orc_system_delete(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def example_solve(nx=50, ny=50, a=0.02, nsweep=2, omega=1.4, mvec=5, vtol=0.01, scaling=0,
                  flavour=0, maxitr=999, tol=1.0e-6, record=False):
    """Run the restated example; returns dict(iters, rnorm[, fseq, gseq, nvec], u)."""
    lib = oracle_lib()
    n = nx * ny
    rnorm = np.zeros(maxitr + 1)
    upad = np.zeros((ny + 2) * (nx + 2))
    fseq = gseq = None
    nvec = None
    if record and mvec > 0:
        fseq = np.zeros((maxitr, n))
        gseq = np.zeros((maxitr, n))
        nvec = np.zeros(maxitr, dtype=np.int32)
    it = lib.orc_example_solve(nx, ny, a, nsweep, omega, mvec, vtol, scaling, flavour, maxitr, tol,
                               _dp(rnorm), _dp(upad),
                               _dp(fseq) if fseq is not None else None,
                               _dp(gseq) if gseq is not None else None,
                               nvec.ctypes.data_as(_int_p) if nvec is not None else None)
    out = {"iters": it, "rnorm": rnorm[: it + 1].copy(), "u": upad.reshape(ny + 2, nx + 2)}
    if fseq is not None:
        out["fseq"] = fseq[:it].copy()
        out["gseq"] = gseq[:it].copy()
        out["nvec"] = nvec[:it].copy()
    return out


def format_table(rnorm: np.ndarray) -> list[str]:
    """The example's per-iteration lines, formatted as the reference prints them."""
    lib = oracle_lib()
    buf = C.create_string_buffer(128)
    lines = []
    for itr, rn in enumerate(rnorm):
        lib.orc_format_line(buf, 128, itr, float(rn), float(rnorm[0]))
        lines.append(buf.value.decode())
    return lines
