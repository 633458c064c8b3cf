"""Residual-growth restarts without a GPU: the restart_growth checks of fixed_point_loop / fixed_point_queue
that raise before any CUDA call, the ctypes bindings of the four new entry points against the header, and
the guard kernels' code generation (cuobjdump on nka_batch_guard.o)."""
import ctypes as C
import os
import re

import pytest

from test_batch_cpu import _unbuilt
from test_loop_cpu import _res_usage

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW = ("nka_batch_loop_create_restart", "nka_batch_queue_create_restart", "nka_batch_loop_restarts",
       "nka_batch_queue_restarts")


def test_restart_growth_is_validated_before_any_cuda_call():
    import numpy as np
    import torch
    b = _unbuilt(4, 10)
    rows = torch.zeros(4, 10, dtype=torch.float64)          # CPU tensors: a valid gamma fails on "CUDA" later
    sp, x0 = torch.zeros(4, dtype=torch.int32), torch.zeros(9, 10, dtype=torch.float64)
    for gamma in (True, False, "1", None, [1.0], -1.0, -1e-300, float("nan"), float("inf"), -float("inf"),
                  np.float64("nan")):
        with pytest.raises(ValueError, match="restart_growth"):
            b.fixed_point_loop(lambda: None, rows, rows, restart_growth=gamma)
        with pytest.raises(ValueError, match="restart_growth"):
            b.fixed_point_queue(lambda: None, rows, rows, sp, x0, restart_growth=gamma)
    for gamma in (0, 0.0, 0.5, 1, 2.0, 1e300, np.float64(1.5), np.int32(3)):
        with pytest.raises(ValueError, match="X must be a CUDA tensor"):
            b.fixed_point_loop(lambda: None, rows, rows, restart_growth=gamma)


def _header_params(name):
    text = open(os.path.join(ROOT, "include", "nka_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    m = re.search(r"\b%s\s*\(([^;]*?)\)\s*;" % name, text, re.S)
    assert m, name
    return [" ".join(p.split()) for p in m.group(1).split(",")]


def _ctype_of(param):
    """The ctypes type _lib binds a header parameter as: device addresses and handles as void pointers, the
    stop test as a pointer to StopTest, host arrays as typed pointers, scalars by value."""
    from nka_b200 import _lib
    name = param.split()[-1].lstrip("*")
    if "nka_stop_test *" in param:
        return C.POINTER(_lib.StopTest)
    if "*" in param:
        if name.endswith("_dev") or param.startswith("struct ") or param.startswith("void *"):
            return C.c_void_p
        return {"int": C.POINTER(C.c_int), "double": C.POINTER(C.c_double)}[param.split()[0]]
    return {"size_t": C.c_size_t, "double": C.c_double, "int": C.c_int}[param.split()[0]]


def test_ctypes_bindings_agree_with_the_header():
    from nka_b200 import _lib
    for name in NEW:
        res, args = _lib.SYMBOLS[name]
        params = _header_params(name)
        assert args == [_ctype_of(p) for p in params], (name, params, args)
        assert res == (None if name.endswith("_restarts") else C.c_void_p), name
    # the _restart creates are the _stop creates plus one double
    for kind in ("loop", "queue"):
        stop = _lib.SYMBOLS["nka_batch_%s_create_stop" % kind][1]
        assert _lib.SYMBOLS["nka_batch_%s_create_restart" % kind][1] == stop + [C.c_double]


def test_guard_kernels_have_no_local_memory():
    from nka_b200 import build
    build.build_library()
    res = _res_usage(os.path.join(build.LIB_DIR, "nka_batch_guard.o"))
    assert len(res) == 2 and all(n.startswith(("_Z14nka_loop_guard", "_Z20nka_loop_guard_reset")) for n in res), res
    assert all(local == 0 for local in res.values()), res
