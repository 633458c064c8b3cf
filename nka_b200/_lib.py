"""Load libnka_b200.so (ctypes).  There is no fallback: if the CUDA library is
missing the import of anything that computes fails loudly."""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

MAX_MVEC = 32


class StateView(C.Structure):
    """include/nka_b200.h: nka_state_view"""
    _fields_ = [
        ("mvec", C.c_int), ("subspace", C.c_int), ("pending", C.c_int), ("first", C.c_int),
        ("last", C.c_int), ("free_slot", C.c_int),
        ("next", C.c_int * (MAX_MVEC + 1)), ("prev", C.c_int * (MAX_MVEC + 1)),
        ("chained", C.c_int * (MAX_MVEC + 1)),
        ("ndrop_last", C.c_int), ("evicted_last", C.c_int), ("relaxed_last", C.c_int), ("error", C.c_int),
        ("vtol", C.c_double), ("min_margin", C.c_double), ("s_last", C.c_double),
        ("c", C.c_double * (MAX_MVEC + 1)), ("s", C.c_double * (MAX_MVEC + 1)),
        ("h", C.c_double * ((MAX_MVEC + 1) * (MAX_MVEC + 1))),
        ("ncalls", C.c_ulonglong),
    ]


class StopTest(C.Structure):
    """include/nka_b200.h: nka_stop_test"""
    _fields_ = [
        ("atol", C.c_double), ("rtol", C.c_double), ("dtol", C.c_double), ("maxit", C.c_int),
        ("atol_dev", C.c_void_p), ("rtol_dev", C.c_void_p), ("maxit_dev", C.c_void_p),
        ("scale_dev", C.c_void_p), ("ldscale", C.c_size_t),
    ]


# every symbol include/*.h declares: name -> (restype, argtypes)
_dp = C.POINTER(C.c_double)
SYMBOLS = {
    # include/nonlinear_krylov_accelerator.h (the reference's nine)
    "nka_init": (C.c_void_p, [C.c_int, C.c_int, C.c_double, C.c_void_p]),
    "nka_delete": (None, [C.c_void_p]),
    "nka_accel_update": (None, [C.c_void_p, C.c_void_p]),
    "nka_restart": (None, [C.c_void_p]),
    "nka_relax": (None, [C.c_void_p]),
    "nka_num_vec": (C.c_int, [C.c_void_p]),
    "nka_max_vec": (C.c_int, [C.c_void_p]),
    "nka_vec_len": (C.c_int, [C.c_void_p]),
    "nka_vec_tol": (C.c_double, [C.c_void_p]),
    # include/nka_b200.h
    "nka_init_ex": (C.c_void_p, [C.c_size_t, C.c_int, C.c_double, C.c_int, C.c_void_p]),
    "nka_set_vec_tol": (None, [C.c_void_p, C.c_double]),
    "nka_set_dot_prod": (None, [C.c_void_p, C.c_void_p]),
    "nka_set_dot_prod_ctx": (None, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "nka_defined": (C.c_int, [C.c_void_p]),
    "nka_vec_len64": (C.c_size_t, [C.c_void_p]),
    "nka_accel_update_dev": (None, [C.c_void_p, C.c_void_p]),
    "nka_accel_update_host": (None, [C.c_void_p, C.c_void_p]),
    "nka_set_stream": (None, [C.c_void_p, C.c_void_p]),
    "nka_get_stream": (C.c_void_p, [C.c_void_p]),
    "nka_synchronize": (None, [C.c_void_p]),
    "nka_stream_capturing": (C.c_int, [C.c_void_p]),
    "nka_comm_unique_id": (C.c_int, [C.c_void_p]),
    "nka_comm_init": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "nka_comm_adopt": (None, [C.c_void_p, C.c_void_p, C.c_int, C.c_int]),
    "nka_comm_mode": (C.c_int, [C.c_void_p]),
    "nka_vec_create": (C.c_void_p, [C.c_size_t, C.c_int, C.c_void_p]),
    "nka_vec_clone": (C.c_void_p, [C.c_void_p]),
    "nka_vec_destroy": (None, [C.c_void_p]),
    "nka_vec_size": (C.c_size_t, [C.c_void_p]),
    "nka_vec_data": (C.c_void_p, [C.c_void_p]),
    "nka_vec_set_host": (None, [C.c_void_p, C.c_void_p]),
    "nka_vec_get_host": (None, [C.c_void_p, C.c_void_p]),
    "nka_vec_copy": (None, [C.c_void_p, C.c_void_p]),
    "nka_vec_setval": (None, [C.c_void_p, C.c_double]),
    "nka_vec_scale": (None, [C.c_void_p, C.c_double]),
    "nka_vec_update1": (None, [C.c_void_p, C.c_double, C.c_void_p]),
    "nka_vec_update2": (None, [C.c_void_p, C.c_double, C.c_void_p, C.c_double]),
    "nka_vec_update3": (None, [C.c_void_p, C.c_double, C.c_void_p, C.c_double, C.c_void_p]),
    "nka_vec_update4": (None, [C.c_void_p, C.c_double, C.c_void_p, C.c_double, C.c_void_p, C.c_double]),
    "nka_vec_dot": (C.c_double, [C.c_void_p, C.c_void_p]),
    "nka_vec_norm2": (C.c_double, [C.c_void_p]),
    "nka_vec_comm_init": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "nka_init_like": (C.c_void_p, [C.c_void_p, C.c_int, C.c_double]),
    "nka_accel_update_vec": (None, [C.c_void_p, C.c_void_p]),
    "nka_get_state": (None, [C.c_void_p, C.POINTER(StateView)]),
    "nka_launch_count": (C.c_ulonglong, [C.c_void_p]),
    "nka_timing_enable": (None, [C.c_void_p, C.c_int]),
    "nka_timing_reset": (None, [C.c_void_p]),
    "nka_timing_read": (None, [C.c_void_p, _dp, C.POINTER(C.c_ulonglong)]),
    "nka_launch_geometry": (None, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "nka_b200_version": (C.c_char_p, []),
    # include/nka_b200.h: batched accelerators
    "nka_batch_init": (C.c_void_p, [C.c_int, C.c_size_t, C.c_int, C.c_double, C.c_int, C.c_void_p]),
    "nka_batch_delete": (None, [C.c_void_p]),
    "nka_batch_accel_update": (None, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "nka_batch_relax": (None, [C.c_void_p, C.c_void_p]),
    "nka_batch_restart": (None, [C.c_void_p, C.c_void_p]),
    "nka_batch_set_vec_tol": (None, [C.c_void_p, C.c_double]),
    "nka_batch_num_vec": (None, [C.c_void_p, C.POINTER(C.c_int)]),
    "nka_batch_defined": (C.c_int, [C.c_void_p]),
    "nka_batch_get_state": (None, [C.c_void_p, C.c_int, C.POINTER(StateView)]),
    "nka_batch_set_stream": (None, [C.c_void_p, C.c_void_p]),
    "nka_batch_synchronize": (None, [C.c_void_p]),
    "nka_batch_stream_capturing": (C.c_int, [C.c_void_p]),
    "nka_batch_launch_count": (C.c_ulonglong, [C.c_void_p]),
    # include/nka_b200.h: device-side fixed-point loops
    "nka_batch_loop_create": (C.c_void_p, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t,
                                           C.c_double, C.c_double, C.c_int]),
    "nka_batch_loop_launch": (None, [C.c_void_p]),
    "nka_batch_loop_results": (None, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), _dp]),
    "nka_batch_loop_history": (None, [C.c_void_p, _dp]),
    "nka_batch_loop_destroy": (None, [C.c_void_p]),
    # include/nka_b200.h: device-side work queues
    "nka_batch_queue_create": (C.c_void_p, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t,
                                            C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_size_t,
                                            C.c_double, C.c_double, C.c_int]),
    "nka_batch_queue_launch": (None, [C.c_void_p]),
    "nka_batch_queue_results": (None, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), _dp]),
    "nka_batch_queue_destroy": (None, [C.c_void_p]),
    # include/nka_b200.h: per-problem stopping tests
    "nka_batch_loop_create_stop": (C.c_void_p, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t,
                                                C.POINTER(StopTest)]),
    "nka_batch_queue_create_stop": (C.c_void_p, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t,
                                                 C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_size_t,
                                                 C.POINTER(StopTest)]),
    # include/nka_b200.h: residual-growth restarts
    "nka_batch_loop_create_restart": (C.c_void_p, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t,
                                                   C.POINTER(StopTest), C.c_double]),
    "nka_batch_queue_create_restart": (C.c_void_p, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t,
                                                    C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_size_t,
                                                    C.POINTER(StopTest), C.c_double]),
    "nka_batch_loop_restarts": (None, [C.c_void_p, C.POINTER(C.c_int)]),
    "nka_batch_queue_restarts": (None, [C.c_void_p, C.POINTER(C.c_int)]),
    # include/nka_b200.h: interleaved batched accelerators
    "nka_ibatch_init": (C.c_void_p, [C.c_int, C.c_size_t, C.c_int, C.c_double, C.c_int, C.c_void_p]),
    "nka_ibatch_delete": (None, [C.c_void_p]),
    "nka_ibatch_accel_update": (None, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "nka_ibatch_relax": (None, [C.c_void_p, C.c_void_p]),
    "nka_ibatch_restart": (None, [C.c_void_p, C.c_void_p]),
    "nka_ibatch_set_vec_tol": (None, [C.c_void_p, C.c_double]),
    "nka_ibatch_num_vec": (None, [C.c_void_p, C.POINTER(C.c_int)]),
    "nka_ibatch_defined": (C.c_int, [C.c_void_p]),
    "nka_ibatch_get_state": (None, [C.c_void_p, C.c_int, C.POINTER(StateView)]),
    "nka_ibatch_set_stream": (None, [C.c_void_p, C.c_void_p]),
    "nka_ibatch_synchronize": (None, [C.c_void_p]),
    "nka_ibatch_stream_capturing": (C.c_int, [C.c_void_p]),
    "nka_ibatch_launch_count": (C.c_ulonglong, [C.c_void_p]),
    # include/nka_example.h
    "nka_system_init": (C.c_void_p, [C.c_int, C.c_int, C.c_double, C.c_int, C.c_int, C.c_void_p]),
    "nka_system_init_slab": (C.c_void_p, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int, C.c_void_p]),
    "nka_system_comm_init": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "nka_comm_share_system": (None, [C.c_void_p, C.c_void_p]),
    "nka_system_delete": (None, [C.c_void_p]),
    "nka_system_size": (C.c_size_t, [C.c_void_p]),
    "nka_system_stream": (C.c_void_p, [C.c_void_p]),
    "nka_system_field": (C.c_void_p, [C.c_void_p, C.c_int]),
    "nka_system_index": (C.c_size_t, [C.c_void_p, C.c_int, C.c_int]),
    "nka_system_set_field": (None, [C.c_void_p, C.c_int, C.c_void_p]),
    "nka_system_get_field": (None, [C.c_void_p, C.c_int, C.c_void_p]),
    "nka_system_residual": (C.c_double, [C.c_void_p, C.c_int]),
    "nka_system_pc_ssor": (C.c_int, [C.c_void_p, C.c_int, C.c_double]),
    "nka_example_solve": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.c_int, C.c_double,
                                    _dp, C.POINTER(C.c_int)]),
    "nka_system_ssor_trace": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "nka_example_division_check": (C.c_ulonglong, [C.c_ulonglong, C.c_ulonglong, C.c_int]),
    "nka_system_timing_enable": (None, [C.c_void_p, C.c_int]),
    "nka_system_timing_read": (None, [C.c_void_p, _dp, C.POINTER(C.c_ulonglong)]),
    "nka_system_launch_count": (C.c_ulonglong, [C.c_void_p]),
}

_lib = None


def lib_path() -> str:
    return _build.LIB_PATH


def load() -> C.CDLL:
    """Return the loaded library; build it first if the tree has none."""
    global _lib
    if _lib is None:
        path = os.environ.get("NKA_B200_LIB")      # tuning builds only (tools/tune.py)
        if not path:
            path = _build.LIB_PATH
            if not os.path.exists(path):
                path = _build.build_library()
        lib = C.CDLL(path)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(lib, name)      # AttributeError if the ABI drifted: loud by design
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib
