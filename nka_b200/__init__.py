"""nka_b200 -- B200-native Nonlinear Krylov Accelerator (drop-in for nncarlson/nka's accel_update path).

Only what the hot path needs: csrc/ (sm_100a CUDA kernels + the C-ABI of
libnka_b200.so), fortran/ (the reference's Fortran modules as thin bind(C)
layers), and this Python mirror of the reference interface for tests and
benchmarks.
"""
from .batch import BatchNKA
from .ibatch import InterleavedBatchNKA
from .nka import (NKA, NKAError, comm_unique_id, nka_accel_update, nka_delete, nka_init, nka_max_vec,
                  nka_num_vec, nka_relax, nka_restart, nka_vec_len, nka_vec_tol)

__all__ = ["NKA", "BatchNKA", "InterleavedBatchNKA", "NKAError", "comm_unique_id", "nka_init", "nka_delete",
           "nka_accel_update", "nka_restart", "nka_relax", "nka_num_vec", "nka_max_vec", "nka_vec_len", "nka_vec_tol"]
