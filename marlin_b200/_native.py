"""ctypes binding of libmarlin_b200.so (include/marlin_b200.h).

The shared library is the product; this module only declares its C ABI for Python callers
(the host mirror in marlin_b200.matrix, the tests and bench.py).  It never computes anything itself
and has no fallback: if the library cannot be loaded, or a call fails, it raises.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

MB_OK = 0
MB_ERR_INVALID_ARG = -1
MB_ERR_DIM_MISMATCH = -2
MB_ERR_UNSUPPORTED = -3
MB_ERR_CUDA = -4
MB_ERR_OOM = -5
MB_ERR_EMPTY = -6
MB_ERR_TIMEOUT = -7

MB_F64, MB_BF16, MB_F32 = 0, 1, 2

_LIB_PATH = Path(__file__).resolve().parent / "lib" / "libmarlin_b200.so"

c_ctx = C.c_void_p
c_blk = C.c_void_p
c_sp = C.c_void_p          # mb_spblock*
c_i32 = C.c_int32
c_i64 = C.c_int64
c_f64 = C.c_double
c_dp = C.POINTER(C.c_double)

# name -> (restype, argtypes); mirrors include/marlin_b200.h one to one
SIGNATURES = {
    "mb_init": (c_i32, [c_i32, C.POINTER(c_ctx)]),
    "mb_shutdown": (c_i32, [c_ctx]),
    "mb_last_error": (C.c_char_p, []),
    "mb_version": (C.c_char_p, []),
    "mb_set_stream": (c_i32, [c_ctx, C.c_void_p]),
    "mb_reset_stream": (c_i32, [c_ctx]),
    "mb_synchronize": (c_i32, [c_ctx]),
    "mb_launch_count": (c_i64, [c_ctx]),
    "mb_timer_start": (c_i32, [c_ctx]),
    "mb_timer_stop": (c_i32, [c_ctx, C.POINTER(C.c_float)]),
    "mb_block_alloc": (c_i32, [c_ctx, c_i32, c_i32, c_i32, C.POINTER(c_blk)]),
    "mb_block_wrap": (c_i32, [c_ctx, C.c_void_p, c_i64, c_i32, c_i32, c_i32, c_i32, c_i32, C.POINTER(c_blk)]),
    "mb_block_upload": (c_i32, [c_ctx, C.c_void_p, c_i64, c_i32, c_i32, c_i32, c_i32, c_i32, C.POINTER(c_blk)]),
    "mb_block_download": (c_i32, [c_ctx, c_blk, C.c_void_p, c_i32]),
    "mb_block_free": (c_i32, [c_ctx, c_blk]),
    "mb_block_info": (c_i32, [c_blk, C.POINTER(c_i32), C.POINTER(c_i32), C.POINTER(c_i32), C.POINTER(c_i32),
                              C.POINTER(c_i32), C.POINTER(C.c_void_p)]),
    "mb_block_set_ready_event": (c_i32, [c_blk, C.c_void_p]),
    "mb_block_view_t": (c_i32, [c_ctx, c_blk, C.POINTER(c_blk)]),
    "mb_block_slice": (c_i32, [c_ctx, c_blk, c_i32, c_i32, c_i32, c_i32, C.POINTER(c_blk)]),
    "mb_block_gemm": (c_i32, [c_ctx, c_blk, c_blk, c_blk, c_i32]),
    "mb_set_fp64_mode": (c_i32, [c_ctx, c_i32, c_i32]),
    "mb_dgemm_device": (c_i32, [c_ctx, C.c_char, C.c_char, c_i32, c_i32, c_i32, c_f64, C.c_void_p, c_i32,
                                C.c_void_p, c_i32, c_f64, C.c_void_p, c_i32]),
    "mb_dgemm_device_generic": (c_i32, [c_ctx, C.c_char, C.c_char, c_i32, c_i32, c_i32, c_f64, C.c_void_p, c_i32,
                                        C.c_void_p, c_i32, c_f64, C.c_void_p, c_i32]),
    "mb_dgemm_host": (c_i32, [c_ctx, C.c_char, C.c_char, c_i32, c_i32, c_i32, c_f64, C.c_void_p, c_i64, c_i32,
                              C.c_void_p, c_i64, c_i32, c_f64, C.c_void_p, c_i64, c_i32]),
    "mb_block_add": (c_i32, [c_ctx, c_blk, c_blk, c_blk]),
    "mb_block_sub": (c_i32, [c_ctx, c_blk, c_blk, c_blk]),
    "mb_block_hadamard": (c_i32, [c_ctx, c_blk, c_blk, c_blk]),
    "mb_block_axpb": (c_i32, [c_ctx, c_blk, c_f64, c_f64, c_blk]),
    "mb_block_fill": (c_i32, [c_ctx, c_blk, c_f64]),
    "mb_block_div": (c_i32, [c_ctx, c_blk, c_f64, c_i32, c_blk]),
    "mb_block_transpose": (c_i32, [c_ctx, c_blk, c_blk]),
    "mb_block_copy": (c_i32, [c_ctx, c_blk, c_blk]),
    "mb_block_sum": (c_i32, [c_ctx, c_blk, c_dp]),
    "mb_block_gemv": (c_i32, [c_ctx, c_blk, c_blk, c_blk, c_i32]),
    "mb_block_dot": (c_i32, [c_ctx, c_blk, c_blk, c_dp]),
    "mb_block_ger": (c_i32, [c_ctx, c_blk, c_blk, c_blk]),
    "mb_block_lu": (c_i32, [c_ctx, c_blk, C.POINTER(c_i32)]),
    "mb_block_cholesky": (c_i32, [c_ctx, c_blk]),
    "mb_block_inverse": (c_i32, [c_ctx, c_blk, c_blk]),
    "mb_block_trsm": (c_i32, [c_ctx, c_blk, c_i32, c_i32, c_blk]),
    "mb_fill_uniform": (c_i32, [c_ctx, c_blk, c_i64, c_i64, c_f64, c_f64, c_i32]),
    "mb_hash_seed": (c_i64, [c_i64]),
    "mb_partition_seeds": (c_i32, [c_i64, c_i32, C.POINTER(c_i64)]),
    "mb_choose_split": (c_i32, [c_i64, c_i64, c_i64, c_i32, C.POINTER(c_i32)]),
    "mb_choose_strategy": (c_i32, [c_i64, c_i64, c_i64, c_i32, c_i32, c_i32, C.POINTER(c_i32), C.POINTER(c_i32)]),
    "mb_mult_partition": (c_i32, [c_i32, c_i32, c_i32, c_i32, c_i32, c_i32]),
    "mb_elem_partition": (c_i32, [c_i32, c_i32, c_i32]),
    "mb_block_len": (c_i32, [c_i64, c_i32, C.POINTER(c_i32), C.POINTER(c_i32)]),
    "mb_matmul_blocked_host": (c_i32, [c_ctx, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), c_i32, c_i32, c_i32,
                                       C.POINTER(c_i32), C.POINTER(c_i32), C.POINTER(c_i32), C.POINTER(C.c_void_p)]),
    "mb_matmul_rowsharded": (c_i32, [c_ctx, c_blk, c_blk, c_blk]),
    "mb_matmul_rowsharded_host": (c_i32, [c_ctx, C.c_void_p, c_i64, c_i32, C.c_void_p, c_i32, C.c_void_p]),
    "mb_ipc_export": (c_i32, [c_ctx, C.c_void_p, C.c_char_p, C.POINTER(c_i64), C.POINTER(c_i64)]),
    "mb_ipc_open": (c_i32, [c_ctx, C.c_char_p, C.POINTER(C.c_void_p)]),
    "mb_ipc_close_all": (c_i32, [c_ctx]),
    "mb_flags_alloc": (c_i32, [c_ctx, c_i32, C.POINTER(C.c_void_p)]),
    "mb_flags_free": (c_i32, [c_ctx, C.c_void_p]),
    "mb_flag_signal": (c_i32, [c_ctx, C.c_void_p, c_i64]),
    "mb_flag_wait": (c_i32, [c_ctx, C.c_void_p, c_i64]),
    "mb_memcpy_async": (c_i32, [c_ctx, C.c_void_p, C.c_void_p, c_i64]),
    "mb_matmul_blocked_subset": (c_i32, [c_ctx, C.POINTER(c_blk), C.POINTER(c_blk), c_i32, c_i32, c_i32, C.POINTER(c_blk),
                                         C.POINTER(c_i32), c_i32]),
    "mb_matmul_blocked": (c_i32, [c_ctx, C.POINTER(c_blk), C.POINTER(c_blk), c_i32, c_i32, c_i32, C.POINTER(c_blk)]),
    "mb_comm_init": (c_i32, [c_ctx, c_i32, c_i32, C.c_char_p, C.POINTER(C.c_void_p)]),
    "mb_comm_destroy": (c_i32, [C.c_void_p]),
    "mb_comm_rank": (c_i32, [C.c_void_p]),
    "mb_comm_world": (c_i32, [C.c_void_p]),
    "mb_comm_barrier": (c_i32, [C.c_void_p]),
    "mb_comm_check": (c_i32, [C.c_void_p]),
    "mb_comm_abort": (c_i32, [C.c_void_p]),
    "mb_dist_plan": (c_i32, [c_i32, c_i32, c_i32, c_i32, C.POINTER(c_i32), C.POINTER(c_i32)]),
    "mb_dist_host_homes": (c_i32, [c_i32, c_i32, c_i32, c_i32, C.POINTER(c_i32), C.POINTER(c_i32)]),
    "mb_matmul_blocked_dist_host": (c_i32, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(c_i32), C.POINTER(C.c_void_p), C.POINTER(c_i32),
                                            c_i32, c_i32, c_i32, C.POINTER(c_i32), C.POINTER(c_i32), C.POINTER(c_i32), C.POINTER(C.c_void_p)]),
    "mb_host_alloc_shared": (c_i32, [C.c_char_p, c_i64, C.POINTER(C.c_void_p)]),
    "mb_host_free_shared": (c_i32, [C.c_char_p, C.c_void_p, c_i64, c_i32]),
    "mb_matmul_blocked_dist": (c_i32, [C.c_void_p, C.POINTER(c_blk), C.POINTER(c_i32), C.POINTER(c_blk), C.POINTER(c_i32), c_i32, c_i32,
                                       c_i32, C.POINTER(c_i32), C.POINTER(c_i32), C.POINTER(c_i32), c_i32, C.POINTER(c_blk)]),
    "mb_csc_check": (c_i32, [c_i32, c_i32, C.POINTER(c_i32), C.POINTER(c_i32)]),
    "mb_spblock_upload": (c_i32, [c_ctx, c_i32, c_i32, C.POINTER(c_i32), C.POINTER(c_i32), c_dp, C.POINTER(c_sp)]),
    "mb_spblock_download": (c_i32, [c_ctx, c_sp, C.POINTER(c_i32), C.POINTER(c_i32), c_dp]),
    "mb_spblock_info": (c_i32, [c_sp, C.POINTER(c_i32), C.POINTER(c_i32), C.POINTER(c_i64)]),
    "mb_spblock_free": (c_i32, [c_ctx, c_sp]),
    "mb_spblock_copy": (c_i32, [c_ctx, c_sp, C.POINTER(c_sp)]),
    "mb_spblock_values": (c_i32, [c_ctx, c_sp, C.POINTER(c_blk)]),
    "mb_spblock_to_dense": (c_i32, [c_ctx, c_sp, c_blk]),
    "mb_sparse_rand_count": (c_i32, [c_i32, c_i32, c_f64, C.POINTER(c_i32)]),
    "mb_spblock_rand": (c_i32, [c_ctx, c_i32, c_i32, c_f64, c_i64, C.POINTER(c_sp)]),
    "mb_spmm_dense_sparse": (c_i32, [c_ctx, c_blk, c_sp, c_blk, c_i32]),
    "mb_spmm_sparse_dense": (c_i32, [c_ctx, c_sp, c_blk, c_blk, c_i32]),
    "mb_spgemm_to_dense": (c_i32, [c_ctx, c_sp, c_sp, c_blk, c_i32]),
}


class MarlinError(RuntimeError):
    """Raised for MB_ERR_CUDA / MB_ERR_OOM / MB_ERR_EMPTY (RuntimeException on the JVM side)."""

    def __init__(self, code: int, message: str):
        super().__init__(f"[marlin_b200 {code}] {message}")
        self.code = code


class MarlinArgumentError(ValueError):
    """Raised for INVALID_ARG / DIM_MISMATCH / UNSUPPORTED (Scala `require` -> IllegalArgumentException)."""

    def __init__(self, code: int, message: str):
        super().__init__(message)
        self.code = code


_lib = None


def lib_path() -> Path:
    return _LIB_PATH


def load(build_if_missing: bool = True) -> C.CDLL:
    """Load the shared library (building it in-tree with nvcc if it is missing or stale)."""
    global _lib
    if _lib is not None:
        return _lib
    if build_if_missing and os.environ.get("MARLIN_B200_NO_BUILD") != "1":
        from . import build as _build
        if _build.needs_build():
            _build.build_library()
    if not _LIB_PATH.exists():
        raise MarlinError(MB_ERR_CUDA, f"{_LIB_PATH} is missing: run `python -m marlin_b200.build` (needs nvcc). "
                          "marlin_b200 has no CPU fallback.")
    lib = C.CDLL(str(_LIB_PATH))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)      # AttributeError here means header and library are out of sync
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status: int) -> None:
    if status == MB_OK:
        return
    msg = load().mb_last_error().decode("utf-8", "replace")
    if status in (MB_ERR_INVALID_ARG, MB_ERR_DIM_MISMATCH, MB_ERR_UNSUPPORTED):
        raise MarlinArgumentError(status, msg)
    raise MarlinError(status, msg)
