"""ctypes binding of libcvmx.so (include/cvmx.h).  No fallback: a missing library is an error."""

from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libcvmx.so")

OK, ERR_INVALID, ERR_CUDA, ERR_NEG_WEIGHT, ERR_INDEX, ERR_NO_Y, ERR_NOMEM = range(7)
F32, F64 = 0, 1
HOST, DEVICE = 0, 1
WANT_XTX, WANT_XTY, WANT_STATS = 1, 2, 4
FOLD_NO_NONZERO_W, FOLD_NNZ_LE_DDOF = 1, 2

# cvmx_ridge_plan (include/cvmx.h): kernels (CVMX_RK_*) and plan entries (CVMX_RIDGE_*)
(RK_LOAD, RK_POTRF, RK_TRSM, RK_SYRK, RK_BSOLVE_DIAG, RK_BSOLVE_UPDATE, RK_PRESS, RK_PRESS_ACCUM, RK_FINISH,
 RK_COEFS) = range(10)
RK_COUNT = 10
RIDGE_KERNELS = ("k_ridge_load", "k_ridge_potrf_diag", "k_ridge_trsm", "k_ridge_syrk", "k_ridge_bsolve_diag",
                 "k_ridge_bsolve_update", "k_ridge_press", "k_ridge_press_accum", "k_ridge_finish", "k_ridge_coefs")
(RIDGE_FEASIBLE, RIDGE_FOLDS_PER_WINDOW, RIDGE_PENALTIES_PER_PASS, RIDGE_SCRATCH_BYTES, RIDGE_END_A, RIDGE_END_STATE,
 RIDGE_END_ACC, RIDGE_END_ACC_W, RIDGE_END_PRESS, RIDGE_END_INFO, RIDGE_END_B, RIDGE_END_SUM_W, RIDGE_END_STATUS,
 RIDGE_WINDOW_BYTES, RIDGE_PART_BYTES, RIDGE_CHUNKS_PER_LAUNCH) = range(16)
RIDGE_GRID = 16
RIDGE_SMEM = RIDGE_GRID + 2 * RK_COUNT
RIDGE_PLAN_LEN = RIDGE_SMEM + RK_COUNT

_vp, _i64, _i32, _u32, _dbl = C.c_void_p, C.c_int64, C.c_int32, C.c_uint32, C.c_double

# name -> (restype, argtypes); mirrors include/cvmx.h one to one (tests check the export list)
SIGNATURES = {
    "cvmx_version": (_i32, []),
    "cvmx_last_error": (C.c_char_p, [_vp]),
    "cvmx_create": (_i32, [_i32, _i32, _u32, _i64, _dbl, C.POINTER(_vp)]),
    "cvmx_destroy": (_i32, [_vp]),
    "cvmx_set_stream": (_i32, [_vp, _vp]),
    "cvmx_sync": (_i32, [_vp]),
    "cvmx_fit": (_i32, [_vp, _vp, _i64, _i64, _i64, _vp, _i64, _i64, _vp, _i32, _i64, _i64]),
    "cvmx_fit_begin": (_i32, [_vp, _i64, _i64, _i64, _i32, _i64]),
    "cvmx_fit_rows": (_i32, [_vp, _i64, _i64, _vp, _i64, _vp, _i64, _vp, _i32, _i32]),
    "cvmx_fit_end": (_i32, [_vp, _i32, _i32]),
    "cvmx_data_ptr": (_i32, [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_i64)]),
    "cvmx_moments_ptr": (_i32, [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_i64)]),
    "cvmx_totals_ptr": (_i32, [_vp, C.POINTER(_vp), C.POINTER(_i64), C.POINTER(_i64)]),
    "cvmx_commit_totals": (_i32, [_vp]),
    "cvmx_get_totals": (_i32, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, C.POINTER(_dbl), C.POINTER(_i64)]),
    "cvmx_set_folds": (_i32, [_vp, _vp, _vp, _i64, _i32]),
    "cvmx_fit_folds": (_i32, [_vp, _vp, _i64, _i64, _i64, _vp, _i64, _i64, _vp, _i32, _vp, _vp, _i64, _i32]),
    "cvmx_folds_are_cached": (_i32, [_vp]),
    "cvmx_training_batch": (_i32, [_vp, _i64, _i64, _u32, _vp, _vp, _vp, _vp, _vp, _i32]),
    "cvmx_training_indices": (_i32, [_vp, _vp, _i64, _i32, _u32, _vp, _vp, _vp, _vp, _vp, _i32]),
    "cvmx_sharded_stats": (_i32, [_vp, _i64, _i64, _i32, _i32, C.POINTER(_vp), C.POINTER(_i64)]),
    "cvmx_sharded_stats_wait": (_i32, [_vp]),
    "cvmx_sharded_gram_count": (_i64, [_vp, _i64, _i64, _u32]),
    "cvmx_sharded_gram": (_i32, [_vp, _i64, _i64, _u32, _i32, _i32, _vp]),
    "cvmx_sharded_finish": (_i32, [_vp, _i64, _i64, _i64, _u32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "cvmx_sharded_finish_peers": (_i32, [_vp, _i64, _i64, _i64, _i64, _u32, _vp, _i32, _i64, _vp, _vp, _vp, _vp, _vp]),
    "cvmx_fit_end_slab": (_i32, [_vp, _vp, _vp, _vp, _i64, _i64]),
    "cvmx_slab_begin": (_i32, [_vp, _vp, _i64, _i64]),
    "cvmx_slab_scan_local": (_i32, [_vp, _i64, _i64, _vp, _i64, _i64, _vp, C.POINTER(_i32)]),
    "cvmx_slab_scan_prepare": (_i32, [_vp, _i64, _i64, _vp]),
    "cvmx_set_weight_folds": (_i32, [_vp, _vp, _vp, _i64]),
    "cvmx_slab_fold_sums": (_i32, [_vp, _i64, _i64, _vp]),
    "cvmx_slab_finalize_stats": (_i32, [_vp, _i64, _i64, _vp]),
    "cvmx_validation_rows": (_i32, [_vp, _i64, _vp, _u32, _vp, _vp, _i32]),
    "cvmx_pls_cv": (_i32, [_vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _i32]),
    "cvmx_ridge_cv": (_i32, [_vp, _i64, _i64, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _i32]),
    "cvmx_pls_cv_predict": (_i32, [_vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _i32]),
    "cvmx_ridge_cv_predict": (_i32, [_vp, _i64, _i64, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _i32]),
    "cvmx_ridge_plan": (_i32, [_i64, _i64, _i64, _i64, _i32, _i32, _i32, _vp]),
    "cvmx_profile_enable": (_i32, [_vp, _i32]),
    "cvmx_profile_read": (_i32, [_vp, C.POINTER(_dbl), C.POINTER(_i64)]),
    "cvmx_partition_labels": (_i64, [_vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp]),
    "cvmx_launch_count": (_i64, [_vp]),
    "cvmx_ld": (_i64, [_vp]),
    "cvmx_set_scan_mode": (_i32, [_vp, _i32]),
    "cvmx_scan_launch_count": (_i64, [_vp]),
    "cvmx_set_loo_mode": (_i32, [_vp, _i32]),
}

_lib = None


def load():
    """Loads libcvmx.so.  Raises ImportError if it has not been built (python -m cvmatrix_b200.build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing. cvmatrix_b200 has no CPU fallback: build the CUDA library with "
                "`python -m cvmatrix_b200.build` (needs nvcc; targets sm_100a)."
            )
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


class CvmxError(RuntimeError):
    pass


def check(rc: int, handle=None):
    """Maps a non-zero cvmx_status to the Python exception the reference would raise."""
    if rc == OK:
        return
    msg = load().cvmx_last_error(handle)
    msg = msg.decode() if msg else f"cvmx error {rc}"
    if rc == ERR_NEG_WEIGHT:
        raise ValueError("Weights must be non-negative.")
    if rc == ERR_INDEX:
        raise IndexError(msg)
    if rc == ERR_NO_Y:
        raise ValueError("Response variables `Y` are not provided.")
    if rc == ERR_NOMEM:
        raise MemoryError(msg)
    if rc == ERR_INVALID:
        raise ValueError(msg)
    raise CvmxError(msg)
