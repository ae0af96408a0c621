"""ctypes binding of the C ABI in include/poismf_b200.h (libpoismf_b200.so).

Fails loudly: importing the symbols raises if the in-tree library has not been built;
every compute call raises if no CUDA device is usable.  There is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libpoismf_b200.so")

PMF_F32, PMF_F64 = 0, 1
METHODS = {"tncg": 1, "cg": 2, "pg": 3}
SIDE_CSR, SIDE_CSC = 0, 1
FLAG_STRICT, FLAG_NO_CACHED, FLAG_NO_LOCKSTEP = 1, 2, 4

# every symbol include/poismf_b200.h declares (tests check that all are exported)
SYMBOLS = [
    "pmf_b200_device_count", "pmf_b200_last_error", "pmf_b200_kernel_launches",
    "pmf_b200_create", "pmf_b200_destroy", "pmf_b200_ldf", "pmf_b200_set_matrix",
    "pmf_b200_set_factors", "pmf_b200_get_factors", "pmf_b200_bind_factors", "pmf_b200_set_factor_rows", "pmf_b200_factor_ptr",
    "pmf_b200_set_stream", "pmf_b200_sweeps", "pmf_b200_half_sweep", "pmf_b200_sync",
    "pmf_b200_set_profiling", "pmf_b200_get_profile", "pmf_b200_ipc_export", "pmf_b200_ipc_import",
    "pmf_b200_run_poismf", "pmf_b200_factors_multiple", "pmf_b200_factors_single", "pmf_b200_predict_multiple", "pmf_b200_topN", "pmf_b200_topN_batch", "pmf_b200_topN_fitted", "pmf_b200_topN_stats",
    "pmf_b200_topN_batch_include", "pmf_b200_topN_fitted_include",
    "pmf_b200_topN_new_batch", "pmf_b200_topN_new_fitted", "pmf_b200_fit_stats",
    "pmf_b200_release_cache", "pmf_b200_fit_coo", "pmf_b200_coo_to_csr_csc",
    "pmf_b200_predict_fitted", "pmf_b200_set_coo",
]


class Params(C.Structure):
    _fields_ = [("l2_reg", C.c_double), ("l1_reg", C.c_double), ("w_mult", C.c_double),
                ("step_size", C.c_double), ("method", C.c_int), ("limit_step", C.c_int),
                ("numiter", C.c_size_t), ("maxupd", C.c_size_t), ("early_stop", C.c_int),
                ("reuse_prev", C.c_int), ("flags", C.c_int)]


class BinProfile(C.Structure):
    _fields_ = [("side", C.c_int), ("block_team", C.c_int), ("cap", C.c_int), ("nrows", C.c_int),
                ("nnz", C.c_ulonglong), ("launches", C.c_ulonglong), ("ms", C.c_double)]


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: build it with `python -m poismf_b200.build` "
                          "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    vp, sz, i, d = C.c_void_p, C.c_size_t, C.c_int, C.c_double
    L.pmf_b200_device_count.restype = i
    L.pmf_b200_last_error.restype = C.c_char_p
    L.pmf_b200_kernel_launches.restype = C.c_uint64
    L.pmf_b200_create.restype = vp
    L.pmf_b200_create.argtypes = [i, sz, sz, sz, i]
    L.pmf_b200_destroy.argtypes = [vp]
    L.pmf_b200_destroy.restype = None
    L.pmf_b200_ldf.argtypes = [vp]
    L.pmf_b200_set_matrix.argtypes = [vp, i, vp, vp, vp, sz, i, sz, sz]
    L.pmf_b200_set_factors.argtypes = [vp, vp, vp]
    L.pmf_b200_get_factors.argtypes = [vp, vp, vp]
    L.pmf_b200_bind_factors.argtypes = [vp, vp, vp]
    L.pmf_b200_set_factor_rows.argtypes = [vp, C.c_int, vp, C.c_size_t, C.c_size_t]
    L.pmf_b200_set_factor_rows.restype = C.c_int
    L.pmf_b200_factor_ptr.argtypes = [vp, i]
    L.pmf_b200_factor_ptr.restype = vp
    L.pmf_b200_set_stream.argtypes = [vp, vp]
    L.pmf_b200_sweeps.argtypes = [vp, C.POINTER(Params)]
    L.pmf_b200_half_sweep.argtypes = [vp, i, C.POINTER(Params), d, d, C.POINTER(C.c_ulonglong)]
    L.pmf_b200_sync.argtypes = [vp]
    L.pmf_b200_ipc_export.argtypes = [vp, i, vp]
    L.pmf_b200_ipc_import.argtypes = [vp, i, vp, i, i]
    L.pmf_b200_set_profiling.argtypes = [vp, i]
    L.pmf_b200_get_profile.argtypes = [vp, C.POINTER(BinProfile), i]
    L.pmf_b200_run_poismf.argtypes = [i, i] + [vp] * 8 + [sz, sz, sz, d, d, d, d, i, i, sz, sz, i, i, i, i]
    L.pmf_b200_factors_multiple.argtypes = [i, i] + [vp] * 7 + [i, sz, sz, d, d, d, sz, sz, i, i, i, i]
    L.pmf_b200_factors_single.argtypes = [i, i, vp, sz, vp, i, vp, vp, sz, vp, vp, i, d, d, d, d, i]
    L.pmf_b200_predict_multiple.argtypes = [i, i, vp, vp, vp, vp, vp, sz, i, sz, sz]
    L.pmf_b200_topN.argtypes = [i, i, vp, vp, i, vp, sz, vp, sz, vp, vp, sz, sz]
    L.pmf_b200_topN_batch.argtypes = [i, i, vp, vp, i, vp, sz, sz, vp, vp, vp, vp, sz, sz]
    L.pmf_b200_topN_fitted.argtypes = [vp, i, vp, sz, vp, vp, vp, vp, sz]
    L.pmf_b200_topN_batch_include.argtypes = [i, i, vp, vp, i, vp, sz, sz, vp, vp, vp, vp, sz, sz]
    L.pmf_b200_topN_fitted_include.argtypes = [vp, i, vp, sz, vp, vp, vp, vp, sz]
    L.pmf_b200_topN_new_batch.argtypes = [i, i, vp, vp, vp, i, sz, vp, vp, vp, sz, C.POINTER(Params)] + [vp] * 6 + [sz, vp]
    L.pmf_b200_topN_new_fitted.argtypes = [vp, i, vp, vp, vp, vp, vp, sz, C.POINTER(Params)] + [vp] * 6 + [sz, vp]
    L.pmf_b200_fit_stats.argtypes = [vp, d, vp, vp]
    L.pmf_b200_topN_stats.argtypes = [C.POINTER(C.c_ulonglong), C.POINTER(C.c_ulonglong), i]
    L.pmf_b200_topN_stats.restype = None
    L.pmf_b200_fit_coo.argtypes = [i, i] + [vp] * 5 + [sz, sz, sz, sz, d, d, d, d, i, i, sz, sz, i, i, i]
    L.pmf_b200_coo_to_csr_csc.argtypes = [i, i, vp, vp, vp, sz, sz, sz] + [vp] * 6 + [C.POINTER(C.c_size_t)]
    L.pmf_b200_predict_fitted.argtypes = [vp, i, vp, vp, sz, vp]
    L.pmf_b200_set_coo.argtypes = [vp, vp, vp, vp, sz, i]
    L.pmf_b200_release_cache.argtypes = []
    L.pmf_b200_release_cache.restype = C.c_size_t
    _lib = L
    return L


def dtype_code(dtype):
    dtype = np.dtype(dtype)
    if dtype == np.float32:
        return PMF_F32
    if dtype == np.float64:
        return PMF_F64
    raise TypeError(f"poismf_b200 supports float32/float64, got {dtype}")


def index_bytes(arr):
    if arr.dtype == np.uint64 or arr.dtype == np.int64:
        return 8
    if arr.dtype == np.int32:
        return 4
    raise TypeError(f"index arrays must be uint64 (size_t) or int32, got {arr.dtype}")


def ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def last_error():
    return lib().pmf_b200_last_error().decode()


def require_gpu():
    if lib().pmf_b200_device_count() <= 0:
        raise RuntimeError("poismf_b200: no usable CUDA device (there is no CPU fallback)")


def topn_stats(reset=False):
    """(users scored on tensor cores, users redone exactly) for this thread's topN calls."""
    a, b = C.c_ulonglong(0), C.c_ulonglong(0)
    lib().pmf_b200_topN_stats(C.byref(a), C.byref(b), int(reset))
    return a.value, b.value


def make_params(method, l2_reg, l1_reg=0.0, w_mult=1.0, step_size=1e-7, limit_step=False, numiter=1,
                maxupd=1, early_stop=False, reuse_prev=False, flags=0):
    return Params(float(l2_reg), float(l1_reg), float(w_mult), float(step_size), METHODS[method],
                  int(bool(limit_step)), int(numiter), int(maxupd), int(bool(early_stop)),
                  int(bool(reuse_prev)), int(flags))
