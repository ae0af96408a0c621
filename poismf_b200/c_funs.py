"""Host-side mirror of the reference's Cython wrapper for the hot path.

Same function names, argument order and error behaviour as
/root/reference/poismf/poismf_c_wrapper.pxi (`_run_poismf` :57-107, `_predict_multiple`
:109-112, `_call_topN` :208-249), so that `poismf.PoisMF` can use this module in
place of `c_funs_double` / `c_funs_float`:  the value type is taken from the arrays.
Every call goes through the C ABI (include/poismf_b200.h) with HOST buffers.
"""
from __future__ import annotations

import ctypes

import numpy as np

from . import _lib


def _get_has_openmp():
    return True


def _run_poismf(Xr, Xr_indices, Xr_indptr, Xc, Xc_indices, Xc_indptr, A, B,
                method="tncg", limit_step=False, l2_reg=1e9, l1_reg=0.0, w_mult=1.0,
                step_size=1e-7, niter=10, maxupd=1, early_stop=True, reuse_prev=True,
                handle_interrupt=True, nthreads=1, flags=0):
    if Xr.shape[0] == 0:
        raise ValueError("'X' contains no non-zero entries.")
    INT_MAX = np.iinfo(ctypes.c_int).max
    if max(A.shape[0], A.shape[1], B.shape[0]) > INT_MAX:
        raise ValueError("Error: integer overflow. Dimensions cannot be larger than 2^31-1.")
    if A.dtype != B.dtype or A.dtype != Xr.dtype or A.dtype != Xc.dtype:
        raise TypeError("A, B, Xr, Xc must share one dtype")
    for a in (Xr, Xr_indices, Xr_indptr, Xc, Xc_indices, Xc_indptr, A, B):
        if not a.flags.c_contiguous:
            raise ValueError("arrays must be C-contiguous")
    _lib.require_gpu()
    L = _lib.lib()
    rc = L.pmf_b200_run_poismf(
        _lib.dtype_code(A.dtype), _lib.index_bytes(Xr_indptr),
        _lib.ptr(A), _lib.ptr(Xr), _lib.ptr(Xr_indptr), _lib.ptr(Xr_indices),
        _lib.ptr(B), _lib.ptr(Xc), _lib.ptr(Xc_indptr), _lib.ptr(Xc_indices),
        A.shape[0], B.shape[0], A.shape[1],
        float(l2_reg), float(l1_reg), float(w_mult), float(step_size),
        _lib.METHODS[method], int(bool(limit_step)), int(niter), int(maxupd),
        int(bool(early_stop)), int(bool(reuse_prev)), int(bool(handle_interrupt)), int(flags))
    if rc == 1:
        raise MemoryError("Could not allocate enough memory.")
    elif rc == 2 and not handle_interrupt:
        raise InterruptedError("Procedure was interrupted")
    return rc


def _predict_factors(counts, ix, B, Bsum, Amean, reuse_mean=True, maxupd=20, l2_reg=1e5, l1_new=0.0, l1_old=0.0,
                     w_mult=1.0, limit_step=False, flags=0):
    """poismf_c_wrapper.pxi:114-145 — factors of one new row (PoisMF.predict_factors / topN_new)."""
    _lib.require_gpu()
    if counts.dtype != B.dtype:
        raise TypeError("counts and B must share one dtype")
    out = np.empty(Amean.shape[0], dtype=B.dtype)
    rc = _lib.lib().pmf_b200_factors_single(
        _lib.dtype_code(B.dtype), _lib.index_bytes(ix), _lib.ptr(out), out.shape[0], _lib.ptr(Amean),
        int(bool(reuse_mean)), _lib.ptr(counts) if counts.shape[0] else None, _lib.ptr(ix) if ix.shape[0] else None,
        counts.shape[0], _lib.ptr(B), _lib.ptr(Bsum), int(maxupd), float(l2_reg), float(l1_new), float(l1_old),
        float(w_mult), int(flags))
    if rc:
        raise MemoryError("Could not allocate enough memory.")
    return out


def _predict_factors_multiple(B, Bsum, Amean, Xr_indptr, Xr_indices, Xr, l2_reg=1e9, w_mult=1.0, step_size=1e-7,
                              niter=10, maxupd=1, method="tncg", limit_step=False, reuse_mean=True, nthreads=1,
                              flags=0):
    """poismf_c_wrapper.pxi:147-206 — factors for new rows (PoisMF.transform / predict_factors)."""
    _lib.require_gpu()
    k = B.shape[1]
    dimA = Xr_indptr.shape[0] - 1
    A = np.empty((dimA, k), dtype=B.dtype)
    rc = _lib.lib().pmf_b200_factors_multiple(
        _lib.dtype_code(B.dtype), _lib.index_bytes(Xr_indptr), _lib.ptr(A), _lib.ptr(B), _lib.ptr(Bsum),
        _lib.ptr(Amean), _lib.ptr(Xr), _lib.ptr(Xr_indptr), _lib.ptr(Xr_indices), k, dimA, B.shape[0],
        float(l2_reg), float(w_mult), float(step_size), int(niter), int(maxupd), _lib.METHODS[method],
        int(bool(limit_step)), int(bool(reuse_mean)), int(flags))
    if rc:
        raise MemoryError("Could not allocate enough memory.")
    return A


def _predict_multiple(out, A, B, ix_u, ix_i, nthreads=1):
    _lib.require_gpu()
    rc = _lib.lib().pmf_b200_predict_multiple(
        _lib.dtype_code(A.dtype), _lib.index_bytes(ix_u), _lib.ptr(out), _lib.ptr(A), _lib.ptr(B),
        _lib.ptr(ix_u), _lib.ptr(ix_i), ix_u.shape[0], A.shape[1], A.shape[0], B.shape[0])
    if rc:
        raise MemoryError(_lib.last_error())


def _call_topN(a_vec, B, include_ix, exclude_ix, top_n=10, output_score=False, nthreads=1, check=False):
    """poismf_c_wrapper.pxi:208-249.  Like the reference's wrapper the return code 2 (invalid arguments,
    src/topN.c:124-128) is NOT turned into an exception — PoisMF.topN validates its arguments before the
    call (poismf/__init__.py:933-975); `check=True` raises ValueError instead."""
    _lib.require_gpu()
    ixdt = np.uint64
    inc = np.ascontiguousarray(include_ix, dtype=ixdt)
    exc = np.ascontiguousarray(exclude_ix, dtype=ixdt)
    n_include = inc.shape[0]
    n_exclude = 0 if n_include else exc.shape[0]      # pxi :224-229: include wins
    outp_ix = np.empty(top_n, dtype=ixdt)
    outp_score = np.empty(top_n if output_score else 0, dtype=B.dtype)
    rc = _lib.lib().pmf_b200_topN(
        _lib.dtype_code(B.dtype), 8, _lib.ptr(a_vec), _lib.ptr(B), B.shape[1],
        _lib.ptr(inc) if n_include else None, n_include,
        _lib.ptr(exc) if n_exclude else None, n_exclude,
        _lib.ptr(outp_ix), _lib.ptr(outp_score) if output_score else None, top_n, B.shape[0])
    if rc == 1:
        raise MemoryError(_lib.last_error())
    if rc == 2 and check:
        raise ValueError("topN: invalid arguments")
    return outp_ix, outp_score


def _include_lists(incl_ptr, incl_ix, excl_ptr, excl_ix, n_users):
    """(incl_ptr, incl_ix) as uint64 arrays, or None without include lists.  Include and exclude lists together
    are invalid, as in the reference (src/topN.c:124-128), and so are offsets that do not cover n_users lists
    inside incl_ix."""
    if incl_ptr is None and incl_ix is None:
        return None
    if incl_ptr is None or incl_ix is None:
        raise ValueError("topN: incl_ptr and incl_ix go together")
    if excl_ptr is not None or excl_ix is not None:
        raise ValueError("topN: include and exclude lists cannot be combined")
    ptr = np.ascontiguousarray(incl_ptr, dtype=np.uint64)
    ix = np.ascontiguousarray(incl_ix, dtype=np.uint64)
    if ptr.ndim != 1 or ptr.shape[0] != n_users + 1 or int(ptr.max()) > ix.shape[0]:
        raise ValueError("topN: incl_ptr must hold n_users + 1 offsets into incl_ix")
    return ptr, ix


def _topN_batch(A, B, users=None, excl_ptr=None, excl_ix=None, top_n=10, output_score=False, incl_ptr=None,
                incl_ix=None):
    """Batched top-N for many users at once (no reference equivalent; include/poismf_b200.h).  With
    `incl_ptr` / `incl_ix` user u ranks only the items incl_ix[incl_ptr[u]:incl_ptr[u+1]]."""
    _lib.require_gpu()
    ixdt = np.uint64
    u = None if users is None else np.ascontiguousarray(users, dtype=ixdt)
    n_users = A.shape[0] if u is None else u.shape[0]
    include = _include_lists(incl_ptr, incl_ix, excl_ptr, excl_ix, n_users)
    outp_ix = np.empty((n_users, top_n), dtype=ixdt)
    outp_score = np.empty((n_users, top_n) if output_score else (0, 0), dtype=B.dtype)
    if include is not None:
        rc = _lib.lib().pmf_b200_topN_batch_include(
            _lib.dtype_code(B.dtype), 8, _lib.ptr(A), _lib.ptr(B), B.shape[1], _lib.ptr(u), n_users, A.shape[0],
            _lib.ptr(include[0]), _lib.ptr(include[1]), _lib.ptr(outp_ix),
            _lib.ptr(outp_score) if output_score else None, top_n, B.shape[0])
        if rc == 1:
            raise MemoryError(_lib.last_error())
        if rc == 2:
            raise ValueError("topN_batch: invalid arguments")
        return outp_ix, outp_score
    ep = None if excl_ptr is None else np.ascontiguousarray(excl_ptr, dtype=ixdt)
    ei = None if excl_ix is None else np.ascontiguousarray(excl_ix, dtype=ixdt)
    rc = _lib.lib().pmf_b200_topN_batch(
        _lib.dtype_code(B.dtype), 8, _lib.ptr(A), _lib.ptr(B), B.shape[1], _lib.ptr(u), n_users, A.shape[0],
        _lib.ptr(ep), _lib.ptr(ei), _lib.ptr(outp_ix), _lib.ptr(outp_score) if output_score else None,
        top_n, B.shape[0])
    if rc == 1:
        raise MemoryError(_lib.last_error())
    if rc == 2:
        raise ValueError("topN_batch: invalid arguments")
    return outp_ix, outp_score


def _fit_coo(rows, cols, counts, A, B, method="tncg", limit_step=False, l2_reg=1e9, l1_reg=0.0, w_mult=1.0,
             step_size=1e-7, niter=10, maxupd=1, early_stop=True, reuse_prev=True, flags=0):
    """PoisMF._process_data + _fit (poismf/__init__.py:376-440) in one call: the COO triplets are turned
    into CSR and CSC on the device (duplicates summed, ids sorted, as coo.tocsr()/tocsc()) and swept
    there.  No reference equivalent at the C level (include/poismf_b200.h)."""
    if counts.shape[0] == 0:
        raise ValueError("'X' contains no non-zero entries.")
    if rows.dtype != cols.dtype or A.dtype != B.dtype or A.dtype != counts.dtype:
        raise TypeError("rows/cols and A/B/counts must share their dtypes")
    _lib.require_gpu()
    rc = _lib.lib().pmf_b200_fit_coo(
        _lib.dtype_code(A.dtype), _lib.index_bytes(rows), _lib.ptr(A), _lib.ptr(B), _lib.ptr(rows), _lib.ptr(cols),
        _lib.ptr(counts), counts.shape[0], A.shape[0], B.shape[0], A.shape[1],
        float(l2_reg), float(l1_reg), float(w_mult), float(step_size), _lib.METHODS[method], int(bool(limit_step)),
        int(niter), int(maxupd), int(bool(early_stop)), int(bool(reuse_prev)), int(flags))
    if rc == 1:
        raise MemoryError(_lib.last_error() or "Could not allocate enough memory.")
    if rc == 2:
        raise ValueError(_lib.last_error() or "fit_coo: invalid triplets")
    return rc


def _coo_to_csr_csc(rows, cols, counts, dimA, dimB):
    """coo.tocsr(), coo.tocsc() on the device: ((data, indptr, indices) of CSR, same of CSC)."""
    _lib.require_gpu()
    n = counts.shape[0]
    ixdt = rows.dtype
    Xr, Xc = np.empty(n, counts.dtype), np.empty(n, counts.dtype)
    ri, ci = np.empty(n, ixdt), np.empty(n, ixdt)
    rp, cp = np.empty(dimA + 1, ixdt), np.empty(dimB + 1, ixdt)
    nnz = ctypes.c_size_t(0)
    rc = _lib.lib().pmf_b200_coo_to_csr_csc(
        _lib.dtype_code(counts.dtype), _lib.index_bytes(rows), _lib.ptr(rows), _lib.ptr(cols), _lib.ptr(counts),
        n, dimA, dimB, _lib.ptr(Xr), _lib.ptr(rp), _lib.ptr(ri), _lib.ptr(Xc), _lib.ptr(cp), _lib.ptr(ci),
        ctypes.byref(nnz))
    if rc == 2:
        raise ValueError(_lib.last_error() or "invalid triplets")
    if rc:
        raise MemoryError(_lib.last_error())
    m = nnz.value
    return (Xr[:m].copy(), rp, ri[:m].copy()), (Xc[:m].copy(), cp, ci[:m].copy())

