"""Device-resident fit: the handle API of include/poismf_b200.h from Python.

`DeviceFit` keeps the factors and both orientations of the count matrix in HBM
between sweeps; this is what bench.py times as the kernel-level figure, and what
the sharding layer drives half-sweep by half-sweep.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib


class DeviceFit:
    def __init__(self, dimA, dimB, k, dtype=np.float32, device=0):
        _lib.require_gpu()
        self.L = _lib.lib()
        self.dtype = np.dtype(dtype)
        self.dimA, self.dimB, self.k = int(dimA), int(dimB), int(k)
        self.h = self.L.pmf_b200_create(_lib.dtype_code(dtype), self.dimA, self.dimB, self.k, int(device))
        if not self.h:
            raise MemoryError(_lib.last_error())
        self.ldf = self.L.pmf_b200_ldf(self.h)

    def close(self):
        if getattr(self, "h", None):
            self.L.pmf_b200_destroy(self.h)
            self.h = None

    __del__ = close

    def _ck(self, rc):
        if rc == 1:
            raise MemoryError(_lib.last_error())
        return rc

    def set_matrix(self, side, values, indptr, indices, row_begin=0, n_rows=None):
        n_rows = (indptr.shape[0] - 1) if n_rows is None else n_rows
        assert values.dtype == self.dtype and values.flags.c_contiguous
        self._ck(self.L.pmf_b200_set_matrix(self.h, side, _lib.ptr(values), _lib.ptr(indptr), _lib.ptr(indices),
                                            values.shape[0], _lib.index_bytes(indptr), row_begin, n_rows))

    def set_csr_csc(self, csr, csc):
        self.set_matrix(_lib.SIDE_CSR, *csr)
        self.set_matrix(_lib.SIDE_CSC, *csc)

    def set_factors(self, A=None, B=None):
        for M in (A, B):
            assert M is None or (M.dtype == self.dtype and M.flags.c_contiguous)
        self._ck(self.L.pmf_b200_set_factors(self.h, _lib.ptr(A), _lib.ptr(B)))

    def get_factors(self, A=None, B=None):
        A = np.empty((self.dimA, self.k), self.dtype) if A is None else A
        B = np.empty((self.dimB, self.k), self.dtype) if B is None else B
        self._ck(self.L.pmf_b200_get_factors(self.h, _lib.ptr(A), _lib.ptr(B)))
        return A, B

    def bind_factors(self, A_dev_ptr=None, B_dev_ptr=None):
        self._ck(self.L.pmf_b200_bind_factors(self.h, A_dev_ptr, B_dev_ptr))

    def set_factor_rows(self, which, rows, row_begin):
        """Rows [row_begin, row_begin + len(rows)) of A (0) / B (1) into this replica and every peer's."""
        assert rows.dtype == self.dtype and rows.flags.c_contiguous
        self._ck(self.L.pmf_b200_set_factor_rows(self.h, which, _lib.ptr(rows), row_begin, rows.shape[0]))

    def topN(self, users=None, excl_ptr=None, excl_ix=None, top_n=10, output_score=False, incl_ptr=None,
             incl_ix=None):
        """Batched top-N of `users` (default: every user) against the factors resident in this handle — after a
        fit nothing but the ids travels (include/poismf_b200.h: pmf_b200_topN_fitted).  With `incl_ptr` /
        `incl_ix` user u ranks only the items incl_ix[incl_ptr[u]:incl_ptr[u+1]] (pmf_b200_topN_fitted_include)."""
        from .c_funs import _include_lists
        ixdt = np.uint64
        u = None if users is None else np.ascontiguousarray(users, dtype=ixdt)
        n_users = self.dimA if u is None else u.shape[0]
        include = _include_lists(incl_ptr, incl_ix, excl_ptr, excl_ix, n_users)
        ids = np.empty((n_users, top_n), dtype=ixdt)
        sc = np.empty((n_users, top_n) if output_score else (0, 0), dtype=self.dtype)
        if include is not None:
            rc = self.L.pmf_b200_topN_fitted_include(self.h, 8, _lib.ptr(u), n_users, _lib.ptr(include[0]),
                                                     _lib.ptr(include[1]), _lib.ptr(ids),
                                                     _lib.ptr(sc) if output_score else None, top_n)
        else:
            ep = None if excl_ptr is None else np.ascontiguousarray(excl_ptr, dtype=ixdt)
            ei = None if excl_ix is None else np.ascontiguousarray(excl_ix, dtype=ixdt)
            rc = self.L.pmf_b200_topN_fitted(self.h, 8, _lib.ptr(u), n_users, _lib.ptr(ep), _lib.ptr(ei),
                                             _lib.ptr(ids), _lib.ptr(sc) if output_score else None, top_n)
        if rc == 2:
            raise ValueError("topN: invalid arguments")
        self._ck(rc)
        return ids, sc

    def fit_stats(self, l1_reg=0.0):
        """(Bsum, Amean) of the resident factors: column sums of B plus l1_reg, column means of A — the attributes
        PoisMF keeps after a fit (pmf_b200_fit_stats; fixed summation order, the same bits on every replica)."""
        Bsum, Amean = np.empty(self.k, self.dtype), np.empty(self.k, self.dtype)
        self._ck(self.L.pmf_b200_fit_stats(self.h, float(l1_reg), _lib.ptr(Bsum), _lib.ptr(Amean)))
        return Bsum, Amean

    def _new_users(self, Xr_indptr, Xr_indices, Xr, params, Bsum, Amean, **kw):
        from .c_funs import _new_users
        Bs = None if Bsum is None else np.ascontiguousarray(Bsum, dtype=self.dtype)
        Am = None if Amean is None else np.ascontiguousarray(Amean, dtype=self.dtype)

        def call(ib, *args):
            return self.L.pmf_b200_topN_new_fitted(self.h, ib, _lib.ptr(Bs), _lib.ptr(Am), *args)
        return _new_users(call, Xr_indptr, Xr_indices, Xr, self.k, self.dtype, params, **kw)

    def topN_new(self, Xr_indptr, Xr_indices, Xr, top_n=10, output_score=False, excl_ptr=None, excl_ix=None,
                 incl_ptr=None, incl_ix=None, reuse_mean=True, maxupd=20, l2_reg=1e5, l1_new=0.0, l1_old=0.0,
                 w_mult=1.0, return_factors=False, flags=0, Bsum=None, Amean=None, l1_reg=0.0):
        """c_funs._topN_new_batch against the item factors resident in this handle (pmf_b200_topN_new_fitted): the new
        users' CSR rows are folded in and ranked without B leaving the device.  With Bsum=None the column sums come
        from the resident B and the model's total `l1_reg` is added to them; with the model's Bsum given, the positive
        part of l1_new - l1_old is (as in `_predict_factors`).  Amean=None: the column means of the resident A."""
        from .c_funs import _positive_l1
        l1 = float(self.dtype.type(l1_reg)) if Bsum is None else _positive_l1(self.dtype, l1_new, l1_old)
        params = _lib.make_params("tncg", l2_reg, l1_reg=l1, w_mult=w_mult, step_size=0.0, numiter=1, maxupd=maxupd,
                                  reuse_prev=reuse_mean, flags=flags)
        return self._new_users(Xr_indptr, Xr_indices, Xr, params, Bsum, Amean, top_n=top_n, output_score=output_score,
                               excl_ptr=excl_ptr, excl_ix=excl_ix, incl_ptr=incl_ptr, incl_ix=incl_ix,
                               return_factors=return_factors)

    def transform(self, Xr_indptr, Xr_indices, Xr, method="tncg", niter=10, maxupd=1, l2_reg=1e9, w_mult=1.0,
                  step_size=1e-7, limit_step=False, reuse_mean=True, Bsum=None, Amean=None, flags=0):
        """Factors of new users' CSR rows against the resident item factors (PoisMF.transform): the fold-in of
        c_funs._predict_factors_multiple (same keywords) with B read in place.  Bsum / Amean default to fit_stats()."""
        params = _lib.make_params(method, l2_reg, w_mult=w_mult, step_size=step_size, limit_step=limit_step,
                                  numiter=niter, maxupd=maxupd, reuse_prev=reuse_mean, flags=flags)
        return self._new_users(Xr_indptr, Xr_indices, Xr, params, Bsum, Amean, rank=False)

    def factor_ptr(self, which):
        return self.L.pmf_b200_factor_ptr(self.h, which)

    def set_stream(self, stream_ptr):
        self._ck(self.L.pmf_b200_set_stream(self.h, stream_ptr))

    def sweeps(self, params):
        return self._ck(self.L.pmf_b200_sweeps(self.h, C.byref(params)))

    def half_sweep(self, side, params, step_size, cnst_div):
        n = C.c_ulonglong(0)
        self._ck(self.L.pmf_b200_half_sweep(self.h, side, C.byref(params), float(step_size), float(cnst_div),
                                            C.byref(n)))
        return n.value

    def ipc_export(self, which):
        buf = (C.c_ubyte * 64)()
        self._ck(self.L.pmf_b200_ipc_export(self.h, which, buf))
        return bytes(buf)

    def ipc_import(self, which, handles, self_rank):
        blob = b"".join(handles)
        self._ck(self.L.pmf_b200_ipc_import(self.h, which, blob, len(handles), self_rank))

    def set_profiling(self, on=True):
        self.L.pmf_b200_set_profiling(self.h, int(on))

    def get_profile(self):
        arr = (_lib.BinProfile * 64)()
        n = self.L.pmf_b200_get_profile(self.h, arr, 64)
        return [dict(side=a.side, block_team=a.block_team, cap=a.cap, nrows=a.nrows, nnz=a.nnz,
                     launches=a.launches, ms=a.ms) for a in arr[:n]]

    def sync(self):
        self._ck(self.L.pmf_b200_sync(self.h))
