"""TEST INFRASTRUCTURE ONLY — ctypes loaders for the CPU checkers.

  * `Ref(dtype, fast=False)`  : the reference's own C sources compiled by
    oracle/Makefile into oracle/_ref/ (prebuilt .so travels to the GPU box).
  * `Restatement(dtype, fast=False)` : this repo's plain-C restatement (oracle/poismf_oracle.c).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
legs may import this module.  The product package (poismf_b200) never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
METHODS = {"tncg": 1, "cg": 2, "pg": 3}
_sz = C.c_size_t


def build(verbose=False):
    """Compile the restatement (always) and oracle/_ref (only where /root/reference exists)."""
    r = subprocess.run(["make", "-C", HERE, "all"], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("oracle build failed:\n" + r.stdout + r.stderr)
    if verbose:
        print(r.stdout)


def _real(dtype):
    dtype = np.dtype(dtype)
    if dtype == np.float64:
        return C.c_double, "double"
    if dtype == np.float32:
        return C.c_float, "float"
    raise TypeError(dtype)


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


class _Base:
    def __init__(self, path, dtype):
        if not os.path.exists(path):
            raise FileNotFoundError(f"{path} missing: run `make -C oracle`")
        self.lib = C.CDLL(path)
        self.dtype = np.dtype(dtype)
        self.creal, _ = _real(dtype)

    def _chk(self, *arrs):
        for a in arrs:
            assert a.flags.c_contiguous


class Ref(_Base):
    """The reference's own implementation (src/poismf.h prototypes)."""

    def __init__(self, dtype, fast=False):
        _, name = _real(dtype)
        stem = "libpoismf_reffast_" if fast else "libpoismf_ref_"
        super().__init__(os.path.join(HERE, "_ref", stem + name + ".so"), dtype)

    @staticmethod
    def available(dtype=np.float64, fast=False):
        _, name = _real(dtype)
        stem = "libpoismf_reffast_" if fast else "libpoismf_ref_"
        return os.path.exists(os.path.join(HERE, "_ref", stem + name + ".so"))

    def run_poismf(self, A, B, csr, csc, method, l2_reg, l1_reg=0.0, w_mult=1.0, step_size=1e-7,
                   limit_step=False, numiter=1, maxupd=1, early_stop=False, reuse_prev=False,
                   nthreads=1):
        r = self.creal
        Xr, Xr_ptr, Xr_ind = csr
        Xc, Xc_ptr, Xc_ind = csc
        self._chk(A, B, Xr, Xr_ptr, Xr_ind, Xc, Xc_ptr, Xc_ind)
        f = self.lib.run_poismf
        f.restype = C.c_int
        f.argtypes = [C.c_void_p] * 8 + [_sz, _sz, _sz, r, r, r, r, C.c_int, C.c_bool, _sz, _sz,
                                         C.c_bool, C.c_bool, C.c_bool, C.c_int]
        return f(_p(A), _p(Xr), _p(Xr_ptr), _p(Xr_ind), _p(B), _p(Xc), _p(Xc_ptr), _p(Xc_ind),
                 A.shape[0], B.shape[0], A.shape[1], l2_reg, l1_reg, w_mult, step_size,
                 METHODS[method], limit_step, numiter, maxupd, early_stop, reuse_prev, False, nthreads)

    def predict_multiple(self, A, B, ixA, ixB, nthreads=1):
        out = np.empty(ixA.shape[0], dtype=self.dtype)
        f = self.lib.predict_multiple
        f.restype = None
        f.argtypes = [C.c_void_p] * 5 + [_sz, C.c_int, C.c_int]
        f(_p(out), _p(A), _p(B), _p(ixA), _p(ixB), ixA.shape[0], A.shape[1], nthreads)
        return out

    def factors_multiple(self, B, Bsum, Amean, csr, method, l2_reg, w_mult=1.0, step_size=1e-7, niter=10,
                         maxupd=1, limit_step=False, reuse_mean=True, nthreads=1):
        r = self.creal
        Xr, ptr, ind = csr
        dimA, k = ptr.shape[0] - 1, B.shape[1]
        A = np.empty((dimA, k), dtype=self.dtype)
        f = self.lib.factors_multiple
        f.restype = C.c_int
        f.argtypes = [C.c_void_p] * 7 + [C.c_int, _sz, r, r, r, _sz, _sz, C.c_int, C.c_bool, C.c_bool, C.c_int]
        rc = f(_p(A), _p(B), _p(Bsum), _p(Amean), _p(Xr), _p(ptr), _p(ind), k, dimA, l2_reg, w_mult, step_size,
               niter, maxupd, METHODS[method], limit_step, reuse_mean, nthreads)
        return rc, A

    def factors_single(self, counts, ix, B, Bsum, Amean, reuse_mean=True, maxupd=20, l2_reg=1e5,
                       l1_new=0.0, l1_old=0.0, w_mult=1.0):
        """src/pred.c:201-304 (argument order of poismf_c_wrapper.pxi:114-145 `_predict_factors`)."""
        r = self.creal
        k = B.shape[1]
        out = np.empty(k, dtype=self.dtype)
        f = self.lib.factors_single
        f.restype = C.c_int
        f.argtypes = [C.c_void_p, _sz, C.c_void_p, C.c_bool, C.c_void_p, C.c_void_p, _sz, C.c_void_p, C.c_void_p,
                      C.c_int, r, r, r, r]
        rc = f(_p(out), k, _p(Amean), reuse_mean, _p(counts) if counts.size else None, _p(ix) if ix.size else None,
               counts.shape[0], _p(B), _p(Bsum), maxupd, l2_reg, l1_new, l1_old, w_mult)
        return rc, out

    def topN(self, a_vec, B, n_top, include=None, exclude=None, nthreads=1):
        out_ix = np.empty(n_top, dtype=np.uint64)
        out_sc = np.empty(n_top, dtype=self.dtype)
        inc = np.ascontiguousarray(include, dtype=np.uint64) if include is not None else np.empty(0, np.uint64)
        exc = np.ascontiguousarray(exclude, dtype=np.uint64).copy() if exclude is not None else np.empty(0, np.uint64)
        f = self.lib.topN
        f.restype = C.c_int
        f.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, _sz, C.c_void_p, _sz,
                      C.c_void_p, C.c_void_p, _sz, _sz, C.c_int]
        rc = f(_p(a_vec), _p(B), B.shape[1], _p(inc) if inc.size else None, inc.size,
               _p(exc) if exc.size else None, exc.size, _p(out_ix), _p(out_sc), n_top, B.shape[0], nthreads)
        return rc, out_ix, out_sc


class Restatement(_Base):
    """This repo's restatement of the same algorithm (oracle/poismf_oracle.c); `fast=True` loads
    it compiled with the reference's fast flags (-O3, FMA contraction)."""

    def __init__(self, dtype, fast=False):
        _, name = _real(dtype)
        stem = "libpoismf_oraclefast_" if fast else "libpoismf_oracle_"
        super().__init__(os.path.join(HERE, stem + name + ".so"), dtype)

    def run_poismf(self, A, B, csr, csc, method, l2_reg, l1_reg=0.0, w_mult=1.0, step_size=1e-7,
                   limit_step=False, numiter=1, maxupd=1, early_stop=False, reuse_prev=False,
                   nthreads=1):
        r = self.creal
        Xr, Xr_ptr, Xr_ind = csr
        Xc, Xc_ptr, Xc_ind = csc
        self._chk(A, B, Xr, Xr_ptr, Xr_ind, Xc, Xc_ptr, Xc_ind)
        f = self.lib.oracle_run_poismf
        f.restype = C.c_int
        f.argtypes = [C.c_void_p] * 8 + [_sz, _sz, _sz, r, r, r, r, C.c_int, C.c_int, _sz, _sz,
                                         C.c_int, C.c_int]
        return f(_p(A), _p(Xr), _p(Xr_ptr), _p(Xr_ind), _p(B), _p(Xc), _p(Xc_ptr), _p(Xc_ind),
                 A.shape[0], B.shape[0], A.shape[1], l2_reg, l1_reg, w_mult, step_size,
                 METHODS[method], int(limit_step), numiter, maxupd, int(early_stop), int(reuse_prev))

    def factors_multiple(self, B, Bsum, Amean, csr, method, l2_reg, w_mult=1.0, step_size=1e-7, niter=10,
                         maxupd=1, limit_step=False, reuse_mean=True):
        r = self.creal
        Xr, ptr, ind = csr
        dimA, k = ptr.shape[0] - 1, B.shape[1]
        A = np.empty((dimA, k), dtype=self.dtype)
        f = self.lib.oracle_factors_multiple
        f.restype = C.c_int
        f.argtypes = [C.c_void_p] * 7 + [C.c_int, _sz, r, r, r, _sz, _sz, C.c_int, C.c_int, C.c_int]
        rc = f(_p(A), _p(B), _p(Bsum), _p(Amean), _p(Xr), _p(ptr), _p(ind), k, dimA, l2_reg, w_mult, step_size,
               niter, maxupd, METHODS[method], int(limit_step), int(reuse_mean))
        return rc, A

    def factors_single(self, counts, ix, B, Bsum, Amean, reuse_mean=True, maxupd=20, l2_reg=1e5,
                       l1_new=0.0, l1_old=0.0, w_mult=1.0):
        r = self.creal
        k = B.shape[1]
        out = np.empty(k, dtype=self.dtype)
        f = self.lib.oracle_factors_single
        f.restype = C.c_int
        f.argtypes = [C.c_void_p, _sz, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, _sz, C.c_void_p, C.c_void_p,
                      C.c_int, r, r, r, r]
        rc = f(_p(out), k, _p(Amean), int(reuse_mean), _p(counts) if counts.size else None,
               _p(ix) if ix.size else None, counts.shape[0], _p(B), _p(Bsum), maxupd, l2_reg, l1_new, l1_old, w_mult)
        return rc, out

    def eval(self, a, F, csum, xval, xind, l2, w):
        """(f_cg, g_cg, f_tn, g_tn) at point a for one row."""
        r = self.creal
        k = a.shape[0]
        g_cg = np.empty(k, self.dtype); g_tn = np.empty(k, self.dtype)
        f_cg = r(); f_tn = r()
        fn = self.lib.oracle_eval
        fn.restype = None
        fn.argtypes = [C.c_void_p] * 5 + [C.c_uint64, C.c_int, r, r, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        fn(_p(a), _p(F), _p(csum), _p(xval), _p(xind), xval.shape[0], k, l2, w,
           C.byref(f_cg), _p(g_cg), C.byref(f_tn), _p(g_tn))
        return f_cg.value, g_cg, f_tn.value, g_tn

    def predict_multiple(self, A, B, ixA, ixB):
        out = np.empty(ixA.shape[0], dtype=self.dtype)
        f = self.lib.oracle_predict_multiple
        f.restype = None
        f.argtypes = [C.c_void_p] * 5 + [_sz, C.c_int]
        f(_p(out), _p(A), _p(B), _p(ixA), _p(ixB), ixA.shape[0], A.shape[1])
        return out

    def topN(self, a_vec, B, n_top, include=None, exclude=None):
        out_ix = np.empty(n_top, dtype=np.uint64)
        out_sc = np.empty(n_top, dtype=self.dtype)
        inc = np.ascontiguousarray(include, dtype=np.uint64) if include is not None else np.empty(0, np.uint64)
        exc = np.ascontiguousarray(exclude, dtype=np.uint64) if exclude is not None else np.empty(0, np.uint64)
        f = self.lib.oracle_topN
        f.restype = C.c_int
        f.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, _sz, C.c_void_p, _sz,
                      C.c_void_p, C.c_void_p, _sz, _sz]
        rc = f(_p(a_vec), _p(B), B.shape[1], _p(inc) if inc.size else None, inc.size,
               _p(exc) if exc.size else None, exc.size, _p(out_ix), _p(out_sc), n_top, B.shape[0])
        return rc, out_ix, out_sc

    def llk(self, A, B, csr):
        Xr, Xr_ptr, Xr_ind = csr
        f = self.lib.oracle_llk
        f.restype = C.c_double
        f.argtypes = [C.c_void_p] * 5 + [_sz, _sz, _sz]
        return f(_p(A), _p(B), _p(Xr), _p(Xr_ptr), _p(Xr_ind), A.shape[0], B.shape[0], A.shape[1])
