import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session", autouse=True)
def _built():
    """Make sure the product library and the CPU checkers exist (no-op when prebuilt)."""
    from poismf_b200 import _lib
    from oracle import oracle
    if not os.path.exists(_lib.LIB_PATH):
        from poismf_b200.build import build
        build()
    if not os.path.exists(os.path.join(ROOT, "oracle", "libpoismf_oracle_double.so")):
        oracle.build()
    yield


def golden():
    """Committed outputs of the reference (tests/golden/make_golden.py), stored one file per dtype."""
    out = {}
    for name in ("float64", "float32"):
        out.update(np.load(os.path.join(ROOT, "tests", "golden", f"reference_outputs_{name}.npz")))
    return out


def has_gpu():
    try:
        from poismf_b200 import _lib
        return _lib.lib().pmf_b200_device_count() > 0
    except Exception:
        return False


# ---- shared problem builders -------------------------------------------------
CASES = {
    # name: (method, hyper-parameters)   [maxupd None -> 15*k as poismf/__init__.py:252]
    "pg": ("pg", dict(l2_reg=1e9, step_size=1e-7, maxupd=1, numiter=2)),
    "pg_w": ("pg", dict(l2_reg=1e3, step_size=1e-4, maxupd=3, numiter=2, w_mult=2.5, l1_reg=0.1)),
    "cg": ("cg", dict(l2_reg=1e4, maxupd=5, numiter=1, limit_step=True)),
    "cg_nolimit_w": ("cg", dict(l2_reg=1e3, maxupd=5, numiter=2, limit_step=False, w_mult=1.5)),
    "tncg": ("tncg", dict(l2_reg=1e3, maxupd=None, numiter=1)),
    "tncg_reuse_stop": ("tncg", dict(l2_reg=1e2, maxupd=None, numiter=3, reuse_prev=True, early_stop=True, l1_reg=0.5)),
    "tncg_w": ("tncg", dict(l2_reg=1e3, maxupd=None, numiter=2, w_mult=3.0)),
}


def problem(name, dtype):
    from poismf_b200.synth import init_factors, powerlaw_counts, readme_counts
    if name == "readme":
        csr, csc = readme_counts(dtype=dtype)
        k = 5
    elif name == "pl2k":
        csr, csc = powerlaw_counts(2000, 800, 60000, dtype=dtype)
        k = 16
    elif name == "pl6k":
        csr, csc = powerlaw_counts(6000, 2500, 300000, dtype=dtype)
        k = 50
    elif name == "ragged":   # empty rows/cols, single-nnz rows, k not a multiple of 4
        csr, csc = powerlaw_counts(300, 4000, 2500, alpha_a=1.2, alpha_b=0.3, dtype=dtype, seed=7)
        k = 7
    else:
        raise KeyError(name)
    dimA, dimB = csr[1].shape[0] - 1, csc[1].shape[0] - 1
    A0, B0 = init_factors(dimA, dimB, k, dtype=dtype)
    return csr, csc, A0, B0, k


def hyper(case, k):
    method, kw = CASES[case]
    kw = dict(kw)
    if kw["maxupd"] is None:
        kw["maxupd"] = 15 * k
    return method, kw


def run_device(csr, csc, A, B, method, kw, flags=0):
    from poismf_b200 import c_funs
    return c_funs._run_poismf(csr[0], csr[2], csr[1], csc[0], csc[2], csc[1], A, B, method=method,
                              limit_step=kw.get("limit_step", False), l2_reg=kw["l2_reg"],
                              l1_reg=kw.get("l1_reg", 0.), w_mult=kw.get("w_mult", 1.),
                              step_size=kw.get("step_size", 1e-7), niter=kw["numiter"], maxupd=kw["maxupd"],
                              early_stop=kw.get("early_stop", False), reuse_prev=kw.get("reuse_prev", False),
                              flags=flags)


def row_rel_err(X, Y):
    return np.linalg.norm(X - Y, axis=1) / np.maximum(np.linalg.norm(Y, axis=1), 1e-30)


FM_CASES = {
    "pg": ("pg", dict(l2_reg=1e3, step_size=1e-4, niter=4, maxupd=2)),
    "pg_w": ("pg", dict(l2_reg=1e3, step_size=1e-4, niter=3, maxupd=1, w_mult=2.0)),
    "cg": ("cg", dict(l2_reg=1e3, niter=3, maxupd=2, limit_step=True)),
    "cg_w": ("cg", dict(l2_reg=1e3, niter=2, maxupd=3, w_mult=1.5)),
    "tncg": ("tncg", dict(l2_reg=1e3, maxupd=None)),
    "tncg_w_nomean": ("tncg", dict(l2_reg=1e3, maxupd=None, reuse_mean=False, w_mult=2.0)),
}


def fm_problem(name, dtype):
    """Inputs of factors_multiple: new rows = the problem's CSR, B random non-negative, Bsum = colsum + l1."""
    csr, csc, A0, B0, k = problem(name, dtype)
    rng = np.random.default_rng(5)
    B = np.ascontiguousarray(rng.gamma(1, 0.3, size=B0.shape).astype(dtype))
    Bsum = np.ascontiguousarray((B.sum(0) + 0.1).astype(dtype))
    Amean = np.ascontiguousarray(rng.gamma(1, .3, size=k).astype(dtype))
    return csr, B, Bsum, Amean, k


# factors_single (src/pred.c:201-304): rows of the factors_multiple problem, one at a time
FS_CASES = {
    "plain": dict(),
    "nomean": dict(reuse_mean=False),
    "w": dict(w_mult=2.0),
    "l1": dict(l1_new=0.5, l1_old=0.1),
    "l1_neg": dict(l1_new=0.0, l1_old=0.3, l2_reg=1e2),
    "l1_w": dict(l1_new=0.5, l1_old=0.1, w_mult=1.5, maxupd=100),
}
FS_ROWS = (0, 3, 7, 50)


def fs_row(csr, row):
    lo, hi = int(csr[1][row]), int(csr[1][row + 1])
    return np.ascontiguousarray(csr[0][lo:hi]), np.ascontiguousarray(csr[2][lo:hi])


def fm_hyper(case, k):
    method, kw = FM_CASES[case]
    kw = dict(kw)
    if kw.get("maxupd", 0) is None:
        kw["maxupd"] = 15 * k
    return method, kw


# ---- per-row objective of the cg sub-problem, in float64 (calc_fun_single, src/poismf.c:194-208) ----
def row_objectives(M, F, mat, l2, w=1.0, l1=0.0, with_l2=True, chunk=1 << 22):
    """f_i = <colsum(F)+l1, m_i> + l2 |m_i|^2 - w * sum_j x_ij log <m_i, F_j> for every row i of the
    compressed matrix `mat` = (values, indptr, indices); rows without non-zeros get the regulariser only.
    `with_l2=False` gives tncg's objective (quirk Q3).  Rows whose prediction is <= 0 get +inf."""
    vals, ptr, ind = mat
    ptr = ptr.astype(np.int64)
    M64 = M.astype(np.float64)
    csum = F.sum(axis=0, dtype=np.float64) + l1
    f = M64 @ csum
    if with_l2:
        f += l2 * np.einsum("ij,ij->i", M64, M64)
    rows = np.repeat(np.arange(M.shape[0]), np.diff(ptr))
    ls = np.zeros(M.shape[0])
    with np.errstate(divide="ignore", invalid="ignore"):
        for s in range(0, rows.shape[0], chunk):
            sl = slice(s, s + chunk)
            p = np.einsum("ij,ij->i", M64[rows[sl]], F[ind[sl].astype(np.int64)].astype(np.float64))
            t = vals[sl].astype(np.float64) * np.log(p)
            t[~(p > 0)] = -np.inf
            ls += np.bincount(rows[sl], weights=t, minlength=M.shape[0])
    return f - w * ls
