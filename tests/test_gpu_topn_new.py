"""Batched top-N for new users (pmf_b200_topN_new_batch / _fitted, pmf_b200_fit_stats): the fold-in of every user is
bitwise the one-row fold-in of `_predict_factors` (a row's kernel follows from its length alone), and the ranking is
bitwise `_topN_batch` / its include-list form on those factors."""
import ctypes as C
import os
import socket

import numpy as np
import pytest

from conftest import FM_CASES, FS_CASES, FS_ROWS, fm_hyper, fm_problem, fs_row, problem, row_rel_err
from oracle.oracle import Restatement

pytestmark = pytest.mark.gpu
DTYPES = [np.float64, np.float32]
STRICT = 1


def _csr(rows):
    """CSR (values, indptr uint64, indices uint64) of a list of (values, ids) rows."""
    ptr = np.concatenate([[0], np.cumsum([len(v) for v, _ in rows])]).astype(np.uint64)
    vals = np.concatenate([v for v, _ in rows]) if rows else np.empty(0)
    ind = np.concatenate([i for _, i in rows]).astype(np.uint64)
    return np.ascontiguousarray(vals), ptr, np.ascontiguousarray(ind)


def _batch_rows(csr, rng, extra=40):
    """FS_ROWS, the longest row, random rows and three empty rows of a problem's CSR, and each row's source row
    (None for the empty ones)."""
    n = csr[1].shape[0] - 1
    lens = np.diff(csr[1].astype(np.int64))
    pick = list(FS_ROWS) + [int(lens.argmax())] + [int(r) for r in rng.choice(n, min(extra, n), replace=False)]
    pick = pick[:2] + [None] + pick[2:] + [None, None]
    empty = (np.empty(0, csr[0].dtype), np.empty(0, np.uint64))
    return [empty if r is None else fs_row(csr, r) for r in pick], pick


def _synthetic(dtype, n_new, n, k, seed, lo=5, hi=60):
    """New users with lo..hi interactions over n items drawn with a popularity skew; B, Bsum, Amean seeded."""
    rng = np.random.default_rng(seed)
    B = np.ascontiguousarray(rng.gamma(1.0, 0.3, size=(n, k)).astype(dtype))
    Bsum = np.ascontiguousarray(B.sum(0, dtype=np.float64).astype(dtype))
    Amean = np.ascontiguousarray(rng.gamma(1.0, 0.3, size=k).astype(dtype))
    pop = 1.0 / np.arange(1, n + 1) ** 0.8
    pop /= pop.sum()
    rows = []
    for m in rng.integers(lo, hi + 1, n_new):
        ids = np.sort(rng.choice(n, int(m), replace=False, p=pop))
        rows.append((rng.integers(1, 6, ids.shape[0]).astype(dtype), ids.astype(np.uint64)))
    return _csr(rows), B, Bsum, Amean


# ---------------------------------------------------------------- 1. fold-in parity with the one-row fold-in
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("case", list(FS_CASES))
@pytest.mark.parametrize("flags", [STRICT, 0])
def test_fold_in_equals_single_row(dtype, case, flags):
    from poismf_b200 import c_funs
    kw = FS_CASES[case]
    tol = 1e-9 if dtype == np.float64 else 1e-5
    for prob in ("readme", "pl2k"):
        csr, B, Bsum, Amean, k = fm_problem(prob, dtype)
        rows, src = _batch_rows(csr, np.random.default_rng(1))
        new = _csr(rows)
        ids, sc, A = c_funs._topN_new_batch(new[1], new[2], new[0], B, Bsum, Amean, top_n=5, return_factors=True,
                                            flags=flags, **kw)
        assert A.shape == (len(rows), k) and ids.shape == (len(rows), 5)
        for r, (c, ix) in enumerate(rows):
            one = c_funs._predict_factors(c, ix, B, Bsum, Amean, flags=flags, **kw)
            assert np.array_equal(A[r], one), (prob, r, len(c))
            if not len(c):
                assert not A[r].any()
            elif flags == STRICT and src[r] in FS_ROWS:        # the rows test_factors_single_matches_oracle gates
                want = Restatement(dtype).factors_single(c, ix, B, Bsum, Amean, **kw)[1]
                assert row_rel_err(A[r][None], want[None]).max() <= tol, (prob, r)


# ---------------------------------------------------------------- 2. ranking parity
def _oracle_ids_outside_ties(dtype, A_rows, B, n_top, excl=None, incl=None):
    """Per user: the oracle's ranking of its own factors, and a mask of the positions whose score is separated from
    its neighbours (the next item beyond n_top included) by more than the factors' rounding noise."""
    orc = Restatement(dtype)
    rel = 1e-3 if dtype == np.float32 else 1e-4
    out = []
    for u, a in enumerate(A_rows):
        kw = {}
        if excl is not None:
            kw["exclude"] = np.array(excl[u])          # (the oracle sorts its exclusion list in place)
        if incl is not None:
            kw["include"] = incl[u]
        m = n_top + 1 if (incl is None or len(incl[u]) > n_top) else n_top
        rc, o_ids, o_sc = orc.topN(np.ascontiguousarray(a), B, m, **kw)
        assert rc == 0
        s = o_sc.astype(np.float64)
        gap = np.abs(np.diff(s)) > rel * np.abs(s[:-1]).clip(1e-30)
        sep = np.ones(m, bool)
        sep[1:] &= gap
        sep[:-1] &= gap
        out.append((o_ids[:n_top], sep[:n_top]))
    return out


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("prob", ["pl2k", "synthetic"])
def test_ranking_equals_topn_batch(dtype, prob):
    from poismf_b200 import _lib, c_funs
    rng = np.random.default_rng(2)
    if prob == "pl2k":
        new, B, Bsum, Amean, k = fm_problem("pl2k", dtype)
        kw = dict(l2_reg=1e3)
    else:
        new, B, Bsum, Amean = _synthetic(dtype, 600, 20_000, 32, 3)
        kw = dict(l2_reg=1e4, maxupd=30)
    n_new, n = new[1].shape[0] - 1, B.shape[0]
    n_top = 10
    ilens = rng.integers(n_top, 400, n_new)
    iptr = np.concatenate([[0], np.cumsum(ilens)]).astype(np.uint64)
    iix = np.concatenate([rng.choice(n, int(m), replace=False) for m in ilens]).astype(np.uint64)
    variants = {"none": {}, "own": dict(excl_ptr=new[1], excl_ix=new[2]), "include": dict(incl_ptr=iptr, incl_ix=iix)}
    sample = rng.choice(n_new, 25, replace=False)
    for name, lists in variants.items():
        _lib.topn_stats(reset=True)
        ids, sc, A = c_funs._topN_new_batch(new[1], new[2], new[0], B, Bsum, Amean, top_n=n_top, output_score=True,
                                            return_factors=True, **lists, **kw)
        tc, _ = _lib.topn_stats(reset=True)
        ref = c_funs._topN_batch(A, B, top_n=n_top, output_score=True, **lists)
        assert np.array_equal(ids, ref[0]) and np.array_equal(sc, ref[1]), name
        if dtype == np.float32 and name != "include":
            assert tc == n_new, (name, tc)            # every user scored on the tensor cores
        if name == "own":
            for u in range(n_new):
                assert not np.isin(ids[u], new[2][int(new[1][u]):int(new[1][u + 1])]).any()
        # the oracle's fold-in and ranking, outside ties
        A_o = np.stack([Restatement(dtype).factors_single(*fs_row(new, int(u)), B, Bsum, Amean, **kw)[1]
                        for u in sample])
        excl = [new[2][int(new[1][u]):int(new[1][u + 1])] for u in sample] if name == "own" else None
        incl = [iix[int(iptr[u]):int(iptr[u + 1])] for u in sample] if name == "include" else None
        for j, (o_ids, sep) in enumerate(_oracle_ids_outside_ties(dtype, A_o, B, n_top, excl, incl)):
            assert np.array_equal(ids[sample[j]][sep], o_ids[sep]), (name, int(sample[j]))


# ---------------------------------------------------------------- 3. resident fit
@pytest.mark.parametrize("dtype", DTYPES)
def test_resident_fit(dtype):
    from poismf_b200 import _lib, c_funs
    from poismf_b200.device import DeviceFit
    csr, csc, A0, B0, k = problem("pl2k", dtype)
    dimA, dimB = A0.shape[0], B0.shape[0]
    sweep = _lib.make_params("cg", l2_reg=1e3, maxupd=5, numiter=2, limit_step=True)
    fits = []
    for _ in range(2):
        f = DeviceFit(dimA, dimB, k, dtype)
        f.set_factors(A0, B0)
        f.set_csr_csc(csr, csc)
        f.sweeps(sweep)
        fits.append(f)
    fit, twin = fits
    A, B = fit.get_factors()
    # fit_stats within the worst-case bound of a float sum of n terms: (n + 1) eps sum|x| (+ eps |mean| for the division)
    eps = np.finfo(dtype).eps
    Bsum, Amean = fit.fit_stats(l1_reg=0.25)
    B64, A64 = B.astype(np.float64), A.astype(np.float64)
    assert (np.abs(Bsum - (B64.sum(0) + 0.25)) <= (dimB + 2) * eps * (np.abs(B64).sum(0) + 0.25)).all()
    assert (np.abs(Amean - A64.mean(0)) <= (dimA + 2) * eps * np.abs(A64).mean(0)).all()
    assert all(np.array_equal(x, y) for x, y in zip(fit.fit_stats(0.25), (Bsum, Amean)))     # reproducible
    # a batch of new users: the computed statistics, the explicit ones and the host-array call agree bitwise
    new, _, _, _ = _synthetic(dtype, 300, dimB, k, 4, lo=1, hi=40)
    kw = dict(top_n=8, output_score=True, return_factors=True, l2_reg=1e3, excl_ptr=new[1], excl_ix=new[2])
    got = fit.topN_new(new[1], new[2], new[0], l1_reg=0.25, **kw)
    explicit = fit.topN_new(new[1], new[2], new[0], Bsum=Bsum, Amean=Amean, **kw)
    host = c_funs._topN_new_batch(new[1], new[2], new[0], B, Bsum, Amean, **kw)
    for x, y, z in zip(got, explicit, host):
        assert np.array_equal(x, y) and np.array_equal(x, z)
    # transform against the resident fit (fold-in only) = the host-array fold-in
    T = fit.transform(new[1], new[2], new[0], l2_reg=1e3, Bsum=Bsum, Amean=Amean)
    assert np.array_equal(T, c_funs._predict_factors_multiple(B, Bsum, Amean, new[1], new[2], new[0], l2_reg=1e3))
    # the handle is untouched: same factors, and a further sweep matches the twin that never served a call
    A2, B2 = fit.get_factors()
    assert np.array_equal(A2, A) and np.array_equal(B2, B)
    fit.sweeps(sweep)
    twin.sweeps(sweep)
    for x, y in zip(fit.get_factors(), twin.get_factors()):
        assert np.array_equal(x, y)
    with pytest.raises(ValueError):
        fit.topN_new(new[1], new[2], new[0], incl_ptr=new[1], incl_ix=new[2], excl_ptr=new[1], excl_ix=new[2])


# ---------------------------------------------------------------- 4. transform
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("case", list(FM_CASES))
def test_transform_equals_factors_multiple(dtype, case):
    from poismf_b200 import c_funs
    from poismf_b200.device import DeviceFit
    for prob in ("readme", "pl2k"):
        csr, B, Bsum, Amean, k = fm_problem(prob, dtype)
        method, kw = fm_hyper(case, k)
        fit = DeviceFit(3, B.shape[0], k, dtype)
        fit.set_factors(np.ascontiguousarray(np.tile(Amean, (3, 1))), B)
        for flags in (0, STRICT):
            got = fit.transform(csr[1], csr[2], csr[0], method=method, Bsum=Bsum, Amean=Amean, flags=flags, **kw)
            ref = c_funs._predict_factors_multiple(B, Bsum, Amean, csr[1], csr[2], csr[0], method=method, flags=flags,
                                                   **kw)
            assert np.array_equal(got, ref), (prob, flags)


# ---------------------------------------------------------------- 5. edges
@pytest.mark.parametrize("k", [1, 64, 128, 200])
def test_shapes_and_index_widths(k):
    from poismf_b200 import _lib, c_funs
    dtype = np.float32
    new, B, Bsum, Amean = _synthetic(dtype, 300, 5000, k, 10 + k)
    n_top = 20
    kw = dict(top_n=n_top, output_score=True, return_factors=True, l2_reg=1e3, excl_ptr=new[1], excl_ix=new[2])
    _lib.topn_stats(reset=True)
    ids, sc, A = c_funs._topN_new_batch(new[1], new[2], new[0], B, Bsum, Amean, **kw)
    tc, _ = _lib.topn_stats(reset=True)
    assert tc == (300 if k <= 128 else 0)                           # k = 200 takes the exact route
    ref = c_funs._topN_batch(A, B, top_n=n_top, output_score=True, excl_ptr=new[1], excl_ix=new[2])
    assert np.array_equal(ids, ref[0]) and np.array_equal(sc, ref[1])
    for r in (0, 1, 299):
        assert np.array_equal(A[r], c_funs._predict_factors(*fs_row(new, r), B, Bsum, Amean, l2_reg=1e3))
    # int32 indices (R's sparse_ix = int): the same users, the same bits
    i32 = dict(kw, excl_ptr=new[1].astype(np.int32), excl_ix=new[2].astype(np.int32))
    ids4, sc4, A4 = c_funs._topN_new_batch(new[1].astype(np.int32), new[2].astype(np.int32), new[0], B, Bsum, Amean,
                                           **i32)
    assert ids4.dtype == np.int32
    assert np.array_equal(ids4.astype(np.uint64), ids) and np.array_equal(sc4, sc) and np.array_equal(A4, A)


def test_include_lists_cross_chunk_seam():
    """More than 32 768 new users with include lists: users on both sides of the ranking's chunk seam are right."""
    from poismf_b200 import c_funs
    dtype = np.float32
    n_new, n, k, n_top = 33_000, 3000, 8, 5
    new, B, Bsum, Amean = _synthetic(dtype, n_new, n, k, 12, lo=1, hi=4)
    rng = np.random.default_rng(13)
    ilens = rng.integers(n_top, 30, n_new)
    iptr = np.concatenate([[0], np.cumsum(ilens)]).astype(np.uint64)
    iix = np.concatenate([rng.choice(n, int(m), replace=False) for m in ilens]).astype(np.uint64)
    ids, sc, A = c_funs._topN_new_batch(new[1], new[2], new[0], B, Bsum, Amean, top_n=n_top, output_score=True,
                                        incl_ptr=iptr, incl_ix=iix, return_factors=True, l2_reg=1e3)
    ref = c_funs._topN_batch(A, B, top_n=n_top, output_score=True, incl_ptr=iptr, incl_ix=iix)
    assert np.array_equal(ids, ref[0]) and np.array_equal(sc, ref[1])
    for r in (0, 32_767, 32_768, n_new - 1):
        assert np.array_equal(A[r], c_funs._predict_factors(*fs_row(new, r), B, Bsum, Amean, l2_reg=1e3))
        assert set(ids[r]) <= set(iix[int(iptr[r]):int(iptr[r + 1])])


@pytest.mark.parametrize("dtype", DTYPES)
def test_single_user_and_exact_exclusions(dtype):
    from poismf_b200 import c_funs
    new, B, Bsum, Amean = _synthetic(dtype, 2, 300, 16, 14)
    c, ix = fs_row(new, 0)
    one = (new[0][:len(c)], new[1][:2], new[2][:len(c)])
    ids, sc, A = c_funs._topN_new_batch(one[1], one[2], one[0], B, Bsum, Amean, top_n=10, output_score=True,
                                        return_factors=True)
    a = c_funs._predict_factors(c, ix, B, Bsum, Amean)
    assert np.array_equal(A[0], a)
    r_ids, r_sc = c_funs._call_topN(a, B, np.empty(0, np.uint64), np.empty(0, np.uint64), top_n=10, output_score=True)
    assert np.array_equal(ids[0], r_ids) and np.array_equal(sc[0], r_sc)
    # exclusions that leave exactly n_top items: those items come back, best first
    n_top, keep = 6, np.array([3, 17, 44, 101, 200, 299], np.uint64)
    excl = np.setdiff1d(np.arange(300, dtype=np.uint64), keep)
    ids, sc = c_funs._topN_new_batch(one[1], one[2], one[0], B, Bsum, Amean, top_n=n_top, output_score=True,
                                     excl_ptr=np.array([0, excl.shape[0]], np.uint64), excl_ix=excl)
    assert set(ids[0]) == set(keep) and (np.diff(sc[0].astype(np.float64)) <= 0).all()


# ---------------------------------------------------------------- 6. invalid arguments
def _raw(new, B, Bsum, Amean, params, n_top, lists=(None,) * 4, outputs=True, A_out=True, n=None):
    """pmf_b200_topN_new_batch through the C ABI with pre-filled outputs: (rc, outputs untouched)."""
    from poismf_b200 import _lib
    n_new = new[1].shape[0] - 1
    ids = np.full((n_new, max(n_top, 1)), 7, np.uint64)
    sc = np.full((n_new, max(n_top, 1)), -1.0, B.dtype)
    A = np.full((n_new, B.shape[1]), -2.0, B.dtype)
    rc = _lib.lib().pmf_b200_topN_new_batch(
        _lib.dtype_code(B.dtype), 8, _lib.ptr(B), _lib.ptr(Bsum), _lib.ptr(Amean), B.shape[1],
        B.shape[0] if n is None else n, _lib.ptr(new[0]), _lib.ptr(new[1]), _lib.ptr(new[2]), n_new, C.byref(params),
        *map(_lib.ptr, lists), _lib.ptr(ids) if outputs else None, _lib.ptr(sc) if outputs else None, n_top,
        _lib.ptr(A) if A_out else None)
    return rc, bool((ids == 7).all() and (sc == -1.0).all() and (A == -2.0).all())


def test_invalid_arguments():
    from poismf_b200 import _lib, c_funs
    from poismf_b200.device import DeviceFit
    dtype, n_top = np.float64, 4
    new, B, Bsum, Amean = _synthetic(dtype, 6, 300, 8, 15, lo=2, hi=20)
    n = B.shape[0]
    ok = _lib.make_params("tncg", 1e3, numiter=1, maxupd=20, step_size=0.0, reuse_prev=True)
    assert _raw(new, B, Bsum, Amean, ok, n_top) == (0, False)
    bad_ptr = new[1].copy(); bad_ptr[2], bad_ptr[3] = bad_ptr[3], bad_ptr[2]
    bad_id = new[2].copy(); bad_id[-1] = n
    P = new[1]
    long_excl = (np.array([0, 0, 0, 0, 0, 0, n - n_top + 1], np.uint64), np.arange(n - n_top + 1, dtype=np.uint64))
    out_excl = (P, np.where(np.arange(new[2].shape[0]) == 3, n, new[2]).astype(np.uint64))
    short_incl = (np.array([0, 10, 20, 30, 40, 50, 53], np.uint64), np.arange(53, dtype=np.uint64))
    cases = [dict(new=(new[0], bad_ptr, new[2])),
             dict(new=(new[0], new[1], bad_id)),
             dict(params=_lib.make_params("tncg", 1e3, numiter=1, maxupd=20, step_size=0.0, early_stop=True)),
             dict(params=_lib.Params(1e3, 0.0, 1.0, 0.0, 7, 0, 1, 20, 0, 1, 0)),
             dict(lists=(P, new[2], P, new[2])),
             dict(n_top=0), dict(n_top=n + 1),
             dict(lists=long_excl + (None, None)), dict(lists=out_excl + (None, None)),
             dict(lists=(None, None) + short_incl, n_top=5),
             dict(Bsum=None), dict(Amean=None),
             dict(outputs=False, A_out=False)]
    for c in cases:
        args = dict(new=new, B=B, Bsum=Bsum, Amean=Amean, params=ok, n_top=n_top)
        args.update(c)
        assert _raw(**args) == (2, True), {key: v for key, v in c.items() if key != "new"} or "ptr/id"
    with pytest.raises(ValueError):
        c_funs._topN_new_batch(bad_ptr, new[2], new[0], B, Bsum, Amean)
    with pytest.raises(ValueError):
        c_funs._topN_new_batch(new[1], bad_id, new[0], B, Bsum, Amean)
    with pytest.raises(ValueError):
        c_funs._topN_new_batch(new[1], new[2], new[0], B, Bsum, Amean, top_n=n + 1)
    with pytest.raises(ValueError):
        c_funs._topN_new_batch(new[1], new[2], new[0], B, Bsum, Amean, excl_ptr=P, excl_ix=new[2], incl_ptr=P,
                               incl_ix=new[2])
    fit = DeviceFit(4, n, 8, dtype)
    fit.set_factors(np.ones((4, 8)), B)
    with pytest.raises(ValueError):
        fit.transform(new[1], bad_id, new[0])
    with pytest.raises(ValueError):
        fit.topN_new(bad_ptr, new[2], new[0])


# ---------------------------------------------------------------- 7. the sharded backend
def _backend_case():
    new, B, Bsum, Amean = _synthetic(np.float32, 501, 20_000, 32, 16, lo=1, hi=80)
    A = np.ascontiguousarray(np.random.default_rng(17).gamma(1.0, 0.3, size=(700, 32)).astype(np.float32))
    return new, A, B


def _backend_calls(be):
    new, _, _ = _backend_case()
    top = be.topN_new(new[1], new[2], new[0], top_n=20, output_score=True, return_factors=True, excl_ptr=new[1],
                      excl_ix=new[2], l2_reg=1e3)
    T = be.transform(new[1], new[2], new[0], l2_reg=1e3)
    return top, T


def _single_handle_calls():
    from poismf_b200.device import DeviceFit
    new, A, B = _backend_case()
    fit = DeviceFit(A.shape[0], B.shape[0], 32, np.float32)
    fit.set_factors(A, B)
    top = fit.topN_new(new[1], new[2], new[0], top_n=20, output_score=True, return_factors=True, excl_ptr=new[1],
                       excl_ix=new[2], l2_reg=1e3)
    return top, fit.transform(new[1], new[2], new[0], l2_reg=1e3)


def test_backend_single_gpu():
    from poismf_b200.sharding import GpuBackend
    _, A, B = _backend_case()
    top, T = _backend_calls(GpuBackend(None, None, A, B, 0, 1, 0))
    ref_top, ref_T = _single_handle_calls()
    assert all(np.array_equal(x, y) for x, y in zip(top, ref_top)) and np.array_equal(T, ref_T)


def _two_gpu_worker(rank, world, port, q):
    import torch
    import torch.distributed as dist
    from poismf_b200.sharding import GpuBackend
    torch.cuda.set_device(rank)
    os.environ["POISMF_B200_DEVICE"] = str(rank)
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    _, A, B = _backend_case()
    be = GpuBackend(None, None, A, B, rank, world, rank)
    q.put((rank,) + _backend_calls(be))
    dist.barrier()
    be.finish()
    dist.destroy_process_group()


def test_two_gpu_new_users_match_single_gpu():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_two_gpu_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=300) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    ref_top, ref_T = _single_handle_calls()
    for _, top, T in res:
        assert all(np.array_equal(x, y) for x, y in zip(top, ref_top)) and np.array_equal(T, ref_T)
