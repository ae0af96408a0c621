"""Batched top-N over per-user candidate lists (pmf_b200_topN_batch_include / _fitted_include): every user's
ids and scores equal the oracle's topN(include=list) bit for bit, ties included (both break them by ascending
item id), on both ranking paths (shared memory for lists up to 16 K items in f32 / 8 K in f64, segmented
radix sort above)."""
import os
import socket

import numpy as np
import pytest

from conftest import problem
from oracle.oracle import Restatement

pytestmark = pytest.mark.gpu
DTYPES = [np.float64, np.float32]


def _lists(rng, n, lens):
    return [rng.choice(n, int(m), replace=False) for m in lens]


def _csr(lists):
    ptr = np.concatenate([[0], np.cumsum([len(x) for x in lists])]).astype(np.uint64)
    return ptr, np.concatenate(lists).astype(np.uint64)


def _oracle_topn(dtype, A, B, users, lists, n_top):
    orc = Restatement(dtype)
    ids = np.empty((len(lists), n_top), np.uint64)
    sc = np.empty((len(lists), n_top), dtype)
    for r, (u, lst) in enumerate(zip(users, lists)):
        rc, ids[r], sc[r] = orc.topN(np.ascontiguousarray(A[int(u)]), B, n_top, include=lst)
        assert rc == 0
    return ids, sc


def _call_int32(A, B, users, ptr, ix, n_top, out_ix=None, out_sc=None):
    """The 4-byte index variant (R's sparse_ix = int) through the C ABI directly."""
    from poismf_b200 import _lib
    u = np.ascontiguousarray(users, np.int32)
    p = np.ascontiguousarray(ptr, np.int32)
    i = np.ascontiguousarray(ix, np.int32)
    out_ix = np.empty((u.shape[0], n_top), np.int32) if out_ix is None else out_ix
    out_sc = np.empty((u.shape[0], n_top), B.dtype) if out_sc is None else out_sc
    rc = _lib.lib().pmf_b200_topN_batch_include(_lib.dtype_code(B.dtype), 4, _lib.ptr(A), _lib.ptr(B), B.shape[1],
                                                _lib.ptr(u), u.shape[0], A.shape[0], _lib.ptr(p), _lib.ptr(i),
                                                _lib.ptr(out_ix), _lib.ptr(out_sc), n_top, B.shape[0])
    return rc, out_ix, out_sc


def _parity_case(dtype):
    rng = np.random.default_rng(11)
    n, k, n_top, n_users = 20_000, 24, 7, 60
    A = np.ascontiguousarray(rng.gamma(1.0, 0.5, size=(n_users, k)).astype(dtype))
    B = rng.gamma(1.0, 0.5, size=(n, k))
    B[1000:1040] = 2.0 * B.max(axis=0)     # 40 tied rows that score above every other item
    B[1040:1060] = B[18]                   # 20 tied rows with ordinary scores
    B = np.ascontiguousarray(B.astype(dtype))
    lens = [n_top, n_top + 1, 10, 12, 40, 150, 300, 700, 1000, 8192, 8193, 9000, 16384, 16385, 17_000, n]
    lens += list(rng.integers(n_top, 1200, n_users - len(lens) - 5))
    lists = _lists(rng, n, lens)
    # duplicates, ranked as given: repeats of top-scoring rows, so that they come out twice
    x = rng.choice(np.arange(2000, n), 50, replace=False)
    lists.append(rng.permutation(np.concatenate([x, x[:20], [1003, 1003, 1005]])))
    lists.append(rng.permutation(np.concatenate([np.arange(2000, 19_000), [1001, 1001, 1002, 1002, 1002]])))  # long path
    lists.append(np.concatenate([np.arange(1000, 1040), rng.choice(n, 20)]))      # ties at the top
    lists.append(rng.permutation(np.arange(1040, 1060)))                          # nothing but ties
    lists.append(rng.permutation(np.arange(1000, 17_500)))                        # ties at the top, long path
    users = rng.permutation(n_users)[:len(lists)].astype(np.uint64)
    return A, B, users, lists, n_top


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("index_bytes", [8, 4])
def test_include_matches_oracle(dtype, index_bytes):
    from poismf_b200 import c_funs
    A, B, users, lists, n_top = _parity_case(dtype)
    ptr, ix = _csr(lists)
    if index_bytes == 8:
        ids, sc = c_funs._topN_batch(A, B, users=users, incl_ptr=ptr, incl_ix=ix, top_n=n_top, output_score=True)
    else:
        rc, ids, sc = _call_int32(A, B, users, ptr, ix, n_top)
        assert rc == 0
    o_ids, o_sc = _oracle_topn(dtype, A, B, users, lists, n_top)
    for r in range(len(lists)):
        assert np.array_equal(ids[r].astype(np.uint64), o_ids[r]) and np.array_equal(sc[r], o_sc[r]), (r, len(lists[r]))
    # the tie cases did tie, the duplicates came out twice
    assert all((o_sc[r] == o_sc[r][0]).all() for r in (-3, -2, -1))
    assert list(o_ids[-5][:3]) == [1003, 1003, 1005] and list(o_ids[-4][:5]) == [1001, 1001, 1002, 1002, 1002]


@pytest.mark.parametrize("dtype", DTYPES)
def test_include_against_resident_factors(dtype):
    from poismf_b200 import _lib, c_funs
    from poismf_b200.device import DeviceFit
    csr, csc, A0, B0, k = problem("pl2k", dtype)
    rng = np.random.default_rng(3)
    dimA, dimB = A0.shape[0], B0.shape[0]
    users = rng.choice(dimA, 50, replace=False).astype(np.uint64)
    lens = np.concatenate([[5], rng.integers(5, 300, users.shape[0] - 2), [dimB]])
    ptr, ix = _csr(_lists(rng, dimB, lens))
    fit = DeviceFit(dimA, dimB, k, dtype)
    fit.set_factors(A0, B0)
    got = fit.topN(users=users, incl_ptr=ptr, incl_ix=ix, top_n=5, output_score=True)
    ref = c_funs._topN_batch(A0, B0, users=users, incl_ptr=ptr, incl_ix=ix, top_n=5, output_score=True)
    assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1])
    with pytest.raises(ValueError):
        fit.topN(users=users, incl_ptr=ptr, incl_ix=ix, excl_ptr=ptr, excl_ix=ix, top_n=5)
    with pytest.raises(ValueError):
        fit.topN(users=users, incl_ptr=ptr, incl_ix=ix, top_n=6)          # a list of 5 items
    fit.set_matrix(_lib.SIDE_CSR, *csr)
    fit.set_matrix(_lib.SIDE_CSC, *csc)
    fit.sweeps(_lib.make_params("cg", l2_reg=1e3, maxupd=5, numiter=2, limit_step=True))
    A, B = fit.get_factors()
    got = fit.topN(users=users, incl_ptr=ptr, incl_ix=ix, top_n=5, output_score=True)
    ref = c_funs._topN_batch(A, B, users=users, incl_ptr=ptr, incl_ix=ix, top_n=5, output_score=True)
    assert not np.array_equal(A, A0)
    assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1])


@pytest.mark.parametrize("dtype,k,signed", [(np.float32, 5, False), (np.float32, 64, False), (np.float32, 128, False),
                                            (np.float32, 200, False), (np.float64, 50, False),
                                            (np.float32, 64, True), (np.float64, 50, True)])
def test_include_shapes(dtype, k, signed):
    from poismf_b200 import c_funs
    rng = np.random.default_rng(k + 7 * signed)
    n, n_users, n_top = 12_000, 24, 10
    if signed:
        A = rng.normal(size=(n_users, k)); B = rng.normal(size=(n, k))
    else:
        A = rng.gamma(1.0, 0.5, size=(n_users, k)); B = rng.gamma(1.0, 0.5, size=(n, k))
    A = np.ascontiguousarray(A.astype(dtype)); B = np.ascontiguousarray(B.astype(dtype))
    lens = np.concatenate([[n_top], rng.integers(n_top, 2000, n_users - 3), [9000, n]])   # [n_top]: every score shows
    lists = _lists(rng, n, lens)
    ptr, ix = _csr(lists)
    users = np.arange(n_users, dtype=np.uint64)
    ids, sc = c_funs._topN_batch(A, B, incl_ptr=ptr, incl_ix=ix, top_n=n_top, output_score=True)
    o_ids, o_sc = _oracle_topn(dtype, A, B, users, lists, n_top)
    assert np.array_equal(ids, o_ids) and np.array_equal(sc, o_sc)
    if signed:
        assert (o_sc < 0).any()


def test_include_crosses_chunk_boundary():
    """More than 32 768 users: the call runs in chunks; users on both sides of every seam equal the oracle."""
    from poismf_b200 import c_funs
    rng = np.random.default_rng(21)
    n_users, n, k, n_top = 70_000, 5000, 8, 5
    A = np.ascontiguousarray(rng.gamma(1.0, 0.5, size=(n_users, k)).astype(np.float32))
    B = np.ascontiguousarray(rng.gamma(1.0, 0.5, size=(n, k)).astype(np.float32))
    lens = rng.integers(n_top, 40, n_users)
    ptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    ix = np.concatenate([rng.choice(n, int(m), replace=False) for m in lens]).astype(np.uint64)
    users = rng.permutation(n_users).astype(np.uint64)
    ids, sc = c_funs._topN_batch(A, B, users=users, incl_ptr=ptr, incl_ix=ix, top_n=n_top, output_score=True)
    rows = np.unique(np.concatenate([np.arange(32_760, 32_776), np.arange(65_530, 65_545), [0, n_users - 1],
                                     rng.choice(n_users, 100, replace=False)]))
    lists = [ix[int(ptr[r]):int(ptr[r + 1])] for r in rows]
    o_ids, o_sc = _oracle_topn(np.float32, A, B, users[rows], lists, n_top)
    assert np.array_equal(ids[rows], o_ids) and np.array_equal(sc[rows], o_sc)


def test_include_invalid_arguments():
    from poismf_b200 import c_funs
    rng = np.random.default_rng(5)
    n_users, n, k, n_top = 6, 300, 8, 4
    A = np.ascontiguousarray(rng.gamma(1.0, 0.5, size=(n_users, k)))
    B = np.ascontiguousarray(rng.gamma(1.0, 0.5, size=(n, k)))
    lists = _lists(rng, n, [10, 20, 4, 30, 50, 9])
    ptr, ix = _csr(lists)
    users = np.arange(n_users, dtype=np.uint64)
    long_ptr, long_ix = _csr(lists[:-1] + [np.concatenate([np.arange(n), [0]])])       # n + 1 items
    short_ptr, short_ix = _csr(lists[:-1] + [lists[-1][:3]])                           # fewer than n_top
    bad_ix = ix.copy(); bad_ix[-1] = n                                                 # an id >= n
    bad_ptr = ptr.copy(); bad_ptr[3], bad_ptr[4] = bad_ptr[4], bad_ptr[3]              # not monotone
    cases = [dict(incl_ptr=ptr, incl_ix=ix, top_n=0),
             dict(incl_ptr=ptr, incl_ix=ix, top_n=n_top, users=np.array([0, 1, 2, 3, 4, n_users], np.uint64)),
             dict(incl_ptr=bad_ptr, incl_ix=ix, top_n=n_top),
             dict(incl_ptr=long_ptr, incl_ix=long_ix, top_n=n_top),
             dict(incl_ptr=short_ptr, incl_ix=short_ix, top_n=n_top),
             dict(incl_ptr=ptr, incl_ix=bad_ix, top_n=n_top),
             dict(incl_ptr=ptr, incl_ix=ix, excl_ptr=ptr, excl_ix=ix, top_n=n_top)]
    for kw in cases:
        kw.setdefault("users", users)
        with pytest.raises(ValueError):
            c_funs._topN_batch(A, B, output_score=True, **kw)
    # rc 2 leaves pre-filled outputs untouched, also when the bad id sits in the last of several chunks
    neg_ptr = ptr.astype(np.int32) - 1; neg_ptr[1:] = ptr[1:].astype(np.int32)                # starts before incl_ix
    for p, i in ((bad_ptr, ix), (ptr, bad_ix), (short_ptr, short_ix), (neg_ptr, ix)):
        out_ix = np.full((n_users, n_top), 7, np.int32); out_sc = np.full((n_users, n_top), -1.0)
        rc, _, _ = _call_int32(A, B, users, p, i, n_top, out_ix, out_sc)
        assert rc == 2 and (out_ix == 7).all() and (out_sc == -1.0).all()
    m = 40_000
    Am = np.ascontiguousarray(np.tile(A[:1], (m, 1)))
    mp_, mi = _csr([np.arange(n_top, dtype=np.uint64)] * m)
    mi[-1] = n
    out_ix = np.full((m, n_top), 7, np.int32); out_sc = np.full((m, n_top), -1.0)
    rc, _, _ = _call_int32(Am, B, np.arange(m), mp_, mi, n_top, out_ix, out_sc)
    assert rc == 2 and (out_ix == 7).all() and (out_sc == -1.0).all()


def _two_gpu_include_worker(rank, world, port, q):
    import torch
    import torch.distributed as dist
    from poismf_b200.sharding import topn_sharded
    torch.cuda.set_device(rank)
    os.environ["POISMF_B200_DEVICE"] = str(rank)
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    A, B, ptr, ix = _sharded_case()
    ids, sc = topn_sharded(A, B, 20, incl_ptr=ptr, incl_ix=ix, output_score=True, rank=rank, world=world)
    q.put((rank, ids, sc))
    dist.barrier()
    dist.destroy_process_group()


def _sharded_case():
    rng = np.random.default_rng(31)
    A = np.ascontiguousarray(rng.gamma(0.5, 0.5, size=(301, 32)).astype(np.float32))
    B = np.ascontiguousarray(rng.gamma(0.5, 0.5, size=(20_000, 32)).astype(np.float32))
    lens = np.concatenate([rng.integers(20, 1000, A.shape[0] - 1), [18_000]])
    ptr, ix = _csr(_lists(rng, B.shape[0], lens))
    return A, B, ptr, ix


def test_backend_topn_include_single_gpu():
    """GpuBackend.topN with include lists ranks against the backend's resident replicas (world 1)."""
    from poismf_b200 import c_funs
    from poismf_b200.sharding import GpuBackend
    A, B, ptr, ix = _sharded_case()
    be = GpuBackend(None, None, A, B, 0, 1, 0)
    ids, sc = be.topN(20, incl_ptr=ptr, incl_ix=ix, output_score=True)
    ref = c_funs._topN_batch(A, B, incl_ptr=ptr, incl_ix=ix, top_n=20, output_score=True)
    assert np.array_equal(ids, ref[0]) and np.array_equal(sc, ref[1])
    users = np.arange(0, A.shape[0], 3, dtype=np.uint64)
    sub = [ix[int(ptr[u]):int(ptr[u + 1])] for u in users]
    sp, si = _csr(sub)
    ids, _ = be.topN(20, users=users, incl_ptr=sp, incl_ix=si)
    assert np.array_equal(ids, ref[0][users.astype(np.int64)])
    with pytest.raises(ValueError):
        be.topN(20, incl_ptr=ptr, incl_ix=ix, excl_ptr=ptr, excl_ix=ix)


def test_two_gpu_user_sharded_include_matches_single_gpu():
    import torch
    from poismf_b200 import c_funs
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_two_gpu_include_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=300) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    A, B, ptr, ix = _sharded_case()
    ids, sc = c_funs._topN_batch(A, B, incl_ptr=ptr, incl_ix=ix, top_n=20, output_score=True)
    for _, i2, s2 in res:
        assert np.array_equal(i2, ids) and np.array_equal(s2, sc)
