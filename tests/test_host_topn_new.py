"""CPU tests of the sharding layer's new-user path: new_users_sharded slices each rank's CSR rows and per-user lists
by user range, and two gloo ranks (the oracle's factors_single + topN as the stand-in fold-in) return what one rank
returns, with and without gathering."""
import socket

import numpy as np
import pytest


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    return port


def _problem():
    rng = np.random.default_rng(9)
    n_new, n_items, k, n_top = 23, 400, 5, 7
    B = rng.gamma(1, 1, size=(n_items, k))
    Bsum = B.sum(0) + 0.2
    Amean = rng.gamma(1, 0.3, size=k)
    lens = rng.integers(0, 30, n_new)
    lens[4] = 0
    ptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    ind = np.concatenate([np.sort(rng.choice(n_items, int(m), replace=False)) for m in lens]).astype(np.uint64)
    vals = rng.integers(1, 5, ind.shape[0]).astype(np.float64)
    ilens = rng.integers(n_top, 60, n_new)
    iptr = np.concatenate([[0], np.cumsum(ilens)]).astype(np.uint64)
    iix = np.concatenate([rng.choice(n_items, int(m), replace=False) for m in ilens]).astype(np.uint64)
    return (vals, ptr, ind), B, Bsum, Amean, n_top, (iptr, iix)


def _oracle_fold(B, Bsum, Amean, n_top, seen):
    """Stand-in fold-in-and-rank callable: the oracle row by row.  `seen` records the slices it was given."""
    from oracle.oracle import Restatement
    orc = Restatement(np.float64)

    def fold(csr, p_, i_, include):
        vals, ptr, ind = csr
        seen.append((csr, p_, i_, include))
        n = ptr.shape[0] - 1
        ids = np.empty((n, n_top), np.uint64); sc = np.empty((n, n_top)); A = np.empty((n, B.shape[1]))
        for u in range(n):
            lo, hi = int(ptr[u]), int(ptr[u + 1])
            A[u] = orc.factors_single(np.ascontiguousarray(vals[lo:hi]), np.ascontiguousarray(ind[lo:hi]), B, Bsum,
                                      Amean, l2_reg=1e3, maxupd=20)[1]
            lst = None if p_ is None else i_[int(p_[u]):int(p_[u + 1])]
            kw = {} if lst is None else ({"include": lst} if include else {"exclude": lst})
            rc, ids[u], sc[u] = orc.topN(np.ascontiguousarray(A[u]), B, n_top, **kw)
            assert rc == 0
        return ids, sc, A
    return fold


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    from poismf_b200.sharding import new_users_sharded, user_ranges
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    csr, B, Bsum, Amean, n_top, (iptr, iix) = _problem()
    vals, ptr, ind = csr
    n_new = ptr.shape[0] - 1
    lo, hi = user_ranges(n_new, world)[rank]
    ok = True
    for lists in ({}, dict(excl_ptr=ptr, excl_ix=ind), dict(incl_ptr=iptr, incl_ix=iix)):
        seen, seen1 = [], []
        got = new_users_sharded(csr, _oracle_fold(B, Bsum, Amean, n_top, seen), rank, world, **lists)
        one = new_users_sharded(csr, _oracle_fold(B, Bsum, Amean, n_top, seen1), **lists)
        mine = new_users_sharded(csr, _oracle_fold(B, Bsum, Amean, n_top, []), rank, world, gather=False, **lists)
        ok &= all(np.array_equal(g, o) for g, o in zip(got, one)) and got[0].shape == (n_new, n_top)
        ok &= all(np.array_equal(m, o[lo:hi]) for m, o in zip(mine, one))
        # the rank's slices: its CSR rows rebased to 0, its users' lists rebased to 0
        (v, p, i), p_, i_, include = seen[0]
        a, b = int(ptr[lo]), int(ptr[hi])
        ok &= np.array_equal(p, ptr[lo:hi + 1] - ptr[lo]) and np.array_equal(i, ind[a:b]) and np.array_equal(v, vals[a:b])
        ok &= include == ("incl_ptr" in lists)
        if lists:
            lp, li = (iptr, iix) if include else (ptr, ind)
            ok &= np.array_equal(p_, lp[lo:hi + 1] - lp[lo]) and np.array_equal(i_, li[int(lp[lo]):int(lp[hi])])
        else:
            ok &= p_ is None and i_ is None
    # own items excluded: none of a user's interactions is ranked
    ids = new_users_sharded(csr, _oracle_fold(B, Bsum, Amean, n_top, []), rank, world, excl_ptr=ptr, excl_ix=ind)[0]
    ok &= all(not np.isin(ids[u], ind[int(ptr[u]):int(ptr[u + 1])]).any() for u in range(n_new))
    q.put((rank, bool(ok)))
    dist.destroy_process_group()


def test_new_users_sharding_gloo_world2():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=240) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert all(ok for _, ok in res), res


def test_new_users_sharded_rejects_include_with_exclude():
    from poismf_b200.sharding import new_users_sharded
    csr = (np.ones(2), np.array([0, 1, 2], np.uint64), np.array([0, 1], np.uint64))
    p = np.array([0, 1, 2], np.uint64); i = np.array([0, 1], np.uint64)
    with pytest.raises(ValueError):
        new_users_sharded(csr, lambda *a: None, incl_ptr=p, incl_ix=i, excl_ptr=p, excl_ix=i)
