"""CPU test of the sharding layer's include lists: topn_sharded slices each user range's candidate lists like
the exclusion lists, and two gloo ranks (the oracle as the stand-in scorer) return what one rank returns."""
import socket

import numpy as np


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    return port


def _gloo_include_worker(rank, world, port, q):
    import torch.distributed as dist
    from oracle.oracle import Restatement
    from poismf_b200.sharding import topn_sharded, user_ranges
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    rng = np.random.default_rng(6)
    n_users, n_items, k, n_top = 37, 500, 6, 9
    A = rng.gamma(1, 1, size=(n_users, k)); B = rng.gamma(1, 1, size=(n_items, k))
    users = rng.permutation(n_users)[:30].astype(np.uint64)
    lens = rng.integers(n_top, 120, users.shape[0])
    ptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    iix = np.concatenate([rng.choice(n_items, int(m), replace=False) for m in lens]).astype(np.uint64)
    orc = Restatement(np.float64)

    def cpu_scorer(A_, B_, u_, p_, i_, n_, s_, include=False):     # test infrastructure: the oracle, user by user
        assert include
        ids = np.empty((u_.shape[0], n_), np.uint64); sc = np.empty((u_.shape[0], n_))
        for j, usr in enumerate(u_):
            lst = i_[int(p_[j]):int(p_[j + 1])]
            _, ids[j], sc[j] = orc.topN(np.ascontiguousarray(A_[int(usr)]), B_, n_, include=lst)
        return ids, sc

    kw = dict(users=users, incl_ptr=ptr, incl_ix=iix, output_score=True, scorer=cpu_scorer)
    ids, sc = topn_sharded(A, B, n_top, rank=rank, world=world, **kw)
    ids1, sc1 = topn_sharded(A, B, n_top, **kw)
    ids_l, sc_l = topn_sharded(A, B, n_top, rank=rank, world=world, gather=False, **kw)
    lo, hi = user_ranges(users.shape[0], world)[rank]
    # every row equals the oracle on the user's own list
    direct = all(np.array_equal(ids1[r], orc.topN(np.ascontiguousarray(A[int(users[r])]), B, n_top,
                                                  include=iix[int(ptr[r]):int(ptr[r + 1])])[1]) for r in range(30))
    ok = (np.array_equal(ids, ids1) and np.array_equal(sc, sc1) and ids.shape == (30, n_top) and direct and
          np.array_equal(ids_l, ids1[lo:hi]) and np.array_equal(sc_l, sc1[lo:hi]))
    q.put((rank, bool(ok)))
    dist.destroy_process_group()


def test_topn_include_user_sharding_gloo_world2():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_gloo_include_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=240) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert all(ok for _, ok in res), res


def test_topn_sharded_rejects_include_with_exclude():
    import pytest
    from poismf_b200.sharding import topn_sharded
    A = np.ones((3, 2)); B = np.ones((5, 2))
    p = np.array([0, 1, 2, 3], np.uint64); i = np.array([0, 1, 2], np.uint64)
    with pytest.raises(ValueError):
        topn_sharded(A, B, 1, incl_ptr=p, incl_ix=i, excl_ptr=p, excl_ix=i, scorer=lambda *a, **k: None)
