"""CPU tests of the sharding layer's predict path: predict_sharded splits the pairs into contiguous ranges, two gloo
ranks (a numpy dot as the stand-in predictor) return what one rank returns, with and without gathering, and an id
out of range in one rank's share makes both ranks raise instead of leaving one waiting in the gather."""
import socket

import numpy as np
import pytest


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    return port


def _problem():
    rng = np.random.default_rng(13)
    A = rng.standard_normal((37, 6))
    B = rng.standard_normal((53, 6))
    n = 1001
    return A, B, rng.integers(0, 37, n).astype(np.uint64), rng.integers(0, 53, n).astype(np.uint64)


def _numpy_predictor(A, B, seen):
    """Stand-in for DeviceFit.predict: ValueError on an id out of range, like the device call."""
    def predict(u, i):
        seen.append((u, i))
        if (u >= A.shape[0]).any() or (i >= B.shape[0]).any():
            raise ValueError("predict_fitted: an id is outside [0, dimA) / [0, dimB)")
        return np.einsum("ij,ij->i", A[u.astype(np.int64)], B[i.astype(np.int64)])
    return predict


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    from poismf_b200.sharding import predict_sharded, user_ranges
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    A, B, u, i = _problem()
    lo, hi = user_ranges(u.shape[0], world)[rank]
    seen = []
    got = predict_sharded(u, i, _numpy_predictor(A, B, seen), rank, world)
    one = predict_sharded(u, i, _numpy_predictor(A, B, []))
    mine = predict_sharded(u, i, _numpy_predictor(A, B, []), rank, world, gather=False)
    ok = np.array_equal(got, one) and got.shape == (u.shape[0],)
    ok &= np.array_equal(mine, one[lo:hi])
    ok &= np.array_equal(seen[0][0], u[lo:hi]) and np.array_equal(seen[0][1], i[lo:hi])
    # a bad id in the last rank's range only, then in the first rank's: every rank raises, with and without gather
    raised = []
    for which, pos in (("u", u.shape[0] - 1), ("i", 0)):
        for gather in (True, False):
            uu, ii = u.copy(), i.copy()
            (uu if which == "u" else ii)[pos] = 10 ** 6
            try:
                predict_sharded(uu, ii, _numpy_predictor(A, B, []), rank, world, gather=gather)
                raised.append(False)
            except ValueError:
                raised.append(True)
    # the group is still usable afterwards
    again = predict_sharded(u, i, _numpy_predictor(A, B, []), rank, world)
    ok &= np.array_equal(again, one)
    q.put((rank, bool(ok), raised))
    dist.destroy_process_group()


def test_predict_sharding_gloo_world2():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    try:
        res = [q.get(timeout=240) for _ in procs]
    finally:
        for p in procs:
            p.join(timeout=60)
        hung = [p.pid for p in procs if p.is_alive()]
        for p in procs:
            if p.is_alive():
                p.kill()
    assert not hung, f"ranks still running: {hung}"
    assert all(ok for _, ok, _ in res), res
    assert all(all(r) for _, _, r in res), res


def test_predict_sharded_checks_shapes():
    from poismf_b200.sharding import predict_sharded
    u = np.arange(4, dtype=np.uint64)
    with pytest.raises(ValueError):
        predict_sharded(u, u[:3], lambda a, b: None)
    with pytest.raises(ValueError):
        predict_sharded(u, u, _numpy_predictor(np.ones((2, 1)), np.ones((5, 1)), []))
