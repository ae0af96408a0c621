"""Resident-fit scoring and ingestion (pmf_b200_predict_fitted, pmf_b200_set_coo): predict against a handle's factors
is bitwise the stateless predict_multiple on the factors read back (and the oracle's sequential dot), across id widths,
chunk boundaries and signed factors; a bad id leaves `out` and the handle as they were; a matrix built from triplets
in the handle sweeps bitwise like one built by SciPy on the host."""
import os
import socket

import numpy as np
import pytest

from conftest import hyper, problem
from oracle.oracle import Restatement

pytestmark = pytest.mark.gpu
DTYPES = [np.float32, np.float64]
IXDTS = [np.uint64, np.int32]
CHUNK = 1 << 21                      # pairs per upload chunk (PREDICT_CHUNK in csrc/api.cu)


def _bits(x):
    return x.view(np.uint32 if x.dtype == np.float32 else np.uint64)


def _same_bits(x, y):
    return x.dtype == y.dtype and x.shape == y.shape and np.array_equal(_bits(x), _bits(y))


def _stateless(A, B, u, i):
    from poismf_b200 import c_funs
    out = np.empty(u.shape[0], A.dtype)
    c_funs._predict_multiple(out, A, B, u, i)
    return out


def _pairs(rng, dimA, dimB, n, ixdt):
    """n pairs in arbitrary order with repeats; every row of A and of B appears when n allows it."""
    u = rng.integers(0, dimA, n)
    i = rng.integers(0, dimB, n)
    m = min(n, dimA)
    u[:m] = rng.permutation(dimA)[:m]
    m = min(n, dimB)
    i[n - m:] = rng.permutation(dimB)[:m]
    return u.astype(ixdt), i.astype(ixdt)


def _fitted(prob, dtype):
    """A handle holding problem `prob` after one cg sweep."""
    from poismf_b200 import _lib
    from poismf_b200.device import DeviceFit
    csr, csc, A0, B0, k = problem(prob, dtype)
    method, kw = hyper("cg", k)
    fit = DeviceFit(A0.shape[0], B0.shape[0], k, dtype)
    fit.set_csr_csc(csr, csc)
    fit.set_factors(A0, B0)
    fit.sweeps(_lib.make_params(method, **kw))
    return fit


def _signed_factors(dtype, dimA, dimB, k, seed):
    """Signed random factors with all-zero rows and exact zeros of both signs."""
    rng = np.random.default_rng(seed)
    A = rng.standard_normal((dimA, k)).astype(dtype)
    B = rng.standard_normal((dimB, k)).astype(dtype)
    A[::17] = 0.0
    B[3::11] = -0.0
    A[rng.random(A.shape) < 0.05] = -0.0
    B[rng.random(B.shape) < 0.05] = 0.0
    return np.ascontiguousarray(A), np.ascontiguousarray(B)


def _check_parity(fit, u, i):
    A, B = fit.get_factors()
    got = fit.predict(u, i)
    assert got.dtype == fit.dtype and got.shape == u.shape
    assert _same_bits(got, _stateless(A, B, u, i))
    orc = Restatement(fit.dtype).predict_multiple(A, B, u.astype(np.uint64), i.astype(np.uint64))
    assert _same_bits(got, orc)
    return got


# ---------------------------------------------------------------- 1. bitwise parity
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("ixdt", IXDTS)
@pytest.mark.parametrize("prob", ["readme", "ragged", "pl6k"])
def test_predict_equals_stateless_and_oracle(dtype, ixdt, prob):
    fit = _fitted(prob, dtype)
    u, i = _pairs(np.random.default_rng(1), fit.dimA, fit.dimB, 20_000, ixdt)
    _check_parity(fit, u, i)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("ixdt", IXDTS)
@pytest.mark.parametrize("k", [100, 130])
def test_predict_signed_factors(dtype, ixdt, k):
    from poismf_b200.device import DeviceFit
    A, B = _signed_factors(dtype, 900, 1300, k, seed=k)
    fit = DeviceFit(A.shape[0], B.shape[0], k, dtype)
    fit.set_factors(A, B)
    u, i = _pairs(np.random.default_rng(2), 900, 1300, 50_000, ixdt)
    got = _check_parity(fit, u, i)
    assert (np.signbit(got) & (got == 0)).sum() == 0       # a sum that starts at +0 never ends at -0
    assert (got == 0).any() and (got < 0).any()


# ---------------------------------------------------------------- 2. waiting for the sweep
def test_predict_waits_for_sweeps():
    from poismf_b200 import _lib
    from poismf_b200.device import DeviceFit
    csr, csc, A0, B0, k = problem("pl6k", np.float32)
    params = _lib.make_params("cg", l2_reg=1e4, maxupd=5, numiter=3, limit_step=True)
    u, i = _pairs(np.random.default_rng(3), A0.shape[0], B0.shape[0], 100_000, np.uint64)
    outs = []
    for explicit_sync in (False, True):
        fit = DeviceFit(A0.shape[0], B0.shape[0], k, np.float32)
        fit.set_csr_csc(csr, csc)
        fit.set_factors(A0, B0)
        fit.sweeps(params)
        if explicit_sync:
            fit.sync()
        outs.append(fit.predict(u, i))
    assert _same_bits(outs[0], outs[1])
    assert _same_bits(outs[0], _stateless(*fit.get_factors(), u, i))


# ---------------------------------------------------------------- 3. sizes
def _pinned(a):
    import torch
    t = torch.empty(a.shape[0], dtype={np.dtype(np.int32): torch.int32, np.dtype(np.uint64): torch.int64,
                                       np.dtype(np.float32): torch.float32}[a.dtype]).pin_memory()
    view = t.numpy().view(a.dtype)
    view[:] = a
    return t, view


@pytest.mark.parametrize("ixdt", IXDTS)
def test_predict_sizes(ixdt):
    from poismf_b200.device import DeviceFit
    A, B = _signed_factors(np.float32, 3000, 2000, 50, seed=4)
    fit = DeviceFit(3000, 2000, 50, np.float32)
    fit.set_factors(A, B)
    empty = np.empty(0, ixdt)
    assert fit.predict(empty, empty).shape == (0,)
    one = fit.predict(np.array([2999], ixdt), np.array([0], ixdt))
    assert _same_bits(one, _stateless(A, B, np.array([2999], ixdt), np.array([0], ixdt)))
    n = 3 * CHUNK + 4321                                      # four chunks, the last one partial
    u, i = _pairs(np.random.default_rng(5), 3000, 2000, n, ixdt)
    want = _stateless(A, B, u, i)
    assert _same_bits(fit.predict(u, i), want)
    # page-locked ids and output: copied directly instead of staged
    keep = [_pinned(u), _pinned(i), _pinned(np.zeros(n, np.float32))]
    got = fit.predict(keep[0][1], keep[1][1], out=keep[2][1])
    assert got is keep[2][1] and _same_bits(got, want)
    sub = np.random.default_rng(6).choice(n, 20_000, replace=False)
    orc = Restatement(np.float32).predict_multiple(A, B, u[sub].astype(np.uint64), i[sub].astype(np.uint64))
    assert _same_bits(want[sub], orc)


def test_predict_argument_checks():
    from poismf_b200.device import DeviceFit
    fit = DeviceFit(10, 20, 4, np.float64)
    fit.set_factors(np.ones((10, 4)), np.ones((20, 4)))
    u = np.arange(5, dtype=np.uint64)
    with pytest.raises(ValueError):
        fit.predict(u, u[:4])
    with pytest.raises(ValueError):
        fit.predict(u, u.astype(np.int32))
    with pytest.raises(ValueError):
        fit.predict(u, u, out=np.empty(5, np.float32))
    rc = fit.L.pmf_b200_predict_fitted(fit.h, 2, u.ctypes.data, u.ctypes.data, 5, np.empty(5).ctypes.data)
    assert rc == 2


# ---------------------------------------------------------------- 4. bad ids
@pytest.mark.parametrize("ixdt", IXDTS)
def test_predict_bad_ids_leave_out_and_handle_untouched(ixdt):
    from poismf_b200 import _lib
    from poismf_b200.device import DeviceFit
    dtype = np.float32
    csr, csc, A0, B0, k = problem("pl6k", dtype)
    dimA, dimB = A0.shape[0], B0.shape[0]
    params = _lib.make_params("cg", l2_reg=1e4, maxupd=5, numiter=1, limit_step=True)
    fit = DeviceFit(dimA, dimB, k, dtype)
    fit.set_csr_csc(csr, csc)
    fit.set_factors(A0, B0)
    n = 2 * CHUNK + 999
    u, i = _pairs(np.random.default_rng(7), dimA, dimB, n, ixdt)
    bads = [("A", 0, dimA), ("B", n - 1, dimB), ("A", n - 5, dimA + 12345), ("B", 17, 2 ** 31 - 1)]
    if ixdt == np.int32:
        bads += [("A", 3, -1), ("B", n - 2, -7)]
    else:
        bads += [("A", 3, 2 ** 63), ("B", n - 2, 2 ** 64 - 1)]
    sentinel = np.full(n, 0x7fc0dead, np.uint32).view(np.float32)
    for which, pos, val in bads:
        uu, ii = u.copy(), i.copy()
        (uu if which == "A" else ii)[pos] = val
        out = sentinel.copy()
        with pytest.raises(ValueError):
            fit.predict(uu, ii, out=out)
        assert np.array_equal(_bits(out), _bits(sentinel)), (which, pos, val)
    # the handle still predicts correctly and sweeps like a fresh one
    _check_parity(fit, u[:50_000], i[:50_000])
    assert _same_bits(fit.predict(u, i), _stateless(*fit.get_factors(), u, i))
    fit.sweeps(params)
    fresh = DeviceFit(dimA, dimB, k, dtype)
    fresh.set_csr_csc(csr, csc)
    fresh.set_factors(A0, B0)
    fresh.sweeps(params)
    for x, y in zip(fit.get_factors(), fresh.get_factors()):
        assert _same_bits(x, y)


# ---------------------------------------------------------------- 5. the handle is left untouched
def test_predict_leaves_handle_untouched():
    fit = _fitted("pl6k", np.float64)
    before = fit.get_factors()
    top_before = fit.topN(users=np.arange(50), top_n=10, output_score=True)
    u, i = _pairs(np.random.default_rng(8), fit.dimA, fit.dimB, CHUNK + 10, np.uint64)
    fit.predict(u, i)
    for x, y in zip(before, fit.get_factors()):
        assert _same_bits(x, y)
    top_after = fit.topN(users=np.arange(50), top_n=10, output_score=True)
    assert np.array_equal(top_before[0], top_after[0]) and _same_bits(top_before[1], top_after[1])


# ---------------------------------------------------------------- 6. set_coo
def _coo_case(dtype, ixdt, seed, n=40_000, dimA=700, dimB=300):
    """Shuffled triplets with many duplicates, heavy columns and an empty row (13)."""
    rng = np.random.default_rng(seed)
    rows = rng.integers(0, dimA, n)
    cols = rng.zipf(1.6, n) % dimB
    vals = (1 + rng.geometric(0.5, n)).astype(dtype)
    rows[rows == 13] = 14
    rows = np.concatenate([rows, rows[:5000]])                       # exact repeats of the first 5000 triplets
    cols = np.concatenate([cols, cols[:5000]])
    vals = np.concatenate([vals, vals[:5000]])
    p = rng.permutation(rows.shape[0])
    return rows[p].astype(ixdt), cols[p].astype(ixdt), np.ascontiguousarray(vals[p]), dimA, dimB


def _scipy_csr_csc(rows, cols, vals, dimA, dimB):
    from scipy.sparse import coo_matrix
    coo = coo_matrix((vals, (rows.astype(np.int64), cols.astype(np.int64))), shape=(dimA, dimB))
    trip = lambda m: (np.ascontiguousarray(m.data, dtype=vals.dtype), np.ascontiguousarray(m.indptr, np.uint64),
                      np.ascontiguousarray(m.indices, np.uint64))
    return trip(coo.tocsr()), trip(coo.tocsc())


def _sweep_from(dimA, dimB, A0, B0, params, coo=None, csr_csc=None):
    from poismf_b200.device import DeviceFit
    fit = DeviceFit(dimA, dimB, A0.shape[1], A0.dtype)
    if coo is not None:
        fit.set_coo(*coo)
    else:
        fit.set_csr_csc(*csr_csc)
    fit.set_factors(A0, B0)
    fit.sweeps(params)
    return fit


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("ixdt", IXDTS)
def test_set_coo_sweeps_equal_scipy_and_fit_coo(dtype, ixdt):
    from poismf_b200 import _lib, c_funs
    from poismf_b200.synth import init_factors
    k = 16
    rows, cols, vals, dimA, dimB = _coo_case(dtype, ixdt, seed=21)
    A0, B0 = init_factors(dimA, dimB, k, dtype=dtype)
    for case in ("pg", "cg"):
        method, kw = hyper(case, k)
        params = _lib.make_params(method, **kw)
        fit = _sweep_from(dimA, dimB, A0, B0, params, coo=(rows, cols, vals))
        host = _sweep_from(dimA, dimB, A0, B0, params, csr_csc=_scipy_csr_csc(rows, cols, vals, dimA, dimB))
        A2, B2 = A0.copy(), B0.copy()
        assert c_funs._fit_coo(rows, cols, vals, A2, B2, method=method, limit_step=kw.get("limit_step", False),
                               l2_reg=kw["l2_reg"], step_size=kw.get("step_size", 1e-7), niter=kw["numiter"],
                               maxupd=kw["maxupd"], early_stop=False, reuse_prev=False) == 0
        A, B = fit.get_factors()
        for x, y, z in zip((A, B), host.get_factors(), (A2, B2)):
            assert _same_bits(x, y) and _same_bits(x, z), case
        assert not A[13].any()                                       # the empty row is zeroed
        # predict and topN on the ingested handle
        u, i = _pairs(np.random.default_rng(9), dimA, dimB, 5000, ixdt)
        assert _same_bits(fit.predict(u, i), _stateless(A, B, u, i))
        ids, sc = fit.topN(users=np.arange(20), top_n=5, output_score=True)
        ids2, sc2 = c_funs._topN_batch(A, B, users=np.arange(20), top_n=5, output_score=True)
        assert np.array_equal(ids, ids2) and _same_bits(sc, sc2)


def test_set_coo_replaces_matrix_and_error_states():
    from poismf_b200 import _lib
    from poismf_b200.synth import init_factors
    dtype, k = np.float64, 8
    rows, cols, vals, dimA, dimB = _coo_case(dtype, np.uint64, seed=31)
    rows2, cols2, vals2, _, _ = _coo_case(dtype, np.uint64, seed=32, n=25_000)
    A0, B0 = init_factors(dimA, dimB, k, dtype=dtype)
    params = _lib.make_params("cg", l2_reg=1e4, maxupd=5, numiter=2, limit_step=True)
    want2 = _sweep_from(dimA, dimB, A0, B0, params, coo=(rows2, cols2, vals2)).get_factors()
    # a second set_coo with other triplets: fits like a fresh handle
    fit = _sweep_from(dimA, dimB, A0, B0, params, coo=(rows, cols, vals))
    fit.set_coo(rows2, cols2, vals2)
    fit.set_factors(A0, B0)
    fit.sweeps(params)
    for x, y in zip(fit.get_factors(), want2):
        assert _same_bits(x, y)
    # zero entries: 2, the handle unchanged (the same matrix sweeps on)
    fit.set_factors(A0, B0)
    with pytest.raises(ValueError):
        fit.set_coo(rows[:0], cols[:0], vals[:0])
    fit.sweeps(params)
    for x, y in zip(fit.get_factors(), want2):
        assert _same_bits(x, y)
    # an id out of range: 2, no matrix (a sweep fails with 1), factors untouched
    for bad in ((rows, cols, dimB), (rows, cols, -1)):
        r_, c_ = bad[0].astype(np.int64), bad[1].astype(np.int64).copy()
        c_[len(c_) // 2] = bad[2]
        before = fit.get_factors()
        with pytest.raises(ValueError):
            fit.set_coo(r_, c_, vals)
        for x, y in zip(before, fit.get_factors()):
            assert _same_bits(x, y)
        with pytest.raises(MemoryError):
            fit.sweeps(params)
        for x, y in zip(before, fit.get_factors()):
            assert _same_bits(x, y)
    # and a valid set_coo restores it
    fit.set_coo(rows2, cols2, vals2)
    fit.set_factors(A0, B0)
    fit.sweeps(params)
    for x, y in zip(fit.get_factors(), want2):
        assert _same_bits(x, y)
    with pytest.raises(ValueError):
        fit.set_coo(rows, cols.astype(np.int32), vals)
    rc = fit.L.pmf_b200_set_coo(fit.h, rows.ctypes.data, cols.ctypes.data, vals.ctypes.data, rows.shape[0], 2)
    assert rc == 2


# ---------------------------------------------------------------- 7. two GPUs
def _two_gpu_case():
    csr, csc, A0, B0, k = problem("pl6k", np.float32)
    u, i = _pairs(np.random.default_rng(11), A0.shape[0], B0.shape[0], CHUNK + 77_777, np.uint64)
    return csr, csc, A0, B0, k, u, i


def _two_gpu_worker(rank, world, port, q):
    import torch
    import torch.distributed as dist
    from poismf_b200 import _lib
    from poismf_b200.sharding import GpuBackend, ShardedSweep, user_ranges
    torch.cuda.set_device(rank)
    os.environ["POISMF_B200_DEVICE"] = str(rank)
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    csr, csc, A0, B0, k, u, i = _two_gpu_case()
    be = GpuBackend(csr, csc, A0, B0, rank, world, rank)
    params = _lib.make_params("cg", l2_reg=1e4, maxupd=5, numiter=2, limit_step=True, flags=_lib.FLAG_NO_LOCKSTEP)
    ShardedSweep(be, A0.shape[0], B0.shape[0], np.float32).run(params)
    scores = be.predict(u, i)                       # right after the sweeps: predict waits for the peers' rows
    lo, hi = user_ranges(u.shape[0], world)[rank]
    mine = be.predict(u, i, gather=False)
    A, B = be.factors()
    bad_raised = False
    uu = u.copy(); uu[-1] = A0.shape[0]             # in the last rank's range only
    try:
        be.predict(uu, i)
    except ValueError:
        bad_raised = True
    rows = np.repeat(np.arange(A0.shape[0], dtype=np.uint64), np.diff(csr[1].astype(np.int64)))
    try:
        be.fit.set_coo(rows, csr[2], csr[0])
        coo_rc = 0
    except ValueError:
        coo_rc = 2
    q.put((rank, scores, np.array_equal(mine, scores[lo:hi]), A, B, bad_raised, coo_rc))
    dist.barrier()
    be.finish()
    dist.destroy_process_group()


def test_two_gpu_predict_matches_single_gpu():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from poismf_b200.device import DeviceFit
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_two_gpu_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=300) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    _, _, A0, B0, k, u, i = _two_gpu_case()
    for rank, scores, own_range, A, B, bad_raised, coo_rc in res:
        one = DeviceFit(A.shape[0], B.shape[0], k, np.float32)
        one.set_factors(A, B)
        assert _same_bits(scores, one.predict(u, i)), rank
        assert own_range and bad_raised and coo_rc == 2, rank
