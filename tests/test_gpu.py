"""GPU parity tests: the CUDA path, called through the C ABI with host buffers (the drop-in
boundary), against the CPU oracle on the same seeded inputs.

Tolerances (BASELINE.json north_star): factors after a sweep within 1e-5 relative in double
and 1e-3 in float; log-likelihood within 1e-4 relative; topN identical outside ties.

  * STRICT mode (sequential sums, no FMA) is the parity mode: it must reproduce the oracle
    to ~1e-9 (bit-exact except where CUDA's log() and glibc's differ by an ulp).
  * FAST mode (FMA, tree reductions, cached line search) meets the north_star gates where the
    reference meets them against ITSELF under a BLAS change (pg both dtypes, cg double:
    SURVEY.md §4.1); for cg-float and tncg, which are chaotic in the rounding, it is held to
    the log-likelihood gate and to never being worse in objective than the oracle.
"""
import ctypes
import os

import numpy as np
import pytest

from conftest import (CASES, FM_CASES, FS_CASES, FS_ROWS, ROOT, fm_hyper, fm_problem, fs_row, golden, hyper, problem,
                      row_rel_err, run_device)
from oracle.oracle import Restatement

pytestmark = pytest.mark.gpu
GOLD = golden()
DTYPES = [np.float64, np.float32]
FLAG_STRICT, FLAG_NO_CACHED, FLAG_NO_LOCKSTEP = 1, 2, 4


def _oracle(dtype, csr, csc, A0, B0, method, kw):
    A, B = A0.copy(), B0.copy()
    assert Restatement(dtype).run_poismf(A, B, csr, csc, method, **kw) == 0
    return A, B


# ---------------------------------------------------------------- strict mode == oracle
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("prob", ["readme", "ragged", "pl2k", "pl6k"])
@pytest.mark.parametrize("case", ["pg", "pg_w", "cg", "cg_nolimit_w", "tncg", "tncg_w"])
def test_strict_matches_oracle(dtype, prob, case):
    csr, csc, A0, B0, k = problem(prob, dtype)
    method, kw = hyper(case, k)
    Ar, Br = _oracle(dtype, csr, csc, A0, B0, method, kw)
    A, B = A0.copy(), B0.copy()
    assert run_device(csr, csc, A, B, method, kw, flags=FLAG_STRICT) == 0
    if method == "pg":                       # no transcendental on the path: bit-exact
        assert np.array_equal(A, Ar) and np.array_equal(B, Br)
        return
    # cg / tncg: identical up to log() ulps, which can flip a branch on rare rows
    tol = 1e-9 if dtype == np.float64 else 1e-5
    for X, Y in ((A, Ar), (B, Br)):
        bad = row_rel_err(X, Y) > tol
        assert bad.mean() <= 0.002, f"{bad.sum()} of {bad.size} rows differ from the oracle"


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("case", list(CASES))
def test_strict_matches_reference_golden(dtype, case):
    """Against outputs of the reference itself (tests/golden, generated from oracle/_ref)."""
    name = np.dtype(dtype).name
    for prob in ("readme", "ragged"):
        csr, csc, A0, B0, k = problem(prob, dtype)
        method, kw = hyper(case, k)
        A, B = A0.copy(), B0.copy()
        assert run_device(csr, csc, A, B, method, kw, flags=FLAG_STRICT) == 0
        tol = 1e-9 if dtype == np.float64 else 1e-5
        for X, Y in ((A, GOLD[f"{prob}/{name}/{case}/A"]), (B, GOLD[f"{prob}/{name}/{case}/B"])):
            bad = row_rel_err(X, Y) > tol
            lim = 0.0 if method == "pg" else (0.05 if "reuse" in case else 0.005)
            assert bad.mean() <= lim, (prob, case, int(bad.sum()), bad.size)


# ---------------------------------------------------------------- fast mode, north_star gates
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("prob", ["readme", "pl2k", "pl6k"])
@pytest.mark.parametrize("case", ["pg", "pg_w"])
def test_fast_pg_within_gate(dtype, prob, case):
    csr, csc, A0, B0, k = problem(prob, dtype)
    method, kw = hyper(case, k)
    Ar, Br = _oracle(dtype, csr, csc, A0, B0, method, kw)
    A, B = A0.copy(), B0.copy()
    assert run_device(csr, csc, A, B, method, kw) == 0
    gate = 1e-5 if dtype == np.float64 else 1e-3
    assert row_rel_err(A, Ar).max() <= gate and row_rel_err(B, Br).max() <= gate


@pytest.mark.parametrize("prob", ["readme", "pl2k", "pl6k"])
@pytest.mark.parametrize("flags", [0, FLAG_NO_CACHED])
def test_fast_cg_double_within_gate(prob, flags):
    dtype = np.float64
    csr, csc, A0, B0, k = problem(prob, dtype)
    method, kw = hyper("cg", k)
    Ar, Br = _oracle(dtype, csr, csc, A0, B0, method, kw)
    A, B = A0.copy(), B0.copy()
    assert run_device(csr, csc, A, B, method, kw, flags=flags) == 0
    # SURVEY §4.1: two CPU builds of the reference agree to <= 3.5e-6 here
    assert (row_rel_err(A, Ar) > 1e-5).mean() <= 0.001 and (row_rel_err(B, Br) > 1e-5).mean() <= 0.001
    assert np.abs(A - Ar).max() <= 1e-4 * np.abs(Ar).max()


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("case", ["cg", "cg_nolimit_w", "tncg", "tncg_w", "tncg_reuse_stop"])
def test_fast_llk_gate(dtype, case):
    """FINAL Poisson log-likelihood within 1e-4 relative of the oracle's (north_star) — the stable
    quantity for the solvers whose coordinates are chaotic in the rounding (SURVEY §4.1).
    Where the algorithm itself, rebuilt with FMA contraction and -O3, misses that gate against its
    strict build, the device is held to 5x that noise floor: the reference's own fast build
    (oracle/_ref) where it has been built, else the restatement's fast build, which is the same C
    code (bit-identical to the reference when strict) and reproduces the floor measured with it."""
    from oracle.oracle import Ref
    csr, csc, A0, B0, k = problem("pl2k", dtype)
    method, kw = hyper(case, k)
    if method == "cg":
        kw["numiter"] = 10          # "final": a fit, not a single sweep
    Ar, Br = _oracle(dtype, csr, csc, A0, B0, method, kw)
    A, B = A0.copy(), B0.copy()
    assert run_device(csr, csc, A, B, method, kw) == 0
    assert np.isfinite(A).all() and np.isfinite(B).all() and (A >= 0).all() and (B >= 0).all()
    orc = Restatement(dtype)
    l_ref, l_dev = orc.llk(Ar, Br, csr), orc.llk(A, B, csr)
    # double: the north_star gate.  float: 2e-3 — measured floor of the reference against itself
    # on this very problem is 3e-6 (cg) .. 3e-2 (tncg), see scripts/dev_llk.py / DESIGN.md §parity
    gate = 1e-4 if dtype == np.float64 else 2e-3
    fast = Ref(dtype, fast=True) if Ref.available(dtype, fast=True) else Restatement(dtype, fast=True)
    A2, B2 = A0.copy(), B0.copy()
    fast.run_poismf(A2, B2, csr, csc, method, **kw)
    noise = abs(orc.llk(A2, B2, csr) - l_ref) / abs(l_ref)
    gate = max(gate, 5 * noise)
    assert abs(l_dev - l_ref) <= gate * abs(l_ref), (l_dev, l_ref, gate)
    # sparsity (EXACT zeros) stays next to the strict reference's, also in float with FMA on
    # (the final unscale is never contracted; the reference's own FMA build loses its zeros)
    assert abs((A == 0).mean() - (Ar == 0).mean()) <= 0.03 and abs((B == 0).mean() - (Br == 0).mean()) <= 0.03


# ---------------------------------------------------------------- edge cases
def test_empty_rows_are_zeroed_and_single_nnz_rows():
    dtype = np.float64
    csr, csc, A0, B0, k = problem("ragged", dtype)
    empty_cols = np.diff(csc[1].astype(np.int64)) == 0
    assert empty_cols.any()
    for case in ("pg", "cg", "tncg"):
        method, kw = hyper(case, k)
        A, B = A0.copy(), B0.copy()
        assert run_device(csr, csc, A, B, method, kw) == 0
        assert (B[empty_cols] == 0).all()                       # src/poismf.c:166-169 etc. (Q6)


def test_int32_index_variant_matches_size_t_variant():
    """The R build's sparse_ix=int path (host drop-in compiled with -DPMF_INDEX_INT)."""
    dtype = np.float64
    csr, csc, A0, B0, k = problem("pl2k", dtype)
    method, kw = hyper("cg", k)
    A1, B1 = A0.copy(), B0.copy()
    assert run_device(csr, csc, A1, B1, method, kw, flags=FLAG_STRICT) == 0
    L = ctypes.CDLL(os.path.join(ROOT, "poismf_b200", "libpoismf_host_double_int.so"))
    sz, d, vp = ctypes.c_size_t, ctypes.c_double, ctypes.c_void_p
    L.run_poismf.restype = ctypes.c_int
    L.run_poismf.argtypes = [vp] * 8 + [sz, sz, sz, d, d, d, d, ctypes.c_int, ctypes.c_bool, sz, sz,
                                        ctypes.c_bool, ctypes.c_bool, ctypes.c_bool, ctypes.c_int]
    i32 = lambda a: np.ascontiguousarray(a.astype(np.int32))
    p = lambda a: a.ctypes.data_as(vp)
    A2, B2 = A0.copy(), B0.copy()
    rp, ri, cp, ci = i32(csr[1]), i32(csr[2]), i32(csc[1]), i32(csc[2])
    os.environ["POISMF_B200_FLAGS"] = "1"
    try:
        rc = L.run_poismf(p(A2), p(csr[0]), p(rp), p(ri), p(B2), p(csc[0]), p(cp), p(ci), A0.shape[0], B0.shape[0], k,
                          kw["l2_reg"], 0., 1., 1e-7, 2, True, kw["numiter"], kw["maxupd"], False, False, True, 1)
    finally:
        del os.environ["POISMF_B200_FLAGS"]
    assert rc == 0 and np.array_equal(A1, A2) and np.array_equal(B1, B2)


def test_sharded_half_sweeps_equal_full_sweep():
    """Rows are independent within a half-sweep: driving two row shards one after the other
    through pmf_b200_half_sweep gives the same bits as the full half-sweep (per-row teams; the
    lock-step path of the heaviest rows sums in an order that depends on the shard's heavy rows:
    it agrees at the log-likelihood level, checked below)."""
    from poismf_b200 import SIDE_CSC, SIDE_CSR, make_params
    from poismf_b200.device import DeviceFit
    from poismf_b200.sharding import nnz_balanced_ranges, slice_compressed
    dtype = np.float32
    csr, csc, A0, B0, k = problem("pl6k", dtype)
    method, kw = hyper("cg", k)
    kw = dict(kw); kw.pop("numiter")
    params = make_params(method, numiter=1, flags=FLAG_NO_LOCKSTEP, **kw)
    full = DeviceFit(A0.shape[0], B0.shape[0], k, dtype)
    full.set_csr_csc(csr, csc); full.set_factors(A0, B0)
    full.sweeps(params)
    Af, Bf = full.get_factors()
    # shards: both share one replica pair, updated in place shard after shard
    shards = []
    for r in range(2):
        f = DeviceFit(A0.shape[0], B0.shape[0], k, dtype)
        a0, a1 = nnz_balanced_ranges(csr[1], 2)[r]
        b0, b1 = nnz_balanced_ranges(csc[1], 2)[r]
        f.set_matrix(SIDE_CSR, *slice_compressed(csr, a0, a1), row_begin=a0, n_rows=a1 - a0)
        f.set_matrix(SIDE_CSC, *slice_compressed(csc, b0, b1), row_begin=b0, n_rows=b1 - b0)
        shards.append(f)
    shards[0].set_factors(A0, B0)
    shards[1].bind_factors(shards[0].factor_ptr(0), shards[0].factor_ptr(1))
    for side in (SIDE_CSC, SIDE_CSR):
        for f in shards:
            f.half_sweep(side, params, 1e-7, 1.0)
            f.sync()
    As, Bs = shards[0].get_factors()
    assert np.array_equal(As, Af) and np.array_equal(Bs, Bf)
    # default flags (lock-step path for the heaviest rows): same fit at the log-likelihood level
    params = make_params(method, numiter=1, **kw)
    full.set_factors(A0, B0); full.sweeps(params)
    Al, Bl = full.get_factors()
    orc = Restatement(dtype)
    l_inv, l_lock = orc.llk(Af, Bf, csr), orc.llk(Al, Bl, csr)
    # (float cg after ONE sweep: the reference's own FMA and strict builds are 2e-3 apart at this point,
    # tests/test_gpu_headline.py)
    assert abs(l_lock - l_inv) <= 1e-3 * abs(l_inv), (l_lock, l_inv)


# ---------------------------------------------------------------- predict_multiple / topN
@pytest.mark.parametrize("dtype", DTYPES)
def test_predict_multiple_bit_exact(dtype):
    from poismf_b200 import c_funs
    name = np.dtype(dtype).name
    csr, csc, A0, B0, k = problem("readme", dtype)
    rng = np.random.default_rng(3)
    ixA = rng.integers(0, A0.shape[0], 257).astype(np.uint64)
    ixB = rng.integers(0, B0.shape[0], 257).astype(np.uint64)
    out = np.empty(257, dtype)
    c_funs._predict_multiple(out, A0, B0, ixA, ixB)
    assert np.array_equal(out, GOLD[f"predict/{name}"])
    # ragged: k = 50, many pairs
    csr, csc, A0, B0, k = problem("pl6k", dtype)
    ixA = rng.integers(0, A0.shape[0], 100_003).astype(np.uint64)
    ixB = rng.integers(0, B0.shape[0], 100_003).astype(np.uint64)
    out = np.empty(ixA.shape[0], dtype)
    c_funs._predict_multiple(out, A0, B0, ixA, ixB)
    assert np.array_equal(out, Restatement(dtype).predict_multiple(A0, B0, ixA, ixB))


@pytest.mark.parametrize("dtype", DTYPES)
def test_topn_matches_reference(dtype):
    from poismf_b200 import c_funs
    name = np.dtype(dtype).name
    csr, csc, A0, B0, k = problem("readme", dtype)
    rng = np.random.default_rng(3)
    rng.integers(0, 1, 514)  # keep the stream aligned with make_golden.py
    rng = np.random.default_rng(3); rng.integers(0, A0.shape[0], 257); rng.integers(0, B0.shape[0], 257)
    Brand = np.ascontiguousarray(rng.gamma(1, 1, size=B0.shape).astype(dtype))
    a = np.ascontiguousarray(A0[3])
    none = np.empty(0, np.uint64)
    ix, sc = c_funs._call_topN(a, Brand, none, none, top_n=10, output_score=True)
    assert np.array_equal(sc, GOLD[f"topn/{name}/score"]) and np.array_equal(ix, GOLD[f"topn/{name}/ix"])
    excl = np.arange(0, 1000, 7, dtype=np.uint64)
    ix, sc = c_funs._call_topN(a, Brand, none, excl, top_n=10, output_score=True)
    assert np.array_equal(sc, GOLD[f"topn_excl/{name}/score"]) and np.array_equal(ix, GOLD[f"topn_excl/{name}/ix"])
    # include list + oracle, and a batch
    orc = Restatement(dtype)
    inc = rng.choice(1000, 120, replace=False).astype(np.uint64)
    ix, sc = c_funs._call_topN(a, Brand, inc, none, top_n=7, output_score=True)
    rc, ix_r, sc_r = orc.topN(a, Brand, 7, include=inc)
    assert rc == 0 and np.array_equal(sc, sc_r) and np.array_equal(ix, ix_r)
    users = np.array([0, 5, 99, 17], dtype=np.uint64)
    lens = [0, 3, 50, 1]
    ptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    eix = np.concatenate([np.sort(rng.choice(1000, n, replace=False)) for n in lens]).astype(np.uint64)
    bix, bsc = c_funs._topN_batch(A0, Brand, users=users, excl_ptr=ptr, excl_ix=eix, top_n=12, output_score=True)
    for u, usr in enumerate(users):
        ex = eix[int(ptr[u]):int(ptr[u + 1])]
        rc, ix_r, sc_r = orc.topN(np.ascontiguousarray(A0[int(usr)]), Brand, 12, exclude=ex if ex.size else None)
        assert np.array_equal(bsc[u], sc_r) and np.array_equal(bix[u], ix_r)


def test_topn_invalid_arguments_return_2():
    from poismf_b200 import c_funs
    B = np.ones((10, 3)); a = np.ones(3)
    none = np.empty(0, np.uint64)
    with pytest.raises(ValueError):
        c_funs._call_topN(a, B, none, none, top_n=0, check=True)
    with pytest.raises(ValueError):
        c_funs._call_topN(a, B, none, np.arange(6, dtype=np.uint64), top_n=5, check=True)
    c_funs._call_topN(a, B, none, np.arange(6, dtype=np.uint64), top_n=5)     # the reference's wrapper ignores the code


# ---------------------------------------------------------------- BASELINE full size (config #2)
def test_lastfm_shaped_full_size_properties():
    """Size-independent properties at the bench size: finite, non-negative factors, the sweep
    improves the log-likelihood of the init, and the first sweeps agree between the cached and
    direct line searches at the log-likelihood gate."""
    from poismf_b200 import c_funs
    from poismf_b200.synth import init_factors, powerlaw_counts
    dtype = np.float32
    dimA, dimB, k = 359_000, 160_000, 50
    csr, csc = powerlaw_counts(dimA, dimB, 17_500_000, dtype=dtype, seed=1)
    A0, B0 = init_factors(dimA, dimB, k, dtype=dtype)
    outs = []
    for flags in (0, FLAG_NO_CACHED):
        A, B = A0.copy(), B0.copy()
        rc = c_funs._run_poismf(csr[0], csr[2], csr[1], csc[0], csc[2], csc[1], A, B, method="cg", limit_step=True,
                                l2_reg=1e4, niter=2, maxupd=5, early_stop=False, reuse_prev=False, flags=flags)
        assert rc == 0 and np.isfinite(A).all() and np.isfinite(B).all() and (A >= 0).all() and (B >= 0).all()
        outs.append((A, B))
    def llk(A, B):
        rows = np.repeat(np.arange(dimA), np.diff(csr[1].astype(np.int64)))
        acc = 0.0
        for s in range(0, rows.shape[0], 1 << 22):
            sl = slice(s, s + (1 << 22))
            pred = np.einsum("ij,ij->i", A[rows[sl]].astype(np.float64), B[csr[2][sl].astype(np.int64)].astype(np.float64))
            acc += (csr[0][sl] * np.log(pred)).sum()
        return acc - A.sum(0, dtype=np.float64) @ B.sum(0, dtype=np.float64)
    l0, l1, l2 = llk(A0, B0), llk(*outs[0]), llk(*outs[1])
    assert l1 > l0 and l2 > l0
    assert abs(l1 - l2) <= 2e-3 * abs(l2)
    # predict_multiple through the drop-in on 1M pairs of the fitted factors
    rng = np.random.default_rng(0)
    ixA = rng.integers(0, dimA, 1_000_000).astype(np.uint64); ixB = rng.integers(0, dimB, 1_000_000).astype(np.uint64)
    out = np.empty(ixA.shape[0], dtype)
    A, B = outs[0]
    c_funs._predict_multiple(out, A, B, ixA, ixB)
    want = np.einsum("ij,ij->i", A[ixA.astype(np.int64)].astype(np.float64), B[ixB.astype(np.int64)].astype(np.float64))
    assert np.abs(out - want).max() <= 1e-5 * max(np.abs(want).max(), 1.0)


# ---------------------------------------------------------------- two GPUs (skipped on one)
def _two_gpu_worker(rank, world, port, exchange, q):
    import torch
    import torch.distributed as dist
    from poismf_b200 import make_params
    from poismf_b200.sharding import GpuBackend, ShardedSweep
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world,
                            device_id=torch.device("cuda", rank))
    dtype = np.float32
    csr, csc, A0, B0, k = problem("pl6k", dtype)
    out = {}
    for case in ("cg", "pg", "tncg"):
        method, kw = hyper(case, k)
        params = make_params(method, flags=FLAG_NO_LOCKSTEP, **kw)      # per-row teams only: partition-invariant bits
        be = GpuBackend(csr, csc, A0, B0, rank, world, rank, exchange=exchange)
        ShardedSweep(be, A0.shape[0], B0.shape[0], dtype).run(params)
        A, B = be.factors()
        out[case] = (A.copy(), B.copy())
        if case == "cg":    # rank the users right after the fit, each rank its share against its own replicas
            out["topn"] = be.topN(10, output_score=True)
        del be
    q.put((rank, out))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("exchange", ["p2p", "nccl"])
def test_two_gpu_sharded_matches_single_gpu(exchange):
    """Sharded over 2 GPUs (replicas refreshed by peer-memory stores fused into the row kernels,
    or by NCCL broadcasts) == the single-GPU fit, bit for bit, on every rank's replica."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import socket
    import torch.multiprocessing as mp
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_two_gpu_worker, args=(r, 2, port, exchange, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=300) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    dtype = np.float32
    csr, csc, A0, B0, k = problem("pl6k", dtype)
    for case in ("cg", "pg", "tncg"):
        method, kw = hyper(case, k)
        A, B = A0.copy(), B0.copy()
        assert run_device(csr, csc, A, B, method, kw, flags=FLAG_NO_LOCKSTEP) == 0
        for r in (0, 1):
            assert np.array_equal(res[r][case][0], A) and np.array_equal(res[r][case][1], B), (case, r)
        if case == "cg":
            from poismf_b200 import c_funs
            ids, sc = c_funs._topN_batch(A, B, top_n=10, output_score=True)
            for r in (0, 1):
                ids_r, sc_r = res[r]["topn"]
                assert np.array_equal(sc_r, sc), r
                assert all((sc[u] == sc[u][t]).sum() > 1 for u, t in zip(*np.nonzero(ids_r != ids)))


def _two_gpu_topn_worker(rank, world, port, q):
    import torch
    import torch.distributed as dist
    from poismf_b200.sharding import topn_sharded
    torch.cuda.set_device(rank)
    os.environ["POISMF_B200_DEVICE"] = str(rank)
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    A, B, ptr, eix = _topn_case()
    ids, sc = topn_sharded(A, B, 20, excl_ptr=ptr, excl_ix=eix, output_score=True, rank=rank, world=world)
    q.put((rank, ids, sc))
    dist.barrier()
    dist.destroy_process_group()


def _topn_case():
    rng = np.random.default_rng(31)
    A = np.ascontiguousarray(rng.gamma(0.5, 0.5, size=(301, 32)).astype(np.float32))
    B = np.ascontiguousarray(rng.gamma(0.5, 0.5, size=(20_000, 32)).astype(np.float32))
    lens = rng.integers(0, 50, A.shape[0])
    ptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    eix = np.concatenate([rng.choice(B.shape[0], int(m), replace=False) for m in lens]).astype(np.uint64)
    return A, B, ptr, eix


def test_two_gpu_user_sharded_topn_matches_single_gpu():
    """topN shards by users, B replicated, no exchange inside the scoring (SURVEY 8e)."""
    import torch
    from poismf_b200 import c_funs
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import socket
    import torch.multiprocessing as mp
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_two_gpu_topn_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=300) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    A, B, ptr, eix = _topn_case()
    ids, sc = c_funs._topN_batch(A, B, excl_ptr=ptr, excl_ix=eix, top_n=20, output_score=True)
    for _, i2, s2 in res:
        assert np.array_equal(i2, ids) and np.array_equal(s2, sc)


# ---------------------------------------------------------------- the other BASELINE shapes, scaled down
def test_netflix_shaped_tncg_k100():
    """BASELINE config #3 shape at 1/100 scale: few, very long columns (every column is a
    cluster/CTA row), k=100, tncg with maxupd = 15k."""
    from poismf_b200.synth import init_factors, powerlaw_counts
    dtype = np.float64
    dimA, dimB, k = 4800, 177, 100
    csr, csc = powerlaw_counts(dimA, dimB, 250_000, alpha_a=0.5, alpha_b=0.7, dtype=dtype, seed=3)
    A0, B0 = init_factors(dimA, dimB, k, dtype=dtype)
    kw = dict(l2_reg=1e3, maxupd=15 * k, numiter=1)
    Ar, Br = _oracle(dtype, csr, csc, A0, B0, "tncg", kw)
    orc = Restatement(dtype)
    l_ref = orc.llk(Ar, Br, csr)
    for flags, gate in ((FLAG_STRICT, 1e-7), (0, 1e-4)):
        A, B = A0.copy(), B0.copy()
        assert run_device(csr, csc, A, B, "tncg", kw, flags=flags) == 0
        assert np.isfinite(A).all() and np.isfinite(B).all() and (A >= 0).all() and (B >= 0).all()
        l_dev = orc.llk(A, B, csr)
        assert abs(l_dev - l_ref) <= gate * abs(l_ref), (flags, l_dev, l_ref)
        if flags == FLAG_STRICT:
            assert (row_rel_err(A, Ar) > 1e-9).mean() <= 0.01 and (row_rel_err(B, Br) > 1e-9).mean() <= 0.02


@pytest.mark.parametrize("dtype", DTYPES)
def test_midsize_tncg_all_bins_populated(dtype):
    """1/8-scale config #2 (45k x 20k, 1.9M nnz, k=50): every bin of the planner is populated at once
    (sub-warp ... streaming clusters).  Regression test for a shared-memory race of the CTA / cluster
    teams in the tncg line search (a warp overwrote a vector another warp was still summing; the
    double-precision kernels then faulted on this problem, r1): the sweep must complete, stay finite
    and non-negative, and raise the log-likelihood over the initial factors."""
    from poismf_b200.synth import init_factors, powerlaw_counts
    dimA, dimB, k = 45_000, 20_000, 50
    csr, csc = powerlaw_counts(dimA, dimB, 2_200_000, dtype=dtype, seed=1)
    A0, B0 = init_factors(dimA, dimB, k, seed=1, dtype=dtype)
    kw = dict(l2_reg=1e3, maxupd=20, numiter=1)
    orc = Restatement(dtype)
    l0 = orc.llk(A0, B0, csr)
    for _ in range(2):
        A, B = A0.copy(), B0.copy()
        assert run_device(csr, csc, A, B, "tncg", kw) == 0
        assert np.isfinite(A).all() and np.isfinite(B).all() and (A >= 0).all() and (B >= 0).all()
        assert orc.llk(A, B, csr) > l0


def test_webscale_shaped_pg_k64():
    """BASELINE config #4 shape at 1/500 scale: k=64, pg, maxupd=1 (SURVEY Q5), float32."""
    from poismf_b200.synth import init_factors, powerlaw_counts
    dtype = np.float32
    dimA, dimB, k = 20_000, 2_000, 64
    csr, csc = powerlaw_counts(dimA, dimB, 4_000_000, dtype=dtype, seed=4)
    A0, B0 = init_factors(dimA, dimB, k, dtype=dtype)
    kw = dict(l2_reg=1e9, step_size=1e-7, maxupd=1, numiter=3)
    Ar, Br = _oracle(dtype, csr, csc, A0, B0, "pg", kw)
    assert (Ar > 0).any() and (Br > 0).any()
    A, B = A0.copy(), B0.copy()
    assert run_device(csr, csc, A, B, "pg", kw, flags=FLAG_STRICT) == 0
    assert np.array_equal(A, Ar) and np.array_equal(B, Br)            # heavy rows included: bit-exact
    A, B = A0.copy(), B0.copy()
    assert run_device(csr, csc, A, B, "pg", kw) == 0
    assert row_rel_err(A, Ar).max() <= 1e-3 and row_rel_err(B, Br).max() <= 1e-3


# ---------------------------------------------------------------- factors_multiple (SURVEY §8f rank 1)
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("case", list(FM_CASES))
def test_factors_multiple_matches_oracle(dtype, case):
    from poismf_b200 import c_funs
    for prob in ("readme", "pl2k"):
        csr, B, Bsum, Amean, k = fm_problem(prob, dtype)
        method, kw = fm_hyper(case, k)
        rc, Ar = Restatement(dtype).factors_multiple(B, Bsum, Amean, csr, method, **kw)
        assert rc == 0
        A = c_funs._predict_factors_multiple(B, Bsum, Amean, csr[1], csr[2], csr[0], method=method,
                                             flags=FLAG_STRICT, **kw)
        if method == "pg":
            assert np.array_equal(A, Ar)
        else:
            tol = 1e-9 if dtype == np.float64 else 1e-5
            assert (row_rel_err(A, Ar) > tol).mean() <= 0.005
        if method == "pg" or (method == "cg" and dtype == np.float64 and kw.get("limit_step")):
            A = c_funs._predict_factors_multiple(B, Bsum, Amean, csr[1], csr[2], csr[0], method=method, **kw)
            gate = 1e-5 if dtype == np.float64 else 1e-3
            assert (row_rel_err(A, Ar) > gate).mean() <= 0.002


# ---------------------------------------------------------------- COO ingestion (SURVEY §8f rank 4)
def _coo_case(dtype, ixdt, seed=11, n=40000, dimA=700, dimB=300):
    rng = np.random.default_rng(seed)
    rows = rng.integers(0, dimA, n).astype(ixdt)
    cols = (rng.zipf(1.6, n) % dimB).astype(ixdt)                 # heavy columns, many duplicates
    vals = (1 + rng.geometric(0.5, n)).astype(dtype)
    rows[rows == 13] = 14                                          # an empty row; column dimB-1 stays rare
    return rows, cols, vals, dimA, dimB


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("ixdt", [np.uint64, np.int32])
def test_coo_ingestion_matches_scipy(dtype, ixdt):
    """coo.tocsr() / coo.tocsc() (poismf/__init__.py:402-404) on the device: same offsets, ids and
    summed counts, bit for bit."""
    from scipy.sparse import coo_matrix
    from poismf_b200 import c_funs
    rows, cols, vals, dimA, dimB = _coo_case(dtype, ixdt)
    coo = coo_matrix((vals, (rows.astype(np.int64), cols.astype(np.int64))), shape=(dimA, dimB))
    for got, want in zip(c_funs._coo_to_csr_csc(rows, cols, vals, dimA, dimB), (coo.tocsr(), coo.tocsc())):
        assert want.has_sorted_indices
        assert np.array_equal(got[1].astype(np.int64), want.indptr.astype(np.int64))
        assert np.array_equal(got[2].astype(np.int64), want.indices.astype(np.int64))
        assert np.array_equal(got[0], want.data.astype(dtype))
    bad = rows.copy(); bad[5] = dimA
    with pytest.raises(ValueError):
        c_funs._coo_to_csr_csc(bad, cols, vals, dimA, dimB)


@pytest.mark.parametrize("case", ["pg", "cg", "tncg"])
def test_fit_from_coo_equals_fit_from_scipy_csr_csc(case):
    from scipy.sparse import coo_matrix
    from poismf_b200 import c_funs
    from poismf_b200.synth import init_factors
    dtype, k = np.float32, 16
    rows, cols, vals, dimA, dimB = _coo_case(dtype, np.uint64, seed=12)
    coo = coo_matrix((vals, (rows.astype(np.int64), cols.astype(np.int64))), shape=(dimA, dimB))
    csr, csc = coo.tocsr(), coo.tocsc()
    trip = lambda m: (np.ascontiguousarray(m.data, dtype=dtype), np.ascontiguousarray(m.indptr, dtype=np.uint64),
                      np.ascontiguousarray(m.indices, dtype=np.uint64))
    A0, B0 = init_factors(dimA, dimB, k, dtype=dtype)
    method, kw = hyper(case, k)
    A, B = A0.copy(), B0.copy()
    assert run_device(trip(csr), trip(csc), A, B, method, kw) == 0
    A2, B2 = A0.copy(), B0.copy()
    rc = c_funs._fit_coo(rows, cols, vals, A2, B2, method=method, limit_step=kw.get("limit_step", False),
                         l2_reg=kw["l2_reg"], step_size=kw.get("step_size", 1e-7), niter=kw["numiter"],
                         maxupd=kw["maxupd"], early_stop=False, reuse_prev=False)
    assert rc == 0 and np.array_equal(A, A2) and np.array_equal(B, B2)
    assert not A2[13].any()                                        # the empty row is zeroed (Q6)


# ---------------------------------------------------------------- matrix cache (SURVEY §8f rank 3)
def test_matrix_cache_between_dropin_calls(monkeypatch):
    """POISMF_B200_CACHE_X=1 keeps the uploaded matrix for the next run_poismf on the same arrays:
    results are those of the uncached call, a changed method re-plans, and in-place edits of the
    arrays are noticed."""
    from poismf_b200 import _lib
    dtype = np.float32
    csr, csc, A0, B0, k = problem("pl6k", dtype)

    def fit(case, flags=0):
        method, kw = hyper(case, k)
        A, B = A0.copy(), B0.copy()
        assert run_device(csr, csc, A, B, method, kw, flags=flags) == 0
        return A, B

    want = {c: fit(c) for c in ("cg", "pg", "tncg")}
    monkeypatch.setenv("POISMF_B200_CACHE_X", "1")
    for c in ("cg", "cg", "pg", "tncg", "cg"):           # first call fills the cache, the others hit it
        A, B = fit(c)
        assert np.array_equal(A, want[c][0]) and np.array_equal(B, want[c][1]), c
    A, B = fit("pg", flags=FLAG_STRICT)                   # strict numerics re-plan on the cached matrix
    monkeypatch.delenv("POISMF_B200_CACHE_X")
    As, Bs = fit("pg", flags=FLAG_STRICT)
    assert np.array_equal(A, As) and np.array_equal(B, Bs)
    monkeypatch.setenv("POISMF_B200_CACHE_X", "1")
    fit("cg")
    csr[0][:] *= 2; csc[0][:] *= 2                        # same pointers, new contents
    A, B = fit("cg")
    monkeypatch.delenv("POISMF_B200_CACHE_X")
    A2, B2 = fit("cg")
    assert np.array_equal(A, A2) and np.array_equal(B, B2)
    assert not np.array_equal(A, want["cg"][0])
    _lib.lib().pmf_b200_release_cache()


# ---------------------------------------------------------------- factors_single (SURVEY §8f rank 2)
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("case", list(FS_CASES))
def test_factors_single_matches_oracle(dtype, case):
    from poismf_b200 import c_funs
    kw = FS_CASES[case]
    tol = 1e-9 if dtype == np.float64 else 1e-5
    for prob in ("readme", "pl2k"):
        csr, B, Bsum, Amean, k = fm_problem(prob, dtype)
        for r in FS_ROWS:
            c, ix = fs_row(csr, r)
            want = Restatement(dtype).factors_single(c, ix, B, Bsum, Amean, **kw)[1]
            got = c_funs._predict_factors(c, ix, B, Bsum, Amean, flags=FLAG_STRICT, **kw)
            assert row_rel_err(got[None], want[None]).max() <= tol, (prob, r)
            fast = c_funs._predict_factors(c, ix, B, Bsum, Amean, **kw)
            assert np.isfinite(fast).all() and (fast >= 0).all()
        z = c_funs._predict_factors(np.empty(0, dtype), np.empty(0, np.uint64), B, Bsum, Amean, **kw)
        assert z.shape == (k,) and not z.any()
    assert GOLD[f"factors_single/{np.dtype(dtype).name}/{case}"].shape == (len(FS_ROWS) + 1, 5)


# ---------------------------------------------------------------- batched topN on the tensor cores
@pytest.mark.parametrize("k,n_top", [(64, 100), (50, 10), (7, 37), (96, 20), (128, 10)])
def test_topn_batch_tensor_core_path_is_exact(k, n_top):
    """The tcgen05/TF32 scorer only proposes candidates; rankings must equal the exact FP32 ones
    (ids identical wherever the exact scores are not tied) and most users must NOT need the exact
    fallback.  Items 30k, users 300, per-user exclusion lists."""
    from poismf_b200 import _lib, c_funs
    rng = np.random.default_rng(11)
    n_items, n_users = 30_000, 300
    A = np.ascontiguousarray(rng.gamma(0.5, 0.5, size=(n_users, k)).astype(np.float32))
    B = np.ascontiguousarray(rng.gamma(0.5, 0.5, size=(n_items, k)).astype(np.float32))
    lens = rng.integers(0, 300, n_users)
    ptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    eix = np.concatenate([np.sort(rng.choice(n_items, int(m), replace=False)) for m in lens]).astype(np.uint64)
    _lib.topn_stats(reset=True)
    ix, sc = c_funs._topN_batch(A, B, excl_ptr=ptr, excl_ix=eix, top_n=n_top, output_score=True)
    n_tc, n_redo = _lib.topn_stats(reset=True)
    assert n_tc == n_users, "tensor-core scorer was not used"
    assert n_redo <= 0.1 * n_users, f"{n_redo} of {n_users} users fell back to the exact scorer"
    orc = Restatement(np.float32)
    for u in range(0, n_users, 7):
        ex = eix[int(ptr[u]):int(ptr[u + 1])]
        rc, ix_r, sc_r = orc.topN(np.ascontiguousarray(A[u]), B, n_top, exclude=ex if ex.size else None)
        assert rc == 0 and np.array_equal(sc[u], sc_r)                 # exact FP32 scores, reference bits
        diff = np.nonzero(ix[u] != ix_r)[0]
        assert all((sc_r == sc_r[t]).sum() > 1 for t in diff), "ranking differs outside score ties"
        assert not np.isin(ix[u], ex).any()


def test_topn_fused_select_edge_cases(monkeypatch):
    """The fused select (group maxima -> threshold -> candidates) against the exact route and the
    oracle: items sorted by popularity (the worst case for group maxima), an item count that is not a
    multiple of the tile, unsorted exclusion lists, and massive score ties (candidate overflow ->
    exact fallback)."""
    from poismf_b200 import _lib, c_funs
    rng = np.random.default_rng(21)
    k, n_items, n_users, n_top = 40, 30_001, 260, 50
    A = np.ascontiguousarray(rng.gamma(0.5, 0.5, size=(n_users, k)).astype(np.float32))
    pop = np.sort(rng.pareto(1.5, n_items))[::-1].astype(np.float32)          # descending popularity
    B = np.ascontiguousarray((rng.gamma(2.0, 0.5, size=(n_items, k)) * pop[:, None]).astype(np.float32))
    lens = rng.integers(0, 200, n_users)
    ptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    eix = np.concatenate([rng.choice(400, int(m), replace=False) for m in lens]).astype(np.uint64)  # unsorted, popular
    _lib.topn_stats(reset=True)
    ix, sc = c_funs._topN_batch(A, B, excl_ptr=ptr, excl_ix=eix, top_n=n_top, output_score=True)
    n_tc, n_redo = _lib.topn_stats(reset=True)
    assert n_tc == n_users and n_redo <= 0.1 * n_users
    monkeypatch.setenv("POISMF_B200_TOPN_EXACT", "1")                          # exact route
    ix2, sc2 = c_funs._topN_batch(A, B, excl_ptr=ptr, excl_ix=eix, top_n=n_top, output_score=True)
    monkeypatch.delenv("POISMF_B200_TOPN_EXACT")
    assert np.array_equal(sc, sc2)
    assert all((sc[u] == sc[u][t]).sum() > 1 for u, t in zip(*np.nonzero(ix != ix2)))
    orc = Restatement(np.float32)
    for u in range(0, n_users, 13):
        ex = eix[int(ptr[u]):int(ptr[u + 1])]
        rc, ix_r, sc_r = orc.topN(np.ascontiguousarray(A[u]), B, n_top, exclude=ex if ex.size else None)
        assert rc == 0 and np.array_equal(sc[u], sc_r) and not np.isin(ix[u], ex).any()
    # ties: every item scores the same for every user -> more candidates than slots -> exact fallback
    Bt = np.ascontiguousarray(np.tile(B[:1], (n_items, 1)))
    _lib.topn_stats(reset=True)
    ix3, sc3 = c_funs._topN_batch(A[:8], Bt, top_n=n_top, output_score=True)
    assert _lib.topn_stats(reset=True)[1] == 8
    assert all(len(set(r.tolist())) == n_top for r in ix3) and (sc3 == sc3[:, :1]).all()


@pytest.mark.parametrize("n_items,n_top,n_users", [(300, 10, 48), (300, 100, 48), (1000, 10, 48), (1000, 100, 48),
                                                   (5000, 10, 48), (5000, 100, 48), (5000, 100, 256), (1328, 10, 48),
                                                   (1329, 10, 48), (6384, 100, 48), (6385, 100, 48)])
def test_topn_routes_around_fused_threshold(n_items, n_top, n_users, monkeypatch, capfd):
    """Item counts around the fused select's threshold (the items must hold 2 M candidate groups of 16, M =
    max(2 N, N + 32)).  At and above it every user goes through the fused select; below it the TF32 scores are
    sorted when there are >= 256 users and n k >= 2 M (k + 32), else the call is exact (no user on the tensor
    cores).  Host arrays and a fit handle's resident factors, with and without exclusion lists: scores are the
    oracle's bits, ids equal outside score ties, no excluded id."""
    from poismf_b200 import _lib, c_funs
    from poismf_b200.device import DeviceFit
    rng = np.random.default_rng(n_items + n_top + n_users)
    k = 24
    A = np.ascontiguousarray(rng.gamma(0.5, 0.5, size=(n_users, k)).astype(np.float32))
    B = np.ascontiguousarray(rng.gamma(0.5, 0.5, size=(n_items, k)).astype(np.float32))
    lens = rng.integers(0, min(60, n_items - n_top), n_users)
    ptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    eix = np.concatenate([rng.choice(n_items, int(m), replace=False) for m in lens]).astype(np.uint64)
    fused = -(-n_items // 16) >= 2 * max(2 * n_top, n_top + 32)
    on_tc = fused or (n_users >= 256 and n_items * k >= 2 * min(n_items, max(2 * n_top, n_top + 32)) * (k + 32))
    monkeypatch.setenv("POISMF_B200_TOPN_TRACE", "1")          # the fused route's phases include "work arrays"
    orc = Restatement(np.float32)
    fit = DeviceFit(n_users, n_items, k, np.float32)
    try:
        fit.set_factors(A, B)
        for excl in (dict(), dict(excl_ptr=ptr, excl_ix=eix)):
            for rank in (lambda: c_funs._topN_batch(A, B, top_n=n_top, output_score=True, **excl),
                         lambda: fit.topN(top_n=n_top, output_score=True, **excl)):
                capfd.readouterr()
                _lib.topn_stats(reset=True)
                ix, sc = rank()
                n_tc, _ = _lib.topn_stats(reset=True)
                assert n_tc == (n_users if on_tc else 0)
                assert ("[topN] work arrays" in capfd.readouterr().err) == fused
                for u in range(0, n_users, 1 if n_users <= 48 else 5):
                    ex = eix[int(ptr[u]):int(ptr[u + 1])] if excl else np.empty(0, np.uint64)
                    rc, ix_r, sc_r = orc.topN(np.ascontiguousarray(A[u]), B, n_top, exclude=ex if ex.size else None)
                    assert rc == 0 and np.array_equal(sc[u], sc_r)
                    assert all((sc_r == sc_r[t]).sum() > 1 for t in np.nonzero(ix[u] != ix_r)[0])
                    assert not np.isin(ix[u], ex).any()
    finally:
        fit.close()


@pytest.mark.parametrize("dtype", DTYPES)
def test_topn_against_resident_factors(dtype):
    """pmf_b200_topN_fitted ranks against the factors held by a fit handle: same ids and scores as the
    stateless batched entry on the same host arrays, same argument checks; after a sweep it ranks with the
    UPDATED factors."""
    from poismf_b200 import _lib, c_funs
    from poismf_b200.device import DeviceFit
    csr, csc, A0, B0, k = problem("pl2k", dtype)
    rng = np.random.default_rng(3)
    dimA, dimB = A0.shape[0], B0.shape[0]
    users = rng.choice(dimA, 40, replace=False).astype(np.uint64)
    lens = rng.integers(0, 5, users.shape[0])
    ptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    eix = np.concatenate([rng.choice(dimB, int(m), replace=False) for m in lens] + [np.empty(0, np.int64)]).astype(np.uint64)
    fit = DeviceFit(dimA, dimB, k, dtype)
    fit.set_factors(A0, B0)
    for kw in (dict(), dict(users=users, excl_ptr=ptr, excl_ix=eix)):
        ix, sc = fit.topN(top_n=7, output_score=True, **kw)
        ix2, sc2 = c_funs._topN_batch(A0, B0, top_n=7, output_score=True, **kw)
        assert np.array_equal(sc, sc2)
        assert all((sc[u] == sc[u][t]).sum() > 1 for u, t in zip(*np.nonzero(ix != ix2)))
    with pytest.raises(ValueError):
        fit.topN(users=np.array([dimA], np.uint64), top_n=3)
    with pytest.raises(ValueError):
        fit.topN(top_n=dimB + 1)
    # after a fit the handle ranks with the fitted factors
    fit.set_matrix(_lib.SIDE_CSR, *csr)
    fit.set_matrix(_lib.SIDE_CSC, *csc)
    fit.sweeps(_lib.make_params("cg", l2_reg=1e3, maxupd=5, numiter=2, limit_step=True))
    A, B = fit.get_factors()
    ix, sc = fit.topN(users=users, top_n=5, output_score=True)
    ix2, sc2 = c_funs._topN_batch(A, B, users=users, top_n=5, output_score=True)
    assert np.array_equal(sc, sc2) and not np.array_equal(A, A0)
    assert all((sc[u] == sc[u][t]).sum() > 1 for u, t in zip(*np.nonzero(ix != ix2)))


def test_topn_candidates_clustered_in_few_tiles():
    """Every user's best items are the same 800 consecutive ids (6 item tiles): the sampled threshold pass sees
    only two of those tiles, so all 800 become candidates and they land in a handful of the per-CTA candidate
    regions — the regions' slack must hold them (no exact fallback), rankings equal the oracle's."""
    from poismf_b200 import _lib, c_funs
    rng = np.random.default_rng(8)
    k, n_items, n_users, n_top = 24, 30_000, 200, 10
    A = np.ascontiguousarray(rng.gamma(2.0, 0.5, size=(n_users, k)).astype(np.float32))
    B = rng.gamma(2.0, 0.05, size=(n_items, k))
    B[:800] *= 40.0
    B = np.ascontiguousarray(B.astype(np.float32))
    _lib.topn_stats(reset=True)
    ix, sc = c_funs._topN_batch(A, B, top_n=n_top, output_score=True)
    n_tc, n_redo = _lib.topn_stats(reset=True)
    assert n_tc == n_users and n_redo == 0, (n_tc, n_redo)
    assert (ix < 800).all()
    orc = Restatement(np.float32)
    for u in range(0, n_users, 17):
        rc, ix_r, sc_r = orc.topN(np.ascontiguousarray(A[u]), B, n_top)
        assert rc == 0 and np.array_equal(sc[u], sc_r)
        assert all((sc_r == sc_r[t]).sum() > 1 for t in np.nonzero(ix[u] != ix_r)[0])


def test_topn_threshold_select_crowded_bin(monkeypatch):
    """More group maxima in the threshold's histogram bin than the select's shared-memory list holds (70k items
    whose scores lie within 0.1 % of each other): the threshold falls back to the bin's lower edge, every item
    becomes a candidate, the candidate lists overflow and the users are redone exactly — same result as the
    exact scorer."""
    from poismf_b200 import _lib, c_funs
    rng = np.random.default_rng(5)
    k, n_items, n_users, n_top = 32, 70_000, 40, 25
    A = np.ascontiguousarray(rng.gamma(2.0, 0.5, size=(n_users, k)).astype(np.float32))
    base = rng.gamma(2.0, 0.5, size=(1, k))
    B = np.ascontiguousarray((base * (1.0 + 1e-3 * rng.random((n_items, 1)))).astype(np.float32))
    _lib.topn_stats(reset=True)
    ix, sc = c_funs._topN_batch(A, B, top_n=n_top, output_score=True)
    n_tc, n_redo = _lib.topn_stats(reset=True)
    assert n_tc == n_users and n_redo == n_users
    monkeypatch.setenv("POISMF_B200_TOPN_EXACT", "1")
    ix2, sc2 = c_funs._topN_batch(A, B, top_n=n_top, output_score=True)
    assert np.array_equal(sc, sc2)
    assert all((sc[u] == sc[u][t]).sum() > 1 for u, t in zip(*np.nonzero(ix != ix2)))


@pytest.mark.parametrize("dtype", DTYPES)
def test_very_heavy_columns_streaming_clusters(dtype):
    """A handful of items with ~1e4 non-zeros each: every column is a 16-CTA cluster row whose slices
    are streamed from L2 (the cap-0 bin) in double, staged-or-streamed in float.  cg and tncg, fast
    numerics, against the oracle's log-likelihood; pg bit-exact in strict mode (single-CTA path)."""
    from poismf_b200.synth import init_factors, powerlaw_counts
    dimA, dimB, k = 30_000, 40, 50
    csr, csc = powerlaw_counts(dimA, dimB, 500_000, alpha_a=0.3, alpha_b=0.3, dtype=dtype, seed=9)
    assert np.diff(csc[1].astype(np.int64)).max() > 8_000
    A0, B0 = init_factors(dimA, dimB, k, dtype=dtype)
    orc = Restatement(dtype)
    for method, kw, gate in (("cg", dict(l2_reg=1e3, maxupd=5, numiter=2, limit_step=True), 1e-4),
                             ("tncg", dict(l2_reg=1e2, maxupd=15 * k, numiter=1), 1e-4)):
        Ar, Br = _oracle(dtype, csr, csc, A0, B0, method, kw)
        A, B = A0.copy(), B0.copy()
        assert run_device(csr, csc, A, B, method, kw) == 0
        assert np.isfinite(A).all() and np.isfinite(B).all() and (A >= 0).all() and (B >= 0).all()
        l_ref, l_dev = orc.llk(Ar, Br, csr), orc.llk(A, B, csr)
        g = gate if dtype == np.float64 else 2e-2
        assert abs(l_dev - l_ref) <= g * abs(l_ref), (method, l_dev, l_ref)
    kw = dict(l2_reg=1e6, step_size=1e-6, maxupd=2, numiter=2)
    Ar, Br = _oracle(dtype, csr, csc, A0, B0, "pg", kw)
    A, B = A0.copy(), B0.copy()
    assert run_device(csr, csc, A, B, "pg", kw, flags=FLAG_STRICT) == 0
    assert np.array_equal(A, Ar) and np.array_equal(B, Br)
    A, B = A0.copy(), B0.copy()
    assert run_device(csr, csc, A, B, "pg", kw) == 0
    gate = 1e-5 if dtype == np.float64 else 1e-3
    assert row_rel_err(A, Ar).max() <= gate and row_rel_err(B, Br).max() <= gate


# ---------------------------------------------------------------- point queries (VERDICT r1: uploads per call)
def test_topn_batch_rejects_invalid_ids():
    """Ids outside the matrices, non-monotone offsets and users left with fewer than n_top items return 2
    (ValueError), as the single-user entry does (src/topN.c:121-128) — nothing is read out of bounds."""
    from poismf_b200 import c_funs
    rng = np.random.default_rng(2)
    A = np.ascontiguousarray(rng.gamma(1, 1, size=(20, 8)).astype(np.float32))
    B = np.ascontiguousarray(rng.gamma(1, 1, size=(300, 8)).astype(np.float32))
    ok_ptr = np.array([0, 2, 4], np.uint64); ok_ix = np.array([1, 5, 7, 9], np.uint64)
    c_funs._topN_batch(A, B, users=np.array([0, 19], np.uint64), excl_ptr=ok_ptr, excl_ix=ok_ix, top_n=5)
    with pytest.raises(ValueError):
        c_funs._topN_batch(A, B, users=np.array([0, 20], np.uint64), top_n=5)
    with pytest.raises(ValueError):
        c_funs._topN_batch(A, B, users=np.array([0, 1], np.uint64), excl_ptr=ok_ptr, excl_ix=np.array([1, 5, 7, 300], np.uint64), top_n=5)
    with pytest.raises(ValueError):
        c_funs._topN_batch(A, B, users=np.array([0, 1], np.uint64), excl_ptr=np.array([0, 3, 2], np.uint64), excl_ix=ok_ix, top_n=5)
    with pytest.raises(ValueError):
        c_funs._topN_batch(A, B, users=np.array([0], np.uint64), excl_ptr=np.array([0, 298], np.uint64),
                           excl_ix=np.arange(298, dtype=np.uint64), top_n=5)


def test_resident_item_factors_between_topn_calls(monkeypatch):
    """POISMF_B200_CACHE_FACTORS=1 keeps the padded item factors on the device for the next call on the same
    array: same results as without, and an in-place edit of the array is noticed."""
    from poismf_b200 import _lib, c_funs
    rng = np.random.default_rng(4)
    B = np.ascontiguousarray(rng.gamma(1, 1, size=(5000, 50)).astype(np.float32))
    A = np.ascontiguousarray(rng.gamma(1, 1, size=(30, 50)).astype(np.float32))
    none = np.empty(0, np.uint64)
    want = [c_funs._call_topN(np.ascontiguousarray(A[u]), B, none, none, top_n=7, output_score=True) for u in range(5)]
    monkeypatch.setenv("POISMF_B200_CACHE_FACTORS", "1")
    for rep in range(2):
        for u in range(5):
            ix, sc = c_funs._call_topN(np.ascontiguousarray(A[u]), B, none, none, top_n=7, output_score=True)
            assert np.array_equal(ix, want[u][0]) and np.array_equal(sc, want[u][1])
    B *= 0.5                                                  # same pointer, new contents
    ix, sc = c_funs._call_topN(np.ascontiguousarray(A[0]), B, none, none, top_n=7, output_score=True)
    assert np.array_equal(sc, want[0][1] * 0.5)
    monkeypatch.delenv("POISMF_B200_CACHE_FACTORS")
    _lib.lib().pmf_b200_release_cache()


# ---------------------------------------------------------------- lock-step path vs per-row teams
def test_lockstep_path_matches_per_row_teams(monkeypatch):
    """The heaviest rows solved together (dense_rows.cuh: TMA-tiled passes over all their non-zeros) against
    the same rows on per-row cluster teams (PMF_FLAG_NO_LOCKSTEP): same algorithm, different summation
    order.  Per-row objective of the heavy rows agrees to 1e-4 on 90 % of them (never worse in the median), the other side
    (no heavy rows, identical inputs) is bit-identical after the first half-sweep, and the path is
    reproducible run to run.  Forced on for every heavy row here (POISMF_B200_DENSE_MIN_TOTAL=0)."""
    from conftest import row_objectives
    from poismf_b200 import SIDE_CSC, make_params
    from poismf_b200.device import DeviceFit
    from poismf_b200.synth import init_factors, powerlaw_counts
    monkeypatch.setenv("POISMF_B200_DENSE_MIN_TOTAL", "0")
    dtype = np.float32
    dimA, dimB, k = 30_000, 40, 50
    csr, csc = powerlaw_counts(dimA, dimB, 500_000, alpha_a=0.3, alpha_b=0.3, dtype=dtype, seed=9)
    assert np.diff(csc[1].astype(np.int64)).min() > 4096          # every column is a lock-step row
    A0, B0 = init_factors(dimA, dimB, k, dtype=dtype)
    hp = dict(l2_reg=1e3, maxupd=5, limit_step=True)
    outs = {}
    for name, flags in (("lock", 0), ("lock2", 0), ("rows", FLAG_NO_LOCKSTEP)):
        fit = DeviceFit(dimA, dimB, k, dtype)
        fit.set_csr_csc(csr, csc); fit.set_factors(A0, B0)
        fit.half_sweep(SIDE_CSC, make_params("cg", numiter=1, flags=flags, **hp), 1e-7, 1.0)
        fit.sync()
        prof_names = None
        outs[name] = fit.get_factors()[1]
        fit.close()
    assert np.array_equal(outs["lock"], outs["lock2"])             # reproducible
    assert not np.array_equal(outs["lock"], outs["rows"])          # ... and really a different path
    f_lock = row_objectives(outs["lock"], A0, csc, hp["l2_reg"])
    f_rows = row_objectives(outs["rows"], A0, csc, hp["l2_reg"])
    d = (f_lock - f_rows) / np.abs(f_rows)
    # (one row in 40 may take another line-search trial: float cg is chaotic in the rounding)
    assert np.abs(d).max() <= 2e-2 and np.quantile(np.abs(d), 0.9) <= 1e-4 and np.median(d) <= 1e-6, \
        (float(np.abs(d).max()), float(np.quantile(np.abs(d), 0.9)), float(np.median(d)))
    # full fits agree at the log-likelihood level
    kw = dict(numiter=3, **hp)
    A1, B1 = A0.copy(), B0.copy(); assert run_device(csr, csc, A1, B1, "cg", kw) == 0
    A2, B2 = A0.copy(), B0.copy(); assert run_device(csr, csc, A2, B2, "cg", kw, flags=FLAG_NO_LOCKSTEP) == 0
    orc = Restatement(dtype)
    l1, l2 = orc.llk(A1, B1, csr), orc.llk(A2, B2, csr)
    assert abs(l1 - l2) <= 1e-4 * abs(l2), (l1, l2)
