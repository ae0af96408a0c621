"""CPU tests of the checkers: the plain-C restatement against (a) the reference itself
(oracle/_ref, when it has been built here) and (b) the committed golden outputs of the
reference (always).  Bit-exact: both are compiled -O2 -ffp-contract=off with sequential BLAS."""
import numpy as np
import pytest

from conftest import CASES, FM_CASES, FS_CASES, FS_ROWS, fm_hyper, fm_problem, fs_row, golden, hyper, problem
from oracle.oracle import Ref, Restatement

GOLD = golden()
DTYPES = [np.float64, np.float32]


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("prob", ["readme", "ragged"])
@pytest.mark.parametrize("case", list(CASES))
def test_restatement_matches_golden(dtype, prob, case):
    csr, csc, A0, B0, k = problem(prob, dtype)
    name = np.dtype(dtype).name
    chk = GOLD[f"{prob}/{name}/csr_checksum"]
    assert chk[2] == csr[0].shape[0] and chk[0] == csr[0].astype(np.float64).sum(), "synthetic inputs drifted"
    method, kw = hyper(case, k)
    A, B = A0.copy(), B0.copy()
    assert Restatement(dtype).run_poismf(A, B, csr, csc, method, **kw) == 0
    assert np.array_equal(A, GOLD[f"{prob}/{name}/{case}/A"])
    assert np.array_equal(B, GOLD[f"{prob}/{name}/{case}/B"])


@pytest.mark.skipif(not Ref.available(), reason="oracle/_ref not built (needs /root/reference)")
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("case", list(CASES))
def test_restatement_matches_reference_build(dtype, case):
    csr, csc, A0, B0, k = problem("pl2k", dtype)
    method, kw = hyper(case, k)
    A1, B1, A2, B2 = A0.copy(), B0.copy(), A0.copy(), B0.copy()
    assert Ref(dtype).run_poismf(A1, B1, csr, csc, method, **kw) == 0
    assert Restatement(dtype).run_poismf(A2, B2, csr, csc, method, **kw) == 0
    assert np.array_equal(A1, A2) and np.array_equal(B1, B2)


@pytest.mark.parametrize("dtype", DTYPES)
def test_predict_and_topn_match_golden(dtype):
    name = np.dtype(dtype).name
    csr, csc, A0, B0, k = problem("readme", dtype)
    rng = np.random.default_rng(3)
    ixA = rng.integers(0, A0.shape[0], 257).astype(np.uint64)
    ixB = rng.integers(0, B0.shape[0], 257).astype(np.uint64)
    orc = Restatement(dtype)
    assert np.array_equal(orc.predict_multiple(A0, B0, ixA, ixB), GOLD[f"predict/{name}"])
    Brand = np.ascontiguousarray(rng.gamma(1, 1, size=B0.shape).astype(dtype))
    rc, ix, sc = orc.topN(np.ascontiguousarray(A0[3]), Brand, 10)
    assert rc == 0 and np.array_equal(sc, GOLD[f"topn/{name}/score"]) and np.array_equal(ix, GOLD[f"topn/{name}/ix"])
    excl = np.arange(0, 1000, 7, dtype=np.uint64)
    rc, ix, sc = orc.topN(np.ascontiguousarray(A0[3]), Brand, 10, exclude=excl)
    assert rc == 0 and np.array_equal(sc, GOLD[f"topn_excl/{name}/score"])
    assert np.array_equal(ix, GOLD[f"topn_excl/{name}/ix"]) and not np.isin(ix, excl).any()


def test_topn_argument_checks():
    orc = Restatement(np.float64)
    B = np.ones((10, 3)); a = np.ones(3)
    assert orc.topN(a, B, 0)[0] == 2                                    # n_top == 0
    assert orc.topN(a, B, 3, include=[1, 2, 3], exclude=[4])[0] == 2    # both lists
    assert orc.topN(a, B, 5, exclude=list(range(6)))[0] == 2            # n_exclude > n - n_top


def test_llk_matches_numpy():
    csr, csc, A0, B0, k = problem("readme", np.float64)
    orc = Restatement(np.float64)
    rows = np.repeat(np.arange(A0.shape[0]), np.diff(csr[1].astype(np.int64)))
    pred = np.einsum("ij,ij->i", A0[rows], B0[csr[2].astype(np.int64)])
    want = (csr[0] * np.log(pred)).sum() - A0.sum(0) @ B0.sum(0)
    assert abs(orc.llk(A0, B0, csr) - want) <= 1e-9 * abs(want)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("case", list(FM_CASES))
def test_factors_multiple_restatement(dtype, case):
    """factors_multiple (src/pred.c:66-199): restatement == committed reference outputs (README shape)
    and == the reference build on a power-law shape when oracle/_ref is present."""
    name = np.dtype(dtype).name
    csr, B, Bsum, Amean, k = fm_problem("readme", dtype)
    method, kw = fm_hyper(case, k)
    rc, A = Restatement(dtype).factors_multiple(B, Bsum, Amean, csr, method, **kw)
    assert rc == 0 and np.array_equal(A, GOLD[f"factors_multiple/{name}/{case}"])
    if Ref.available(dtype):
        csr, B, Bsum, Amean, k = fm_problem("pl2k", dtype)
        method, kw = fm_hyper(case, k)
        rc1, A1 = Ref(dtype).factors_multiple(B, Bsum, Amean, csr, method, **kw)
        rc2, A2 = Restatement(dtype).factors_multiple(B, Bsum, Amean, csr, method, **kw)
        assert rc1 == 0 and rc2 == 0 and np.array_equal(A1, A2)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("case", list(FS_CASES))
def test_factors_single_restatement(dtype, case):
    """factors_single (src/pred.c:201-304): restatement == committed reference outputs, == the reference
    build when present, and == factors_multiple on the same row where the two share their arithmetic."""
    name = np.dtype(dtype).name
    csr, B, Bsum, Amean, k = fm_problem("readme", dtype)
    kw = FS_CASES[case]
    orc = Restatement(dtype)
    got = [orc.factors_single(*fs_row(csr, r), B, Bsum, Amean, **kw)[1] for r in FS_ROWS]
    got.append(orc.factors_single(np.empty(0, dtype), np.empty(0, np.uint64), B, Bsum, Amean, **kw)[1])
    assert np.array_equal(np.stack(got), GOLD[f"factors_single/{name}/{case}"])
    assert not got[-1].any()                                     # empty row -> zeros (:212-215)
    if Ref.available(dtype):
        for r in FS_ROWS:
            c, ix = fs_row(csr, r)
            assert np.array_equal(Ref(dtype).factors_single(c, ix, B, Bsum, Amean, **kw)[1],
                                  orc.factors_single(c, ix, B, Bsum, Amean, **kw)[1])
    if "l1_new" not in kw:      # same solve as one row of factors_multiple(tncg)
        rc, A = orc.factors_multiple(B, Bsum, Amean, csr, "tncg", l2_reg=kw.get("l2_reg", 1e5),
                                     w_mult=kw.get("w_mult", 1.0), maxupd=kw.get("maxupd", 20),
                                     reuse_mean=kw.get("reuse_mean", True))
        for j, r in enumerate(FS_ROWS):
            assert np.array_equal(A[r], got[j])


@pytest.mark.skipif(not Ref.available(), reason="oracle/_ref not built (needs /root/reference)")
@pytest.mark.parametrize("seed", range(24))
def test_restatement_matches_reference_on_random_small_problems(seed):
    """Random shapes (incl. k = 1, k not a multiple of 4, empty rows/columns), random method and
    hyper-parameters: the restatement and the reference build agree bit for bit in both dtypes."""
    from poismf_b200.synth import init_factors, powerlaw_counts
    rng = np.random.default_rng(1000 + seed)
    dimA, dimB = int(rng.integers(3, 70)), int(rng.integers(3, 90))
    k = int(rng.choice([1, 2, 3, 5, 8, 13]))
    nnz = int(rng.integers(1, dimA * dimB // 2 + 2))
    method = ["pg", "cg", "tncg"][seed % 3]
    kw = dict(l2_reg=float(10.0 ** rng.uniform(0, 5)), l1_reg=float(rng.choice([0.0, 0.3])),
              w_mult=float(rng.choice([1.0, 0.5, 2.5])), numiter=int(rng.integers(1, 4)))
    if method == "pg":
        kw.update(step_size=float(10.0 ** rng.uniform(-7, -3)), maxupd=int(rng.integers(1, 4)))
    elif method == "cg":
        kw.update(maxupd=int(rng.integers(1, 8)), limit_step=bool(rng.integers(0, 2)))
    else:
        kw.update(maxupd=int(rng.integers(1, 15 * k + 1)), reuse_prev=bool(rng.integers(0, 2)),
                  early_stop=bool(rng.integers(0, 2)))
    for dtype in DTYPES:
        csr, csc = powerlaw_counts(dimA, dimB, nnz, alpha_a=float(rng.uniform(0.2, 1.2)),
                                   alpha_b=float(rng.uniform(0.2, 1.2)), dtype=dtype, seed=seed)
        A0, B0 = init_factors(dimA, dimB, k, dtype=dtype, seed=seed)
        A1, B1, A2, B2 = A0.copy(), B0.copy(), A0.copy(), B0.copy()
        rc1 = Ref(dtype).run_poismf(A1, B1, csr, csc, method, **kw)
        rc2 = Restatement(dtype).run_poismf(A2, B2, csr, csc, method, **kw)
        assert rc1 == rc2 == 0
        assert np.array_equal(A1, A2, equal_nan=True) and np.array_equal(B1, B2, equal_nan=True), (method, kw)


@pytest.mark.skipif(not Ref.available(), reason="oracle/_ref not built (needs /root/reference)")
@pytest.mark.parametrize("seed", range(12))
def test_restatement_inference_paths_on_random_problems(seed):
    """factors_multiple, factors_single, predict_multiple and topN (include / exclude lists) of the
    restatement against the reference build on random inputs, bit for bit."""
    from poismf_b200.synth import powerlaw_counts
    rng = np.random.default_rng(2000 + seed)
    dimA, dimB = int(rng.integers(2, 40)), int(rng.integers(12, 120))
    k = int(rng.choice([1, 3, 4, 7, 10]))
    method = ["pg", "cg", "tncg"][seed % 3]
    for dtype in DTYPES:
        csr, _ = powerlaw_counts(dimA, dimB, int(rng.integers(1, dimA * dimB // 3 + 2)), dtype=dtype, seed=seed)
        B = np.ascontiguousarray(rng.gamma(1, 0.3, size=(dimB, k)).astype(dtype))
        Bsum = np.ascontiguousarray((B.sum(0) + 0.05).astype(dtype))
        Amean = np.ascontiguousarray(rng.gamma(1, 0.3, size=k).astype(dtype))
        kw = dict(l2_reg=float(10.0 ** rng.uniform(0, 4)), w_mult=float(rng.choice([1.0, 2.0])),
                  niter=int(rng.integers(1, 4)), maxupd=int(rng.integers(1, 6)), step_size=1e-4,
                  limit_step=bool(rng.integers(0, 2)), reuse_mean=bool(rng.integers(0, 2)))
        r1, A1 = Ref(dtype).factors_multiple(B, Bsum, Amean, csr, method, **kw)
        r2, A2 = Restatement(dtype).factors_multiple(B, Bsum, Amean, csr, method, **kw)
        assert r1 == r2 == 0 and np.array_equal(A1, A2, equal_nan=True), ("factors_multiple", method, kw)
        row = int(rng.integers(0, dimA))
        c, ix = fs_row(csr, row)
        fkw = dict(reuse_mean=kw["reuse_mean"], maxupd=int(rng.integers(1, 40)), l2_reg=kw["l2_reg"],
                   l1_new=float(rng.choice([0.0, 0.4])), l1_old=float(rng.choice([0.0, 0.1])), w_mult=kw["w_mult"])
        assert np.array_equal(Ref(dtype).factors_single(c, ix, B, Bsum, Amean, **fkw)[1],
                              Restatement(dtype).factors_single(c, ix, B, Bsum, Amean, **fkw)[1], equal_nan=True)
        A = np.ascontiguousarray(rng.gamma(1, 0.3, size=(dimA, k)).astype(dtype))
        ixA = rng.integers(0, dimA, 50).astype(np.uint64); ixB = rng.integers(0, dimB, 50).astype(np.uint64)
        assert np.array_equal(Ref(dtype).predict_multiple(A, B, ixA, ixB),
                              Restatement(dtype).predict_multiple(A, B, ixA, ixB))
        n_top = int(rng.integers(1, 8))
        a = np.ascontiguousarray(A[0])
        excl = np.sort(rng.choice(dimB, int(rng.integers(1, dimB - n_top)), replace=False)).astype(np.uint64)
        incl = rng.choice(dimB, int(rng.integers(n_top, dimB)), replace=False).astype(np.uint64)
        for lists in (dict(), dict(exclude=excl), dict(include=incl)):
            t1 = Ref(dtype).topN(a, B, n_top, **lists)
            t2 = Restatement(dtype).topN(a, B, n_top, **lists)
            assert t1[0] == t2[0] == 0 and np.array_equal(t1[2], t2[2])
            diff = np.nonzero(t1[1] != t2[1])[0]                      # ids may differ only inside score ties
            assert all((t1[2] == t1[2][j]).sum() > 1 for j in diff)

