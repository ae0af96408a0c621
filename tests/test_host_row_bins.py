"""CPU checks of the per-bin half-sweep tests (tests/row_bins.py, tests/test_gpu_row_bins.py): the problem
builder gives exactly the requested row lengths, and the per-bin gates pass the restatement's own builds but
fail results that carry a kernel-like bug in one bin."""
import numpy as np
import pytest

import row_bins as rb

# bins of the kind the planner makes: (kind, lo, hi] row lengths, the last one open-ended
TABLE = [("a", 0, 16), ("b", 16, 64), ("c", 64, 256), ("d", 256, 1024), ("e", 1024, None)]


def _lengths(seed=1):
    lengths = np.array(rb.bin_lengths(TABLE, seed=seed, top=3000) + [0, 0, 0])
    np.random.default_rng(seed).shuffle(lengths)
    return lengths


@pytest.mark.parametrize("side", [rb.SIDE_CSC, rb.SIDE_CSR])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_builder_exact_lengths(dtype, side):
    lengths = _lengths()
    prob = rb.build_problem(lengths, side, 3, dtype, seed=2)
    vals, ptr, ind = prob["mat"]
    assert np.array_equal(np.diff(ptr.astype(np.int64)), lengths)
    other = prob["F"].shape[0]
    assert other >= lengths.max()
    for r in range(lengths.shape[0]):
        ids = ind[int(ptr[r]):int(ptr[r + 1])]
        assert np.all(np.diff(ids.astype(np.int64)) > 0) and (ids.shape[0] == 0 or ids[-1] < other)
    assert vals.dtype == dtype and (vals >= 1).all()
    # the other orientation is the transpose, entry for entry
    import scipy.sparse as sp
    t = prob["csr"] if side == rb.SIDE_CSC else prob["csc"]
    X = sp.csr_matrix((vals, ind.astype(np.int64), ptr.astype(np.int64)), shape=(lengths.shape[0], other))
    Y = sp.csr_matrix((t[0], t[2].astype(np.int64), t[1].astype(np.int64)), shape=(other, lengths.shape[0]))
    assert (X.T != Y).nnz == 0
    assert np.array_equal(np.diff(t[1].astype(np.int64)), np.bincount(ind.astype(np.int64), minlength=other))
    # the updated and fixed factors sit where DeviceFit.set_factors expects them
    A0, B0 = prob["A0"], prob["B0"]
    assert (B0 if side == rb.SIDE_CSC else A0) is prob["M0"] and A0.shape[0] == prob["csr"][1].shape[0] - 1
    assert B0.shape[0] == prob["csc"][1].shape[0] - 1


def test_bin_table_from_profile():
    prof = [dict(side=1, block_team=101, cap=16), dict(side=1, block_team=1, cap=900),
            dict(side=1, block_team=2, cap=800), dict(side=1, block_team=16, cap=800),
            dict(side=1, block_team=16, cap=0), dict(side=0, block_team=-32, cap=24)]
    assert rb.bin_table(prof, 1) == [("regtile1w:16", 0, 16), ("cta:900", 16, 900), ("cluster2", 900, 1600),
                                     ("cluster16", 1600, 12800), ("streaming", 12800, None)]
    prof.insert(0, dict(side=1, block_team=200, cap=0))
    assert rb.bin_table(prof, 1, dense_min=1000)[1:] == [("cta:900", 16, 900), ("cluster2", 900, 999),
                                                          ("lockstep", 999, None)]
    assert rb.bin_table(prof, 0) == [("warp32:24", 0, 24)]


_PROBS = {}


def _problem(dtype, k, side):
    key = (dtype, k, side)
    if key not in _PROBS:
        lengths = _lengths()
        _PROBS[key] = (lengths, rb.build_problem(lengths, side, k, dtype, seed=3))
    return _PROBS[key]


def _drop_last(mat, rows):
    """The sub-matrix of `rows` with each row's last non-zero removed."""
    vals, ptr, ind = mat
    n = np.diff(ptr.astype(np.int64))[rows]
    keep = np.maximum(n - 1, 0)
    sel = np.concatenate([np.arange(int(ptr[r]), int(ptr[r]) + int(m)) for r, m in zip(rows, keep)] + [np.zeros(0, np.int64)])
    sub_ptr = np.zeros(rows.shape[0] + 1, np.uint64)
    sub_ptr[1:] = np.cumsum(keep)
    return np.ascontiguousarray(vals[sel]), sub_ptr, np.ascontiguousarray(ind[sel])


CASES = [(v, False) for v in rb.VARIANTS] + [(v, True) for v in ("pg", "cg1", "cg5_nolimit", "tncg2", "tncg")]


@pytest.mark.parametrize("side", [rb.SIDE_CSC, rb.SIDE_CSR])
@pytest.mark.parametrize("variant,strict", CASES)
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_gates_have_teeth(dtype, variant, strict, side):
    """The unmutated stand-in passes every bin's gate; each mutation, applied to one bin at a time, fails that
    bin's gate: (1) the rows computed without their last non-zero (an off-by-one in a tile), (2) component
    k-1 left at its value before the update (a missed chunk), (3) float64 only: the column sums perturbed by
    a relative ~1e-6 (a float intermediate in a double kernel).
    Not asserted where the gate cannot see the mutation among the restatement's own rounding spread:
      * (1) where the gate is the objective after 5 fast iterations in float32, or after 20 of tncg: one
        non-zero fewer barely moves the full objective; the same kernels are gated by coordinates after one
        (cg) or two (tncg) iterations.  Also (1) for float32 cg without limit_step, whose few non-zero
        outputs move by ~1e-5 on rows of 256+ non-zeros.
      * any mutation for fast float32 tncg after 20 iterations (~3 % from S in the median of some bins) and for
        fast float32 cg with limit_step after 5 (the fast builds stall on rounding residuals above the bound,
        ~20 % from S in the median): there the objective gate only bounds gross errors.
      * (3) for tncg, whose branchy line search already moves half the rows of the fast restatement by
        1e-8..1e-4, and for pg on the A side, where the column sums enter scaled by the step twice (Q1)."""
    from oracle.oracle import Restatement
    k = 33
    lengths, prob = _problem(dtype, k, side)
    method, hp, _ = rb.VARIANTS[variant]
    mode = rb.gate_mode(variant, strict, dtype)
    ref = rb.references(method, hp, prob, dtype)
    stand_in = "S" if strict else "Fh"
    orc = Restatement(dtype, fast=not strict)
    groups = rb.group_rows(lengths, TABLE)
    base = dict(ref, M0=prob["M0"])
    fails, stats = rb.check_bins(mode, dtype, dict(base, D=ref[stand_in]), groups, prob, hp)
    assert not fails, (fails, stats)
    # the update is not trivial: most rows move, and not all end at zero
    moved = rb.row_err(ref["T"], prob["M0"], prob["M0"])[lengths > 0]
    assert np.median(moved) > 1e-3 and (ref["T"] == 0).mean() < 0.97

    mutants = {}
    csum = prob["F"].astype(np.float64).sum(0)
    if np.dtype(dtype) == np.float64 and method != "tncg" and not (method == "pg" and side == rb.SIDE_CSR):
        mutants["colsum"] = rb.oracle_half_sweep(orc, method, hp, prob, l1_extra=1e-6 * float(csum.mean()))
    for kind, rows in groups.items():
        D1 = ref[stand_in].copy()
        D1[rows] = rb.oracle_half_sweep(orc, method, hp, prob, M0=prob["M0"][rows], mat=_drop_last(prob["mat"], rows))
        D2 = ref[stand_in].copy()
        D2[rows, k - 1] = prob["M0"][rows, k - 1]
        f32 = np.dtype(dtype) == np.float32
        gross_only = mode == "fast_obj_stall" or (f32 and mode == "fast_tn")
        cases = {} if gross_only else dict(chunk=D2)
        if not (mode in ("fast_tn", "fast_obj_stall") or (mode == "fast_obj" and f32) or (variant == "cg1_nolimit" and f32)):
            cases["last_nnz"] = D1
        if "colsum" in mutants:
            D3 = ref[stand_in].copy()
            D3[rows] = mutants["colsum"][rows]
            cases["colsum"] = D3
        for name, D in cases.items():
            fails, stats = rb.check_bins(mode, dtype, dict(base, D=D), groups, prob, hp)
            assert any(f.startswith(kind + ":") for f in fails), (name, kind, stats[kind])
