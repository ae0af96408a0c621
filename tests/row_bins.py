"""Shared pieces of the per-bin half-sweep tests (tests/test_gpu_row_bins.py, tests/test_host_row_bins.py).

The device's planner (plan_rows, poismf_b200/csrc/row_plan.h) sends every row of the updated side to a kernel
chosen by its non-zero count.  These helpers build count matrices whose rows have exactly the requested
lengths, run the plain-C restatement's one-sided half-sweep (oracle_half_sweep) on the same inputs, and gate
a result per bin against the float64 truth.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from conftest import row_objectives

PG, CG, TNCG = 3, 2, 1
SIDE_CSR, SIDE_CSC = 0, 1


# ---- problem builder -----------------------------------------------------------------------------
def designed_rows(lengths, other, dtype, seed=0):
    """(values, indptr, indices) of a len(lengths) x other count matrix: row r has exactly lengths[r]
    non-zeros at distinct, ascending ids; values are counts >= 1."""
    lengths = np.asarray(lengths, dtype=np.int64)
    assert lengths.max(initial=0) <= other
    rng = np.random.default_rng(seed)
    ptr = np.zeros(lengths.shape[0] + 1, dtype=np.uint64)
    ptr[1:] = np.cumsum(lengths)
    ind = np.empty(int(ptr[-1]), dtype=np.uint64)
    for r, n in enumerate(lengths):
        if n:
            ind[int(ptr[r]):int(ptr[r + 1])] = np.sort(rng.choice(other, size=int(n), replace=False))
    vals = rng.geometric(0.5, size=ind.shape[0]).astype(dtype)
    return vals, ptr, ind


def transpose(mat, n_cols):
    """The same matrix in the other orientation (ids ascending within each row)."""
    import scipy.sparse as sp
    vals, ptr, ind = mat
    t = sp.csr_matrix((vals, ind.astype(np.int64), ptr.astype(np.int64)), shape=(ptr.shape[0] - 1, n_cols)).tocsc()
    t.sort_indices()
    return (np.ascontiguousarray(t.data.astype(vals.dtype)), t.indptr.astype(np.uint64), t.indices.astype(np.uint64))


def build_problem(lengths, side, k, dtype, seed=0, other=None):
    """Counts whose rows on `side` (the one the half-sweep updates) have exactly `lengths` non-zeros.
    Returns dict(csr, csc, A0, B0, M0, F, mat, side): M0 / F are the updated / fixed factors, `mat` the
    orientation whose rows are the updated rows (csc for the B half-sweep, csr for the A half-sweep)."""
    lengths = np.asarray(lengths, dtype=np.int64)
    other = int(max(other or 0, lengths.max(initial=0), 64))
    mat = designed_rows(lengths, other, dtype, seed)
    tr = transpose(mat, other)
    rng = np.random.default_rng(seed + 1)
    M0 = np.ascontiguousarray(rng.gamma(2.0, 0.15, size=(lengths.shape[0], k)).astype(dtype))
    F = np.ascontiguousarray(rng.gamma(2.0, 0.15, size=(other, k)).astype(dtype))
    if side == SIDE_CSC:
        csr, csc, A0, B0 = tr, mat, F, M0
    else:
        csr, csc, A0, B0 = mat, tr, M0, F
    return dict(csr=csr, csc=csc, A0=A0, B0=B0, M0=M0, F=F, mat=mat, side=side, lengths=lengths)


# ---- the cases -----------------------------------------------------------------------------------
# variant: (method, hyper-parameters, extra flags)
VARIANTS = {
    # (one step: at k = 1 a row the first step clips to zero has prediction 0 in the next, and the reference's
    # x / 0 makes it NaN)
    "pg": ("pg", dict(l2_reg=1e3, step_size=1e-6, maxupd=1), 0),
    # one or two iterations: deterministic up to line-search flips, gated by coordinates
    "cg1": ("cg", dict(l2_reg=1e4, maxupd=1, limit_step=True), 0),
    "cg1_nocache": ("cg", dict(l2_reg=1e4, maxupd=1, limit_step=True), 2),       # PMF_FLAG_NO_CACHED
    "cg1_nolimit": ("cg", dict(l2_reg=1e4, maxupd=1, limit_step=False), 0),
    "tncg2": ("tncg", dict(l2_reg=1e3, maxupd=2), 0),
    # more iterations: gated by the per-row objective
    "cg5": ("cg", dict(l2_reg=1e4, maxupd=5, limit_step=True), 0),
    "cg5_nocache": ("cg", dict(l2_reg=1e4, maxupd=5, limit_step=True), 2),
    "cg5_nolimit": ("cg", dict(l2_reg=1e4, maxupd=5, limit_step=False), 0),
    "tncg": ("tncg", dict(l2_reg=1e3, maxupd=20), 0),
}


def step_and_cdiv(method, hp, side, dtype):
    """The step / cnst_div a fit passes to the half-sweep of `side` in its first sweep
    (sharding.ShardedSweep.run): cdiv from the step at the start of the sweep, pg's step halved for A."""
    real = np.dtype(dtype).type
    step = real(hp.get("step_size", 1e-7))
    cdiv = float(real(1. / (1. + 2. * float(real(hp["l2_reg"])) * float(step))))
    if method == "pg" and side == SIDE_CSR:
        step = real(float(step) * 0.5)
    return float(step), cdiv


def oracle_half_sweep(orc, method, hp, prob, M0=None, mat=None, l1_extra=0.0):
    """One half-sweep of the restatement `orc` (oracle.Restatement) on prob's inputs cast to orc's dtype;
    returns the updated rows.  `mat` replaces the matrix, `l1_extra` is added to the column sums."""
    dt = orc.dtype
    side = prob["side"]
    mat = prob["mat"] if mat is None else mat
    M = np.array(prob["M0"] if M0 is None else M0, dtype=dt, order="C", copy=True)
    F = np.ascontiguousarray(prob["F"], dtype=dt)
    xv = np.ascontiguousarray(mat[0], dtype=dt)
    ptr, ind = np.ascontiguousarray(mat[1], np.uint64), np.ascontiguousarray(mat[2], np.uint64)
    step, _ = step_and_cdiv(method, hp, side, dt)
    r, sz, vp, i = orc.creal, C.c_size_t, C.c_void_p, C.c_int
    fn = orc.lib.oracle_half_sweep
    fn.restype = i
    fn.argtypes = [i, vp, vp, vp, vp, vp, sz, sz, sz, r, r, r, r, i, sz, i, i]
    p = lambda a: a.ctypes.data_as(vp)
    rc = fn({"pg": PG, "cg": CG, "tncg": TNCG}[method], p(M), p(F), p(xv), p(ptr), p(ind), M.shape[0], F.shape[0],
            M.shape[1], hp["l2_reg"], hp.get("l1_reg", 0.0) + l1_extra, hp.get("w_mult", 1.0), step,
            int(side == SIDE_CSR), hp["maxupd"], int(hp.get("limit_step", False)), int(hp.get("reuse_prev", False)))
    assert rc == 0
    return M


def references(method, hp, prob, dtype):
    """T: the strict restatement in float64 on the inputs upcast; S: the strict restatement in `dtype`;
    Fh: the restatement's fast build (-O3, FMA) in `dtype` (the rounding noise floor)."""
    from oracle.oracle import Restatement
    return dict(T=oracle_half_sweep(Restatement(np.float64), method, hp, prob),
                S=oracle_half_sweep(Restatement(dtype), method, hp, prob),
                Fh=oracle_half_sweep(Restatement(dtype, fast=True), method, hp, prob))


# ---- bins ----------------------------------------------------------------------------------------
LOCKSTEP = 200


def bin_kind(e):
    """Name of a profile entry (DeviceFit.get_profile): regtile / warp / cta / cluster / streaming / lockstep."""
    bt, cap = e["block_team"], e["cap"]
    if bt == LOCKSTEP:
        return "lockstep"
    if bt > 100:
        return f"regtile{bt - 100}w:{cap}"
    if bt < 0:
        return f"warp{-bt}:{cap}"
    if bt == 1:
        return "cta:0" if cap == 0 else f"cta:{cap}"
    return "streaming" if cap == 0 else f"cluster{bt}"


def bin_table(profile, side, dense_min=None):
    """[(kind, lo, hi)] from the profile of one side: row lengths in (lo, hi] go to the bin (hi = None: no
    upper bound).  The planner puts a row in the first bin whose cap x cluster size it fits; rows of at least
    `dense_min` non-zeros go to the lock-step path when it is on."""
    out, lo = [], 0
    for e in profile:
        if e["side"] != side or e["block_team"] == LOCKSTEP:
            continue
        bt, cap = e["block_team"], e["cap"]
        hi = None if cap == 0 else cap * (bt if 2 <= bt <= 16 else 1)
        if dense_min is not None and (hi is None or hi >= dense_min):
            out.append((bin_kind(e), lo, dense_min - 1))   # the rest of this bin, and the bins above, go lock-step
            break
        out.append((bin_kind(e), lo, hi))
        lo = hi if hi is not None else lo
    if dense_min is not None and any(e["side"] == side and e["block_team"] == LOCKSTEP for e in profile):
        out.append(("lockstep", dense_min - 1, None))
    return out


def probe_lengths(lmax):
    """Every length 1..600, then geometric (x1.08) up to lmax."""
    out = list(range(1, 601))
    v = 600.0
    while v < lmax:
        v = min(v * 1.08, lmax)
        out.append(int(v))
    return out


def bin_lengths(table, seed=0, top=None):
    """Lengths for a problem: per bin 1 (where it belongs to the bin), lo+1, the middle, cap-1 and cap, plus
    random lengths inside the bin, more for short rows; `top` bounds the open-ended last bin."""
    rng = np.random.default_rng(seed)
    out = []
    for kind, lo, hi in table:
        if hi is None:
            hi = top if top is not None else max(2 * lo, lo + 64)
        edges = {lo + 1, (lo + hi + 1) // 2, hi - 1, hi} | ({1} if lo == 0 else set())
        edges = [n for n in edges if lo < n <= hi]
        n_extra = int(np.clip(24000 // hi, 4, 40))
        out += edges + list(rng.integers(lo + 1, hi + 1, size=n_extra))
    return out


def group_rows(lengths, table):
    """{kind: row ids} of the non-empty rows by the (lo, hi] ranges of `table`."""
    out = {}
    for kind, lo, hi in table:
        sel = (lengths > lo) if hi is None else ((lengths > lo) & (lengths <= hi))
        out[kind] = np.nonzero(sel & (lengths > 0))[0]
    return out


# ---- gates ---------------------------------------------------------------------------------------
def row_err(X, Y, M0):
    """Per-row |X - Y| / max(|Y|, |M0|) in float64 (M0: the rows before the update; rows pg zeroed stay
    measured against the input's scale)."""
    X, Y, M0 = (np.asarray(a, dtype=np.float64) for a in (X, Y, M0))
    den = np.maximum(np.maximum(np.linalg.norm(Y, axis=1), np.linalg.norm(M0, axis=1)), 1e-300)
    return np.linalg.norm(X - Y, axis=1) / den


# coordinate tolerance per dtype: strict builds differ from each other by log() ulps at most; fast cg after one
# iteration is deterministic up to line-search flips
STRICT_TOL = {np.float32: 1e-5, np.float64: 1e-11}
CG1_TOL = {np.float32: 1e-5, np.float64: 1e-11}
# objective gates: the median relative excess over S may pass 4 x the fast restatement's by OBJ_MED; a row counts
# as worse beyond OBJ_WORSE.  (Fast cg with limit_step in float32 loses ~0.2 in the median against S by itself:
# the contracted update x + step d leaves the limiting coordinate a rounding residual above its bound, which
# stalls the next iteration.  That mode, "fast_obj_stall", is gated for gross errors only.)
OBJ_MED = {np.float32: 1e-4, np.float64: 1e-6}
OBJ_WORSE = {np.float32: 1e-4, np.float64: 1e-8}
# fast float64: rows further than this from T count, against the fast restatement's count
F64_TOL = 1e-11


def gate_mode(variant, strict, dtype):
    method, hp, _ = VARIANTS[variant]
    if strict:
        return "strict_pg" if method == "pg" else "strict_iter"
    if method == "pg":
        return "fast_pg"
    if variant in ("cg1", "cg1_nocache", "cg1_nolimit", "tncg2"):
        return "fast_cg1"
    if method == "cg" and hp["limit_step"] and np.dtype(dtype) == np.float32:
        return "fast_obj_stall"
    return "fast_tn" if method == "tncg" else "fast_obj"


def check_bins(mode, dtype, res, groups, prob, hp):
    """Per-bin gates of result D against the references (res: dict with D, T, S, Fh, M0 rows).
    Returns (failures, stats): failures is a list of strings (empty: every bin passes)."""
    dt = np.dtype(dtype).type
    D, T, S, Fh, M0 = (res[n] for n in ("D", "T", "S", "Fh", "M0"))
    lengths = prob["lengths"]
    fails, stats = [], {}
    assert np.isfinite(T).all(), "the float64 reference itself is not finite on this problem"
    # every row, whatever its bin
    if not np.isfinite(D).all() or (D < 0).any():
        fails.append("non-finite or negative output")
    empty = lengths == 0
    if D[empty].any():
        fails.append("empty rows not zero")
    eD, eS, eF = row_err(D, T, M0), row_err(S, T, M0), row_err(Fh, T, M0)
    need_obj = mode in ("fast_obj", "fast_obj_stall", "fast_tn")
    if need_obj:
        l2, w, l1 = hp["l2_reg"], hp.get("w_mult", 1.0), hp.get("l1_reg", 0.0)
        fD, fS, fF = (row_objectives(X, prob["F"], prob["mat"], l2, w=w, l1=l1) for X in (D, S, Fh))
    for kind, rows in groups.items():
        if rows.shape[0] == 0:
            continue
        n = rows.shape[0]
        st = dict(rows=int(n), lengths=[int(lengths[rows].min()), int(lengths[rows].max())])
        for nm, e in (("D", eD), ("S", eS), ("Fh", eF)):
            st[f"{nm}_max"] = float(e[rows].max())
            st[f"{nm}_p99"] = float(np.quantile(e[rows], 0.99))
        bad = []
        if mode == "strict_pg":
            nd = int((D[rows] != S[rows]).any(axis=1).sum())
            st["rows_not_bitwise_S"] = nd
            if nd:
                bad.append(f"{nd} rows differ from the strict restatement")
        elif mode == "strict_iter":
            nd = int((row_err(D[rows], S[rows], M0[rows]) > STRICT_TOL[dt]).sum())
            st["rows_off_S"] = nd
            if nd > max(1, int(0.002 * n)):
                bad.append(f"{nd} rows further than {STRICT_TOL[dt]} from the strict restatement")
        elif mode == "fast_pg":
            # (S is T itself in float64: the floor is the device's own summation order over up to 1e5 terms)
            floor = 1e-12 if dt is np.float64 else 1e-7
            gate = 4 * max(st["S_max"], st["Fh_max"]) + floor
            st["gate"] = gate
            if st["D_max"] > gate:
                bad.append(f"max error {st['D_max']:.3g} against T over {gate:.3g}")
        elif mode == "fast_cg1":
            # with limit_step the capped step should put a coordinate on the bound; the contracted update leaves
            # a rounding residual there instead, and whether the line search takes that trial point flips on the
            # residual's sign (at k = 1 it decides the whole row).  Coordinates on the bound in either result are
            # compared by their pattern, the others by value.
            tol = CG1_TOL[dt]
            Tr, Mr = T[rows].astype(np.float64), M0[rows].astype(np.float64)
            bound = 1e-6 * np.abs(Mr).max(axis=1, keepdims=True)
            def off(X):
                X = X[rows].astype(np.float64)
                free = (X > bound) & (Tr > bound)
                e = np.linalg.norm(np.where(free, X - Tr, 0), axis=1) / np.maximum(np.linalg.norm(Mr, axis=1), 1e-300)
                return int((e > tol).sum()), int(((X > bound) != (Tr > bound)).any(axis=1).sum())
            (nd, fd), (nf, ff) = off(D), off(Fh)
            st["rows_off_T"], st["Fh_rows_off_T"], st["bound_flips"], st["Fh_bound_flips"] = nd, nf, fd, ff
            if nd > nf + max(1, int(0.01 * n), int(0.25 * nf)):
                bad.append(f"{nd} rows further than {tol} from T (fast restatement: {nf})")
            if fd > 2 * ff + max(2, int(0.25 * n)):
                bad.append(f"{fd} rows with other coordinates on the bound than T (fast restatement: {ff})")
        if need_obj:
            dD = (fD[rows] - fS[rows]) / np.maximum(np.abs(fS[rows]), 1e-300)
            dF = (fF[rows] - fS[rows]) / np.maximum(np.abs(fS[rows]), 1e-300)
            st.update(obj_median=float(np.median(dD)), obj_worse=float((dD > OBJ_WORSE[dt]).mean()),
                      Fh_obj_median=float(np.median(dF)), Fh_obj_worse=float((dF > OBJ_WORSE[dt]).mean()))
            med_gate = 4 * max(st["Fh_obj_median"], 0.0) + OBJ_MED[dt]
            if mode == "fast_obj_stall":
                # the fast builds stall on those residuals after the first iteration, bin by bin differently
                # (medians of 0.1..0.5 against S on short rows): only gross errors are gated
                med_gate = 4 * max(st["Fh_obj_median"], 0.0) + 0.05
            if not st["obj_median"] <= med_gate:
                bad.append(f"median objective excess {st['obj_median']:.3g} over {med_gate:.3g}")
            if mode != "fast_obj_stall" and st["obj_worse"] > st["Fh_obj_worse"] + 0.1 + 2.0 / n:
                bad.append(f"{st['obj_worse']:.3f} of rows worse by > {OBJ_WORSE[dt]} (fast restatement: "
                           f"{st['Fh_obj_worse']:.3f})")
        if dt is np.float64 and mode in ("fast_pg", "fast_obj"):
            # a float intermediate in a double kernel moves rows by 1e-9..1e-7: count rows off T like cg1 (not for
            # tncg, whose branchy line search moves ~half the rows of the fast restatement by 1e-8..1e-4 already)
            nd, nf = int((eD[rows] > F64_TOL).sum()), int((eF[rows] > F64_TOL).sum())
            st["rows_off_T"], st["Fh_rows_off_T"] = nd, nf
            if nd > nf + max(1, int(0.01 * n)):
                bad.append(f"{nd} rows further than {F64_TOL} from T (fast restatement: {nf})")
        st["pass"] = not bad
        stats[kind] = st
        fails += [f"{kind}: {b}" for b in bad]
    return fails, stats
