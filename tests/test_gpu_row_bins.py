"""Every row-kernel bin of the half-sweep against a float64 reference, bin by bin.

The planner (plan_rows, poismf_b200/csrc/row_plan.h) sends each row of the updated side to a kernel chosen by
its non-zero count: register-tile bins (float32 fast pg / cached cg with limit_step, k <= 64), (sub-)warp and
CTA teams, clusters of 2..16 CTAs, the streaming cluster bin and the lock-step path for the heaviest rows.
Whole-fit gates (log-likelihood, objective statistics over a matrix) do not see a kernel that is wrong on the
few rows of one bin, so here:

  1. a probe half-sweep with profiling on, over every row length 1..600 and then geometric lengths up to
     LMAX, reads back which bins the planner defines for the mode and their caps;
  2. the real problem has, per bin, rows of length 1 (first bin), lo+1, the middle, cap-1 and cap plus random
     lengths inside the bin, and empty rows, with the rows shuffled;
  3. one half-sweep of the device (D) is compared per bin with the plain-C restatement's half-sweep on the
     same inputs: T (float64, inputs upcast), S (strict build, device dtype), Fh (fast build, device dtype;
     the rounding noise floor).  The gates are tests/row_bins.check_bins.

Every case also asserts: outputs finite and >= 0, empty rows zero, the fixed factor untouched, and three
half-sweeps from the same inputs (one with profiling, i.e. bins run one after another, two with the bins
overlapped on side streams) bitwise identical.  Per-bin statistics are written as row_bins_*.json beside the
headline parity reports (test_gpu_headline._dump).

LMAX is 40 000: at small k (float32 k < 32: cluster bins of 8 and 16 CTAs start beyond ~56 K non-zeros) the
largest cluster bins and the streaming bin are not reached; they are covered, and asserted, at k >= 32.
"""
import numpy as np
import pytest

import row_bins as rb
from test_gpu_headline import _dump

pytestmark = pytest.mark.gpu

LMAX = 40000
ACAP = 4096          # per-CTA on-chip non-zeros of the streaming bin (bin_ladder(): b.acap); longer rows use global scratch
DENSE_MIN = 600      # lock-step cases: rows of >= 600 non-zeros take the lock-step path


def _device(prob, variant, strict, dtype, k, lockstep, profile=False):
    """Three half-sweeps of the updated side from the same inputs: profiled (bins serial), then twice with the
    bins overlapped.  Returns ([(A, B)] x 3, profile)."""
    from poismf_b200 import FLAG_NO_LOCKSTEP, FLAG_STRICT, make_params
    from poismf_b200.device import DeviceFit
    method, hp, flags = rb.VARIANTS[variant]
    # the lock-step path only where a case asks for it: elsewhere every row stays in its per-row bin
    flags |= (FLAG_STRICT if strict else 0) | (0 if lockstep else FLAG_NO_LOCKSTEP)
    params = make_params(method, flags=flags, **hp)
    side = prob["side"]
    step, cdiv = rb.step_and_cdiv(method, hp, side, dtype)
    A0, B0 = prob["A0"], prob["B0"]
    fit = DeviceFit(A0.shape[0], B0.shape[0], k, dtype)
    try:
        fit.set_csr_csc(prob["csr"], prob["csc"])
        outs, prof = [], None
        for i in range(1 if profile else 3):
            fit.set_profiling(i == 0)
            fit.set_factors(A0, B0)
            fit.half_sweep(side, params, step, cdiv)
            fit.sync()
            outs.append(fit.get_factors())
            if i == 0:
                prof = fit.get_profile()
        fit.set_profiling(False)
    finally:
        fit.close()
    return outs, prof


_PROBES = {}


def _probe(dtype, k, variant, strict, side, lockstep):
    """The bin table [(kind, lo, hi)] the planner uses for this mode, from a profiled half-sweep over the
    ladder of row lengths."""
    method, hp, flags = rb.VARIANTS[variant]
    key = (np.dtype(dtype).name, k, method, hp.get("limit_step"), flags, strict, side, lockstep)
    if key not in _PROBES:
        lengths = np.array(rb.probe_lengths(LMAX))
        prob = rb.build_problem(lengths, side, k, dtype, seed=11)
        _, prof = _device(prob, variant, strict, dtype, k, lockstep, profile=True)
        _PROBES[key] = (rb.bin_table(prof, side, DENSE_MIN if lockstep else None), prof)
    return _PROBES[key]


def _expected_kinds(table, dtype, k, variant, strict, lockstep):
    """What the planner must define for the mode, as far as LMAX reaches."""
    kinds = [t[0] for t in table]
    method, hp, flags = rb.VARIANTS[variant]
    f32 = np.dtype(dtype) == np.float32
    rt = f32 and not strict and k <= 64 and (method == "pg" or (method == "cg" and hp["limit_step"] and not flags))
    n_rt = sum(x.startswith("regtile") for x in kinds)
    assert n_rt == (11 if rt else 0), kinds
    if lockstep:
        assert kinds[-1] == "lockstep", kinds
        return
    assert any(x.startswith("cta:") and x != "cta:0" for x in kinds), kinds
    if not rt:
        assert any(x.startswith("warp") for x in kinds), kinds
    if strict:
        assert kinds[-1] == "cta:0" and not any(x.startswith(("cluster", "streaming")) for x in kinds), kinds
        return
    assert "cluster2" in kinds and "cluster4" in kinds, kinds
    if (f32 and k >= 32) or (not f32 and k >= 33):
        assert all(c in kinds for c in ("cluster8", "cluster16", "streaming")), kinds


# (dtype, k, variant, strict, side, lockstep)
def _cases():
    f32, f64, B, A = np.float32, np.float64, rb.SIDE_CSC, rb.SIDE_CSR
    out = []
    for k in (1, 3, 32, 33, 64, 65, 200):                       # both NC variants, register-tile edges, smem teams
        for v in ("pg", "cg1"):
            out += [(f32, k, v, False, B, False), (f32, k, v, False, A, False)]
    for k in (1, 33, 65, 200):
        out += [(f32, k, v, False, B, False) for v in ("cg1_nocache", "cg1_nolimit", "tncg2")]
    out += [(f32, 33, v, False, A, False) for v in ("cg1_nocache", "cg1_nolimit", "tncg2")]
    out += [(f32, k, "cg5", False, s, False) for k in (33, 64) for s in (B, A)]
    out += [(f32, 33, v, False, B, False) for v in ("cg5_nocache", "cg5_nolimit", "tncg")]
    for k in (1, 33, 200):
        out += [(f32, k, v, True, B, False) for v in ("pg", "cg1", "cg5_nolimit", "tncg2")]
    out += [(f32, 33, "pg", True, A, False)]
    for k in (1, 33, 256):
        out += [(f64, k, v, False, B, False) for v in ("pg", "cg1", "cg1_nocache", "cg1_nolimit", "tncg2")]
    out += [(f64, 33, v, False, A, False) for v in ("pg", "cg1")]
    out += [(f64, 33, v, False, B, False) for v in ("cg5", "tncg")]
    out += [(f64, 33, v, True, B, False) for v in ("pg", "cg1", "tncg2")] + [(f64, 256, "pg", True, B, False)]
    out += [(f32, k, "cg1", False, B, True) for k in (1, 32, 33, 64)] + [(f32, 64, "cg5", False, A, True)]
    return out


def _id(c):
    dtype, k, variant, strict, side, lockstep = c
    return (f"{np.dtype(dtype).name}-k{k}-{variant}-{'strict' if strict else 'fast'}-{'A' if side == rb.SIDE_CSR else 'B'}"
            + ("-lockstep" if lockstep else ""))


@pytest.mark.parametrize("case", _cases(), ids=_id)
def test_row_bins_against_reference(case, monkeypatch):
    dtype, k, variant, strict, side, lockstep = case
    if lockstep:
        monkeypatch.setenv("POISMF_B200_DENSE_MIN_TOTAL", "0")
        monkeypatch.setenv("POISMF_B200_DENSE_MIN", str(DENSE_MIN))
    table, probe_prof = _probe(dtype, k, variant, strict, side, lockstep)
    _expected_kinds(table, dtype, k, variant, strict, lockstep)

    # the open-ended last bin: up to twice its lower edge, and past 16 x ACAP for the streaming bin
    lo_last = table[-1][1]
    top = max(2 * lo_last, 64)
    if table[-1][0] == "streaming":
        top = max(top, 16 * ACAP + 37)
    lengths = np.array(rb.bin_lengths(table, seed=k, top=top) + [0] * 5)
    np.random.default_rng(k).shuffle(lengths)
    prob = rb.build_problem(lengths, side, k, dtype, seed=k + 100)
    method, hp, _ = rb.VARIANTS[variant]
    ref = rb.references(method, hp, prob, dtype)
    outs, prof = _device(prob, variant, strict, dtype, k, lockstep)

    upd = 1 if side == rb.SIDE_CSC else 0
    D = outs[1][upd]
    # fixed factor untouched; the three runs (serial bins, overlapped bins twice) bitwise identical
    for o in outs:
        assert np.array_equal(o[1 - upd], prob["F"])
        assert np.array_equal(o[upd], D)
    # the device binned the rows as the table says
    groups = rb.group_rows(lengths, table)
    dev_rows = {rb.bin_kind(e): e["nrows"] for e in prof if e["side"] == side}
    assert dev_rows == {kd: int(r.shape[0]) for kd, r in groups.items() if r.shape[0]}, (dev_rows, table)

    mode = rb.gate_mode(variant, strict, dtype)
    fails, stats = rb.check_bins(mode, dtype, dict(ref, D=D, M0=prob["M0"]), groups, prob, hp)
    _dump(f"row_bins_{_id(case)}.json", dict(mode=mode, table=table, bins=stats, nnz=int(lengths.sum()),
                                           rows=int(lengths.shape[0]), zero_frac_T=float((ref["T"] == 0).mean())))
    assert not fails, (fails, stats)
