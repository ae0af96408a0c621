"""Parity of the numerics mode bench.py TIMES (fast arithmetic, float32, cached cg line search, default
flags) against the reference's own C path (oracle/_ref) on the SAME arrays as the bench: the 1/8-scale
sample and the full BASELINE config #2; tncg likewise on the sample.

Coordinates of float cg / tncg are chaotic in the rounding (SURVEY.md 4.1: two CPU builds of the
reference miss the 1e-3 gate against each other on ~100 % of rows), so parity is asserted on what is
stable:
  (i)   total Poisson log-likelihood after 1 and 3 sweeps: within max(1e-4, 5 x the measured distance
        between the reference's FMA/-O3 build and its strict build on this very problem),
  (ii)  per-row OBJECTIVE of one half-sweep on identical inputs (B side from (A0, B0); A side from
        (A0, B_ref)): f_dev <= f_ref (1 + 1e-4) on >= 99.9 % of rows and not worse in the median,
  (iii) exact-zero fractions side by side.
"""
import os
import sys

import numpy as np
import pytest

from conftest import ROOT, row_objectives, row_rel_err

sys.path.insert(0, ROOT)
pytestmark = pytest.mark.gpu


def _dump(name, obj):
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    import json
    with open(os.path.join(ROOT, "gpurun_out", name), "w") as f:
        json.dump(obj, f, indent=1, default=float)


def _reference(dtype):
    """The reference's two builds (oracle/_ref) where they have been built, else the restatement's: bit-identical
    to the reference's strict build, and the same C code under the fast build's flags."""
    from oracle.oracle import Ref, Restatement
    return Ref if Ref.available(dtype) else Restatement


def _fit_ref(Ref, dtype, fast, csr, csc, A0, B0, method, hp, numiter):
    A, B = A0.copy(), B0.copy()
    rc = Ref(dtype, fast=fast).run_poismf(A, B, csr, csc, method, numiter=numiter, nthreads=os.cpu_count() or 1, **hp)
    assert rc == 0
    return A, B


def _fit_dev(csr, csc, A0, B0, method, hp, numiter, flags=0):
    from poismf_b200 import c_funs
    A, B = A0.copy(), B0.copy()
    rc = c_funs._run_poismf(csr[0], csr[2], csr[1], csc[0], csc[2], csc[1], A, B, method=method,
                            limit_step=hp.get("limit_step", False), l2_reg=hp["l2_reg"],
                            step_size=hp.get("step_size", 1e-7), niter=numiter, maxupd=hp["maxupd"],
                            early_stop=False, reuse_prev=hp.get("reuse_prev", False), flags=flags)
    assert rc == 0
    return A, B


def _llk(A, B, csr):
    from oracle.oracle import Restatement
    return Restatement(A.dtype).llk(A, B, csr)


def _objective_stats(dev, ref, F, mat, l2, rel):
    f_dev = row_objectives(dev, F, mat, l2)
    f_ref = row_objectives(ref, F, mat, l2)
    nz = np.diff(mat[1].astype(np.int64)) > 0
    d = (f_dev - f_ref)[nz] / np.maximum(np.abs(f_ref[nz]), 1e-30)
    err = row_rel_err(dev[nz], ref[nz])
    return dict(rows=int(nz.sum()), finite=bool(np.isfinite(f_dev[nz]).all()),
                worse_frac=float((d > rel).mean()), better_frac=float((d < -rel).mean()),
                median=float(np.median(d)), p001=float(np.quantile(d, 0.001)), p999=float(np.quantile(d, 0.999)),
                factor_err_median=float(np.median(err)), factor_err_over_1e3=float((err > 1e-3).mean()),
                empty_rows_zero=bool(not dev[~nz].any()))


def _check_half_sweeps(cfg, csr, csc, A0, B0, strict, fast, rel=1e-4, tag=""):
    """(ii): one half-sweep of the device on exactly the inputs the reference's half-sweep saw, per-row
    objective (the FULL objective; tncg's own f omits the l2 term its gradient keeps, quirk Q3, so the
    point it converges to is the stationary point of the full one) against both builds of the reference
    (`strict`, `fast`: their (A, B) after one sweep)."""
    from poismf_b200 import SIDE_CSC, SIDE_CSR, make_params
    from poismf_b200.device import DeviceFit
    dimA, dimB, k = A0.shape[0], B0.shape[0], A0.shape[1]
    hp = cfg["hp"]
    params = make_params(cfg["method"], numiter=1, **hp)
    fit = DeviceFit(dimA, dimB, k, A0.dtype)
    fit.set_csr_csc(csr, csc)
    fit.set_factors(A0, B0)
    fit.half_sweep(SIDE_CSC, params, hp.get("step_size", 1e-7), 1.0)
    fit.sync()
    _, B_dev = fit.get_factors()
    report = {}
    for name, (A_cmp, B_cmp) in (("strict", strict), ("fast", fast)):
        fit.set_factors(A0, B_cmp)
        fit.half_sweep(SIDE_CSR, params, hp.get("step_size", 1e-7), 1.0)
        fit.sync()
        A_dev, _ = fit.get_factors()
        report[f"B_dev_vs_{name}"] = _objective_stats(B_dev, B_cmp, A0, csc, hp["l2_reg"], rel)
        report[f"A_dev_vs_{name}"] = _objective_stats(A_dev, A_cmp, B_cmp, csr, hp["l2_reg"], rel)
    fit.close()
    # how far the reference's two builds are from each other on the B side (same inputs: A0, B0)
    report["B_fast_vs_strict"] = _objective_stats(fast[1], strict[1], A0, csc, hp["l2_reg"], rel)
    _dump(f"parity_headline_{tag}_half_sweeps.json", report)
    for key, r in report.items():
        assert r["finite"] and r["empty_rows_zero"], (key, r)
    return report


def _check_llk_and_zeros(Ref, cfg, csr, csc, A0, B0, sweeps, tag):
    dtype = A0.dtype
    out = {}
    for n in sweeps:
        A_r, B_r = _fit_ref(Ref, dtype, False, csr, csc, A0, B0, cfg["method"], cfg["hp"], n)
        A_f, B_f = _fit_ref(Ref, dtype, True, csr, csc, A0, B0, cfg["method"], cfg["hp"], n)
        A_d, B_d = _fit_dev(csr, csc, A0, B0, cfg["method"], cfg["hp"], n)
        assert np.isfinite(A_d).all() and np.isfinite(B_d).all() and (A_d >= 0).all() and (B_d >= 0).all()
        l_r, l_f, l_d = _llk(A_r, B_r, csr), _llk(A_f, B_f, csr), _llk(A_d, B_d, csr)
        floor = abs(l_f - l_r) / abs(l_r)
        gate = max(1e-4, 5 * floor)
        z = lambda M: float((M == 0).mean())
        out[n] = dict(llk_ref=l_r, llk_reffast=l_f, llk_dev=l_d, rel=abs(l_d - l_r) / abs(l_r), floor=floor,
                      rel_to_reffast=abs(l_d - l_f) / abs(l_f),
                      zeros_A=dict(dev=z(A_d), ref=z(A_r), reffast=z(A_f)),
                      zeros_B=dict(dev=z(B_d), ref=z(B_r), reffast=z(B_f)))
        _dump(f"parity_headline_{tag}_{n}sweeps.json", out[n])
        assert abs(l_d - l_r) <= gate * abs(l_r), out[n]
        # exact-zero fractions next to the strict reference's, allowing what the reference's own FMA build moves
        for zz in (out[n]["zeros_A"], out[n]["zeros_B"]):
            assert abs(zz["dev"] - zz["ref"]) <= 0.03 + abs(zz["reffast"] - zz["ref"]), out[n]
        if n == 1:
            out["first"] = ((A_r, B_r), (A_f, B_f))
    return out


@pytest.mark.parametrize("config", ["small", "c2"])
def test_benchmarked_mode_cg_f32_vs_reference(config):
    import bench
    Ref = _reference(np.float32)
    cfg = bench.CONFIGS[config]
    csr, csc, A0, B0 = bench.make_problem(cfg)
    rep = _check_llk_and_zeros(Ref, cfg, csr, csc, A0, B0, sweeps=(1, 3), tag=config)
    strict, fast = rep.pop("first")
    hs = _check_half_sweeps(cfg, csr, csc, A0, B0, strict, fast, tag=config)
    # The device's fast arithmetic contracts a*b+c like the reference's own -O3 / FMA build (what
    # `pip install poismf` compiles): against THAT build the per-row objective is unbiased ...
    for side in ("A", "B"):
        r = hs[f"{side}_dev_vs_fast"]
        assert r["median"] <= 2e-5 and abs(r["median"]) <= 1e-3, (side, r)      # never worse in the median
        assert r["worse_frac"] <= r["better_frac"] + 0.05, (side, r)
    # ... and against the strict (no-FMA, sequential) build it is no further away than the reference's
    # FMA build itself is (with limit_step the contracted update x + step*d leaves the limiting
    # coordinate a rounding residual above 0 instead of on the bound, which stalls the next iteration:
    # both FMA paths lose objective against the strict build in the same way)
    assert hs["B_dev_vs_strict"]["worse_frac"] <= hs["B_fast_vs_strict"]["worse_frac"] + 0.05, hs


def test_benchmarked_mode_tncg_f32_vs_reference():
    import bench
    Ref = _reference(np.float32)
    cfg = dict(bench.CONFIGS["small"])
    cfg["method"] = "tncg"
    cfg["hp"] = dict(l2_reg=1e3, maxupd=15 * cfg["k"])
    csr, csc, A0, B0 = bench.make_problem(cfg)
    rep = _check_llk_and_zeros(Ref, cfg, csr, csc, A0, B0, sweeps=(1,), tag="tncg_small")
    strict, fast = rep.pop("first")
    hs = _check_half_sweeps(cfg, csr, csc, A0, B0, strict, fast, tag="tncg_small")
    # tncg stops on |df| <= 1e-4 f (ftol) along branchy paths: rows end within that band of the strict
    # build's, better about as often as worse
    for side in ("A", "B"):
        r = hs[f"{side}_dev_vs_strict"]
        assert abs(r["median"]) <= 1e-4, (side, r)
        assert r["worse_frac"] <= r["better_frac"] + 0.05, (side, r)
