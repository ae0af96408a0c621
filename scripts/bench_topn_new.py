"""Batched top-N for new users (pmf_b200_topN_new_fitted / _batch): fold-in + ranking in one call, on one GPU.

    python scripts/bench_topn_new.py [--steps 10] [--warmup 3] [--sample 256] [--out profiles/r5_topn_new.json]

Workload (float32, k = 64, 1 M items, top 100): 32 768 new users with 5-200 interactions each, items drawn from a
popularity-skewed distribution, every user's own items excluded (the fold-in CSR passed as the exclusion lists).
B, Bsum = B.sum(0) and Amean come from a seeded generator.  The fold-in parameters are PoisMF.topN_new's defaults.

Timed: the resident call (DeviceFit.topN_new), the host-array call (c_funs._topN_new_batch, which uploads B unless
POISMF_B200_CACHE_FACTORS=1), the fold-in alone (DeviceFit.transform with the same fold-in parameters), 1-user and
64-user resident latency, and the per-user _predict_factors + _call_topN loop (POISMF_B200_CACHE_FACTORS=1) on a
subsample of users, extrapolated to all users and labelled so.  A separate torch.profiler run of one resident call
gives the device time of the fold-in kernels against the ranking kernels, and the host-to-device copies of that call:
the check fails when one of them, or their sum, reaches the size of B.  A sample of users is checked after the timed
region: factors bitwise against the one-row fold-in, ids against the oracle's fold-in and ranking outside ties.  The
card's name and power limit are read in the same run and written beside the numbers.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from bench_topn_include import card, skewed_lists, timed  # noqa: E402

N_ITEMS, K, TOP_N, N_NEW = 1_000_000, 64, 100, 32_768
FOLD = dict(l2_reg=1e5, maxupd=20)          # PoisMF.topN_new / _predict_factors defaults


def profile_call(fn):
    """(device ms per kernel family, H2D copy sizes in bytes) of one call, from a torch.profiler trace."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    fam = {}
    for ev in prof.events():
        if ev.device_type.name != "CUDA":
            continue
        nm = ev.name
        key = ("memcpy" if "Memcpy" in nm or "memcpy" in nm else
               "memset" if "Memset" in nm or "memset" in nm else
               "fold_in" if any(s in nm for s in ("rows_warp_kernel", "rows_block_kernel", "rows_cluster_kernel",
                                                  "regtile", "fill_rows_kernel", "zero_rows_kernel",
                                                  "narrow_indices_kernel", "pad_rows_kernel", "unpad_rows_kernel")) else
               "rank" if any(s in nm for s in ("tf32", "select", "rescore", "sort_candidates", "exclusion_bitmap",
                                               "gather_rows", "any_negative", "any_id_out_of_range", "score_items",
                                               "mask_excluded", "SegmentedRadixSort", "include_")) else "other")
        fam[key] = fam.get(key, 0.0) + ev.device_time_total / 1e3
    h2d = []
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            trace = json.load(f)
    for ev in trace.get("traceEvents", []):
        if ev.get("cat") == "gpu_memcpy" and "HtoD" in ev.get("name", ""):
            h2d.append(int(ev.get("args", {}).get("bytes", 0)))
    return fam, h2d


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--sample", type=int, default=256, help="users in the per-user loop and the output check")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r5_topn_new.json"))
    args = ap.parse_args()

    import torch
    from oracle.oracle import Restatement
    from poismf_b200 import _lib, c_funs
    from poismf_b200.device import DeviceFit
    _lib.require_gpu()
    torch.cuda.init()
    res = {"card": card(), "items": N_ITEMS, "k": K, "top_n": TOP_N, "dtype": "float32", "new_users": N_NEW,
           "fold_in": dict(FOLD, method="tncg", niter=1), "own_items_excluded": True,
           "cache_factors_env": os.environ.get("POISMF_B200_CACHE_FACTORS")}
    rng = np.random.default_rng(7)
    B = np.ascontiguousarray(rng.gamma(0.5, 0.5, size=(N_ITEMS, K)).astype(np.float32))
    Bsum = np.ascontiguousarray(B.sum(0, dtype=np.float64).astype(np.float32))
    Amean = np.ascontiguousarray(rng.gamma(1.0, 0.3, size=K).astype(np.float32))
    ptr, ix = skewed_lists(rng, N_NEW, 5, 200, N_ITEMS)
    vals = rng.integers(1, 6, ix.shape[0]).astype(np.float32)
    res["interactions"] = int(ix.shape[0])
    fit = DeviceFit(1, N_ITEMS, K, np.float32)
    fit.set_factors(Amean[None, :].copy(), B)
    last = []

    def resident(m=N_NEW):
        p = ptr[:m + 1]
        last[:] = fit.topN_new(p, ix, vals, top_n=TOP_N, output_score=True, excl_ptr=p, excl_ix=ix, Bsum=Bsum,
                               Amean=Amean, return_factors=m == N_NEW, **FOLD)

    def host_arrays():
        c_funs._topN_new_batch(ptr, ix, vals, B, Bsum, Amean, top_n=TOP_N, output_score=True, excl_ptr=ptr,
                               excl_ix=ix, **FOLD)

    def transform():
        fit.transform(ptr, ix, vals, method="tncg", niter=1, step_size=0.0, Bsum=Bsum, Amean=Amean, **FOLD)

    w = {}
    w["resident_ms_median"], w["resident_ms_min"] = timed(resident, args.steps, args.warmup)
    ids, sc, A = last
    w["host_arrays_ms_median"], w["host_arrays_ms_min"] = timed(host_arrays, max(args.steps // 2, 1), 1)
    w["transform_ms_median"], w["transform_ms_min"] = timed(transform, args.steps, args.warmup)
    w["latency_1_user_ms_median"], _ = timed(lambda: resident(1), args.steps * 3, args.warmup)
    w["latency_64_users_ms_median"], _ = timed(lambda: resident(64), args.steps * 3, args.warmup)
    w["users_per_s_resident"] = round(N_NEW / (w["resident_ms_median"] / 1e3))

    fam, h2d = profile_call(lambda: resident(N_NEW - 1))
    w["kernel_ms"] = {k_: round(v, 4) for k_, v in sorted(fam.items())}
    split = fam.get("fold_in", 0.0) + fam.get("rank", 0.0)
    w["fold_in_share_of_kernel_time"] = round(fam.get("fold_in", 0.0) / split, 3) if split else None
    b_bytes = N_ITEMS * K * 4
    w["transfer_check"] = {"h2d_copies": len(h2d), "h2d_bytes_total": int(sum(h2d)),
                           "h2d_largest_bytes": int(max(h2d)) if h2d else 0, "B_bytes": b_bytes,
                           "passed": bool(h2d) and max(h2d) < b_bytes and sum(h2d) < b_bytes}

    # per-user loop on a subsample: one-row fold-in + one-user topN, B resident in both
    sample = np.sort(rng.choice(N_NEW, min(args.sample, N_NEW), replace=False))
    rows = [(np.ascontiguousarray(vals[int(ptr[u]):int(ptr[u + 1])]), np.ascontiguousarray(ix[int(ptr[u]):int(ptr[u + 1])]))
            for u in sample]
    os.environ["POISMF_B200_CACHE_FACTORS"] = "1"
    empty = np.empty(0, np.uint64)
    a0 = c_funs._predict_factors(*rows[0], B, Bsum, Amean, **FOLD)
    c_funs._call_topN(a0, B, empty, rows[0][1].copy(), top_n=TOP_N, output_score=True)   # warm: B goes resident
    singles = []
    t0 = time.perf_counter()
    for c, i in rows:
        a = c_funs._predict_factors(c, i, B, Bsum, Amean, **FOLD)
        c_funs._call_topN(a, B, empty, i.copy(), top_n=TOP_N, output_score=True)    # (it sorts the list in place)
        singles.append(a)
    per_user_ms = 1e3 * (time.perf_counter() - t0) / len(sample)
    if res["cache_factors_env"] is None:
        del os.environ["POISMF_B200_CACHE_FACTORS"]
    _lib.lib().pmf_b200_release_cache()
    w["per_user_loop"] = {"subsample_users": len(sample), "ms_per_user": round(per_user_ms, 4),
                          "extrapolated_all_users_ms": round(per_user_ms * N_NEW, 1),
                          "what": "_predict_factors + _call_topN once per user, B resident "
                                  "(POISMF_B200_CACHE_FACTORS=1); the all-users figure is extrapolated, not measured"}
    w["speedup_vs_per_user_loop_extrapolated"] = round(per_user_ms * N_NEW / w["resident_ms_median"], 1)

    # the results of the last full timed resident call: factors bitwise against the one-row fold-in; ids against the
    # oracle's fold-in and ranking wherever the oracle's scores are separated by more than the rounding noise
    orc = Restatement(np.float32)
    f_bad = sum(not np.array_equal(A[u], a) for u, a in zip(sample, singles))
    r_bad, checked = 0, min(32, len(sample))
    for u, (c, i) in zip(sample[:checked], rows[:checked]):
        a_o = orc.factors_single(c, i, B, Bsum, Amean, **FOLD)[1]
        _, oi, os_ = orc.topN(a_o, B, TOP_N + 1, exclude=i)
        s = os_.astype(np.float64)
        gap = np.abs(np.diff(s)) > 1e-3 * np.abs(s[:-1]).clip(1e-30)
        sep = np.ones(TOP_N + 1, bool)
        sep[1:] &= gap
        sep[:-1] &= gap
        r_bad += not np.array_equal(ids[u][sep[:TOP_N]], oi[:TOP_N][sep[:TOP_N]])
    w["output_check"] = {"factors_vs_single_row_users": len(sample), "factors_mismatches": int(f_bad),
                         "ranking_vs_oracle_users": checked, "ranking_mismatches_outside_ties": int(r_bad)}
    res["result"] = w
    res["card_after"] = card()
    print(json.dumps(w), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"wrote": args.out, "card": res["card"]}))
    ok = f_bad == 0 and r_bad == 0 and w["transfer_check"]["passed"]
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
