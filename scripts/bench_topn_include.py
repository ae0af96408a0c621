"""Batched top-N over per-user candidate lists (pmf_b200_topN_batch_include / _fitted_include) on one GPU.

    python scripts/bench_topn_include.py [--steps 10] [--warmup 3] [--sample 256] [--out profiles/r3_topn_include.json]

Workloads (float32, k = 64, 1 M items, top 100):
  rerank  32 768 users, 200-1 000 candidates each, drawn without replacement from a popularity-skewed
          distribution: the retrieval-then-rerank serving pattern.  Every list is ranked in shared memory.
  mixed   8 192 users, most lists 100-5 000 items, 2 % of them 20 K-200 K: both ranking paths in one call.

Timed: the resident handle (DeviceFit.topN with include lists), the host-array call (c_funs._topN_batch,
which uploads A and B unless POISMF_B200_CACHE_FACTORS=1), and as reference points the full-catalogue
resident ranking of the same users, the per-user pmf_b200_topN(include) loop and the reference's topN(include)
loop on a subsample of users.  Kernel times come from a separate torch.profiler run of one resident call.
A sample of users is checked against the oracle after the timed region.  The card's name and power limit are
read in the same run and written beside the numbers.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N_ITEMS, K, TOP_N = 1_000_000, 64, 100
HBM_TBS = 7.7          # HGX B200 data sheet, one GPU


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as e:
        return {"name": None, "error": str(e)}


def skewed_lists(rng, n_users, lo, hi, n_items):
    """Per user lo..hi distinct items, drawn from a popularity-skewed distribution (item rank r ~ n u^3)."""
    perm = rng.permutation(n_items)
    lens = rng.integers(lo, hi + 1, n_users)
    out = []
    for m in lens:
        got = np.empty(0, np.int64)
        while got.shape[0] < m:
            draws = perm[(n_items * rng.random(2 * int(m)) ** 3).astype(np.int64)]
            got = np.unique(np.concatenate([got, draws]))
        out.append(rng.permutation(got)[:m])
    ptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    return ptr, np.concatenate(out).astype(np.uint64)


def workload(name, rng):
    if name == "rerank":
        n_users = 32_768
        ptr, ix = skewed_lists(rng, n_users, 200, 1000, N_ITEMS)
    else:
        n_users = 8_192
        long_users = rng.random(n_users) < 0.02
        lens = np.where(long_users, rng.integers(20_000, 200_001, n_users), rng.integers(100, 5001, n_users))
        ptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
        ix = np.concatenate([rng.choice(N_ITEMS, int(m), replace=False) for m in lens]).astype(np.uint64)
    return n_users, ptr, ix


def timed(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        fn()                     # every call ends by copying its results to the host: synchronised
        ts.append(time.perf_counter() - t0)
    return 1e3 * float(np.median(ts)), 1e3 * float(np.min(ts))


def kernel_ms(fn):
    """Device time per kernel family of one call (torch.profiler, CUDA activities)."""
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
        key = ("smem_select" if "include_select_smem_kernel" in nm else
               "long_score" if "include_score_long_kernel" in nm else
               "long_emit" if "include_emit_long_kernel" in nm else
               "segmented_sort" if "DeviceSegmentedRadixSort" in nm or "SegmentedRadixSort" in nm else
               "gather_rows" if "gather_rows_kernel" in nm else
               "id_check" if "any_id_out_of_range" in nm else
               "memcpy" if "Memcpy" in nm or "memcpy" in nm else "other")
        fam[key] = fam.get(key, 0.0) + ev.device_time_total / 1e3
    return fam


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--sample", type=int, default=256, help="users in the per-user loops and the oracle check")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_topn_include.json"))
    args = ap.parse_args()

    import torch
    from oracle.oracle import Ref, Restatement
    from poismf_b200 import _lib, c_funs
    from poismf_b200.device import DeviceFit
    _lib.require_gpu()
    torch.cuda.init()
    res = {"card": card(), "items": N_ITEMS, "k": K, "top_n": TOP_N, "dtype": "float32",
           "cache_factors_env": os.environ.get("POISMF_B200_CACHE_FACTORS"), "workloads": {}}
    rng = np.random.default_rng(7)
    B = np.ascontiguousarray(rng.gamma(0.5, 0.5, size=(N_ITEMS, K)).astype(np.float32))
    orc = Restatement(np.float32)
    if Ref.available(np.float32, fast=True):
        ref, ref_kind = Ref(np.float32, fast=True), "reference (-O3 OpenMP build of the reference's src/topN.c)"
    else:
        ref, ref_kind = Restatement(np.float32), "port (scalar restatement: the reference's build is not present)"
    cores = os.cpu_count() or 1
    for name in ("rerank", "mixed"):
        n_users, ptr, ix = workload(name, rng)
        A = np.ascontiguousarray(rng.gamma(0.5, 0.5, size=(n_users, K)).astype(np.float32))
        users = np.arange(n_users, dtype=np.uint64)
        lens = np.diff(ptr.astype(np.int64))
        cand = int(lens.sum())
        w = {"users": n_users, "candidates": cand, "list_len_min": int(lens.min()), "list_len_max": int(lens.max()),
             "users_long_path": int((lens > 16384).sum()),
             "candidates_long_path": int(lens[lens > 16384].sum())}
        fit = DeviceFit(n_users, N_ITEMS, K, np.float32)
        fit.set_factors(A, B)
        last = []

        def resident():
            last[:] = fit.topN(users=users, incl_ptr=ptr, incl_ix=ix, top_n=TOP_N, output_score=True)

        def host_arrays():
            c_funs._topN_batch(A, B, users=users, incl_ptr=ptr, incl_ix=ix, top_n=TOP_N, output_score=True)

        def full_catalogue():
            fit.topN(users=users, top_n=TOP_N, output_score=True)

        w["resident_ms_median"], w["resident_ms_min"] = timed(resident, args.steps, args.warmup)
        w["host_arrays_ms_median"], w["host_arrays_ms_min"] = timed(host_arrays, max(args.steps // 2, 1), 1)
        w["full_catalogue_resident_ms_median"], _ = timed(full_catalogue, args.steps, args.warmup)
        fam = kernel_ms(resident)
        w["kernel_ms"] = {k_: round(v, 4) for k_, v in sorted(fam.items())}
        gather_ms = fam.get("smem_select", 0.0) + fam.get("long_score", 0.0)
        # bytes the gather must read: one k-wide row of B and one list entry per candidate
        gbytes = cand * (K * 4 + 8)
        w["gather_bytes"] = gbytes
        w["gather_kernels_ms"] = round(gather_ms, 4)
        w["gather_bandwidth_TBs"] = round(gbytes / (gather_ms / 1e3) / 1e12, 3) if gather_ms else None
        w["gather_bandwidth_note"] = ("candidates x (k*4 + 8 index bytes) over the device time of the scoring kernels "
                                      "(include_select_smem_kernel incl. its in-CTA sort, include_score_long_kernel), "
                                      f"against the {HBM_TBS} TB/s HBM3e data-sheet figure; rows of B that repeat "
                                      "across users are served from L2, so this can exceed what HBM alone gives")
        w["gather_share_of_hbm_datasheet"] = round(gbytes / (gather_ms / 1e3) / (HBM_TBS * 1e12), 3) if gather_ms else None

        # per-user loops on a subsample (B resident in the single-user path, as in profiles/r2_point_queries.txt)
        sample = rng.choice(n_users, min(args.sample, n_users), replace=False)
        os.environ["POISMF_B200_CACHE_FACTORS"] = "1"
        a_rows = [np.ascontiguousarray(A[int(u)]) for u in sample]
        lists = [np.ascontiguousarray(ix[int(ptr[u]):int(ptr[u + 1])]) for u in sample]
        empty = np.empty(0, np.uint64)
        c_funs._call_topN(a_rows[0], B, lists[0], empty, top_n=TOP_N, output_score=True)    # warm: B goes resident
        t0 = time.perf_counter()
        for a, lst in zip(a_rows, lists):
            c_funs._call_topN(a, B, lst, empty, top_n=TOP_N, output_score=True)
        per_user_ms = 1e3 * (time.perf_counter() - t0) / len(sample)
        if res["cache_factors_env"] is None:
            del os.environ["POISMF_B200_CACHE_FACTORS"]
        _lib.lib().pmf_b200_release_cache()
        t0 = time.perf_counter()
        for a, lst in zip(a_rows, lists):
            ref.topN(a, B, TOP_N, include=lst, **({"nthreads": cores} if isinstance(ref, Ref) else {}))
        ref_ms = 1e3 * (time.perf_counter() - t0) / len(sample)
        w["per_user_loop"] = {"subsample_users": len(sample), "ms_per_user": round(per_user_ms, 4),
                              "extrapolated_all_users_ms": round(per_user_ms * n_users, 1),
                              "what": "pmf_b200_topN(include) once per user, B resident (POISMF_B200_CACHE_FACTORS=1)"}
        w["reference_loop"] = {"subsample_users": len(sample), "ms_per_user": round(ref_ms, 4),
                               "extrapolated_all_users_ms": round(ref_ms * n_users, 1), "kind": ref_kind,
                               "cores": cores if isinstance(ref, Ref) else 1}
        w["speedup_vs_per_user_loop"] = round(per_user_ms * n_users / w["resident_ms_median"], 1)
        w["speedup_vs_reference_loop"] = round(ref_ms * n_users / w["resident_ms_median"], 1)
        w["vs_full_catalogue"] = round(w["full_catalogue_resident_ms_median"] / w["resident_ms_median"], 2)

        # the results of the last timed resident call against the oracle
        ids, sc = last
        bad = 0
        for u in sample[:64]:
            _, oi, os_ = orc.topN(np.ascontiguousarray(A[int(u)]), B, TOP_N, include=ix[int(ptr[u]):int(ptr[u + 1])])
            bad += not (np.array_equal(ids[u], oi) and np.array_equal(sc[u], os_))
        w["oracle_check"] = {"users": int(min(64, len(sample))), "mismatches": int(bad)}
        res["workloads"][name] = w
        print(json.dumps({name: w}), flush=True)
        fit.close()
        del fit
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"wrote": args.out, "card": res["card"]}))
    return 0 if all(w["oracle_check"]["mismatches"] == 0 for w in res["workloads"].values()) else 1


if __name__ == "__main__":
    sys.exit(main())
