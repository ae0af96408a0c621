"""Scoring (user, item) pairs against a resident fit, and building a resident matrix from COO triplets, on one GPU.

    python scripts/bench_predict_fitted.py [--max-pairs 1e8] [--out profiles/r6_predict_fitted.json]

Shape of BASELINE config #2 (359k users x 160k items, k = 50, float32); factors from a seeded generator, pairs drawn
uniformly (repeats and arbitrary order), ids uint64 (the reference's size_t).

Timed, n = 1e3 .. 1e8 pairs, host clock around calls that return with their scores on the host:
  * resident, pageable ids   DeviceFit.predict (pmf_b200_predict_fitted) on ordinary numpy arrays
  * resident, page-locked    the same ids and output in page-locked memory (copied without staging)
  * stateless                c_funs._predict_multiple on the factors as host arrays (uploads A and B every call)
  * reference                the reference's predict_multiple built with its fast flags, on every host core, where
                             oracle/_ref holds that build (as profiles/r2_point_queries.txt)
The resident scores are checked bitwise against the stateless call's at every n.

Kernel: device time of predict_resident_kernel from a torch.profiler capture of one resident call (CUDA activity
timestamps), and the bytes per pair of the model in `bytes_per_pair` over it.  Two id distributions: pairs over every
row, and pairs whose rows come from 2048 users and 2048 items (a working set far below the L2).  A and B together
are 108 MB, below the B200's 126 MB of L2: when the two kernel times agree, the rows of the full-range pairs are
served from L2 after the first touch, and the byte rate is an L2 rate, not an HBM one.

Ingestion: DeviceFit.set_coo against SciPy coo.tocsr() / coo.tocsc() + set_csr_csc for the same shuffled triplets
(the config #2 draws, 17.5M with duplicates).

The card's name and power limit are read in the same run and written beside the numbers.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from bench_topn_include import card  # noqa: E402

DIM_A, DIM_B, K, NNZ = 359_000, 160_000, 50, 17_500_000


def bytes_per_pair(k, real_bytes=4, id_bytes=8):
    """Bytes the resident kernel moves per pair: two ids in, two rows read as whole 16-byte vectors (k padded to
    the vector width), one score out."""
    v = 16 // real_bytes
    return 2 * id_bytes + 2 * ((k + v - 1) // v) * 16 + real_bytes


def best_ms(fn, reps, warmup=1):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return round(1e3 * float(np.median(ts)), 4), round(1e3 * float(np.min(ts)), 4)


def kernel_ms(fn):
    """(device ms of predict_resident_kernel, its launches) in one call, from a torch.profiler capture."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    ms, n = 0.0, 0
    for ev in prof.events():
        if ev.device_type.name == "CUDA" and "predict_resident_kernel" in ev.name:
            ms += ev.device_time_total / 1e3
            n += 1
    return ms, n


def pinned_like(a):
    """A page-locked array with a's dtype and contents, and the torch tensor that owns its memory."""
    import torch
    t = torch.empty(a.nbytes, dtype=torch.uint8).pin_memory()
    view = t.numpy().view(a.dtype)
    view[:] = a
    return view, t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--max-pairs", type=float, default=1e8)
    ap.add_argument("--dims", default=f"{DIM_A},{DIM_B},{NNZ}", help="users,items,triplet draws (rehearsal: smaller)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r6_predict_fitted.json"))
    args = ap.parse_args()
    dimA, dimB, nnz = (int(float(x)) for x in args.dims.split(","))

    from oracle.oracle import Ref
    from poismf_b200 import c_funs
    from poismf_b200.device import DeviceFit
    from poismf_b200.synth import powerlaw_counts
    rng = np.random.default_rng(0)
    A = np.ascontiguousarray(rng.gamma(0.5, 0.5, size=(dimA, K)).astype(np.float32))
    B = np.ascontiguousarray(rng.gamma(0.5, 0.5, size=(dimB, K)).astype(np.float32))
    cores = os.cpu_count()
    has_ref = Ref.available(np.float32, fast=True)
    ref = Ref(np.float32, fast=True) if has_ref else None
    fit = DeviceFit(dimA, dimB, K, np.float32)          # the first device call
    import torch
    torch.cuda.init()
    res = {"card": card(), "shape": {"users": dimA, "items": dimB, "k": K, "dtype": "float32", "ids": "uint64"},
           "reference": f"oracle/_ref fast build, {cores} threads" if has_ref else "not present on this host"}
    fit.set_factors(A, B)

    rows = []
    n = 1000
    ok = True
    while n <= args.max_pairs:
        u = rng.integers(0, dimA, n).astype(np.uint64)
        i = rng.integers(0, dimB, n).astype(np.uint64)
        reps = 20 if n <= 1e5 else 5 if n <= 1e7 else 3
        out = np.empty(n, np.float32)
        r = {"pairs": n}
        r["resident_pageable_ms"], _ = best_ms(lambda: fit.predict(u, i, out=out), reps)
        got = out.copy()
        pu, tu = pinned_like(u)
        pi, ti = pinned_like(i)
        po, to = pinned_like(out)
        r["resident_pinned_ms"], _ = best_ms(lambda: fit.predict(pu, pi, out=po), reps)
        ok &= np.array_equal(po.view(np.uint32), got.view(np.uint32))
        del pu, pi, po, tu, ti, to
        want = np.empty(n, np.float32)
        r["stateless_ms"], _ = best_ms(lambda: c_funs._predict_multiple(want, A, B, u, i), reps)
        r["bitwise_equal_stateless"] = bool(np.array_equal(got.view(np.uint32), want.view(np.uint32)))
        ok &= r["bitwise_equal_stateless"]
        if ref is not None:
            r["reference_ms"], _ = best_ms(lambda: ref.predict_multiple(A, B, u, i, nthreads=cores), reps)
        rows.append(r)
        print(json.dumps(r), flush=True)
        n *= 10
    res["predict"] = rows

    # kernel: full-range pairs against pairs over 2048 x 2048 rows
    kern = {"bytes_per_pair_model": bytes_per_pair(K), "what": "torch.profiler device time of predict_resident_kernel"}
    n = int(min(args.max_pairs, 1e7))
    for label, (hi_a, hi_b) in (("full_range", (dimA, dimB)), ("hot_2048_rows", (min(2048, dimA), min(2048, dimB)))):
        u = rng.integers(0, hi_a, n).astype(np.uint64)
        i = rng.integers(0, hi_b, n).astype(np.uint64)
        fit.predict(u, i)
        ms, launches = kernel_ms(lambda: fit.predict(u, i))
        kern[label] = {"pairs": n, "kernel_ms": round(ms, 4), "launches": launches,
                       "ns_per_pair": round(1e6 * ms / n, 4),
                       "achieved_GB_per_s": round(bytes_per_pair(K) * n / (ms / 1e3) / 1e9, 1) if ms else None}
        print(json.dumps({label: kern[label]}), flush=True)
    if kern["full_range"]["kernel_ms"] and kern["hot_2048_rows"]["kernel_ms"]:
        ratio = kern["full_range"]["kernel_ms"] / kern["hot_2048_rows"]["kernel_ms"]
        kern["full_over_hot"] = round(ratio, 3)
    kern["factor_bytes"] = (dimA + dimB) * 52 * 4
    res["kernel"] = kern

    # ingestion: the config #2 draws as shuffled triplets (duplicates kept)
    from scipy.sparse import coo_matrix
    csr, _ = powerlaw_counts(dimA, dimB, nnz, dtype=np.float32, seed=1)
    r_ = np.repeat(np.arange(dimA, dtype=np.uint64), np.diff(csr[1].astype(np.int64)))
    dup = rng.integers(0, r_.shape[0], r_.shape[0] // 20)         # 5% exact duplicates on top
    perm = rng.permutation(r_.shape[0] + dup.shape[0])
    rows_, cols_, vals_ = (np.ascontiguousarray(np.concatenate([a, a[dup]])[perm]) for a in (r_, csr[2], csr[0]))

    def host_path():
        coo = coo_matrix((vals_, (rows_.astype(np.int64), cols_.astype(np.int64))), shape=(dimA, dimB))
        m, c = coo.tocsr(), coo.tocsc()
        t = lambda x: (np.ascontiguousarray(x.data), x.indptr.astype(np.uint64), x.indices.astype(np.uint64))
        fit.set_csr_csc(t(m), t(c))

    ing = {"triplets": int(vals_.shape[0])}
    ing["set_coo_ms"], ing["set_coo_ms_min"] = best_ms(lambda: fit.set_coo(rows_, cols_, vals_), 5)
    ing["scipy_tocsr_tocsc_set_csr_csc_ms"], _ = best_ms(host_path, 3)
    res["ingestion"] = ing
    print(json.dumps(ing), flush=True)
    res["card_after"] = card()
    res["all_bitwise_equal"] = bool(ok)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"wrote": args.out, "card": res["card"], "all_bitwise_equal": bool(ok)}))
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
