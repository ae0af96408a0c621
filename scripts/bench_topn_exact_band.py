"""Batched top-N below the fused tensor-core select's threshold: the route the call takes against the exact route.

    python scripts/bench_topn_exact_band.py [--steps 5] [--warmup 2] [--out profiles/r4_topn_exact_band.json]

The fused select needs the items to hold 2 M groups of 16 (M = max(2 N, N + 32) candidates for a top-N), i.e.
more than 16 (2 M - 1) items: 1 328 for top-10, 6 384 for top-100.  Below that a float32 call either sorts the
TF32 score matrix and re-scores the best M exactly, or is exact (every item scored with the reference's sums,
then a segmented sort of each user's scores).  For every shape of the grid (users x items x k x top-N, factors
resident in a fit handle, gamma-distributed) the default call and the exact one (POISMF_B200_TOPN_EXACT=1) are
timed alternately, twice each; `route` is what pmf_b200_topN_stats reports for the default call.  Each figure
is the median wall time of calls that end by copying their results to the host; `spread_ms` is the largest
difference between the two repetitions of one route.  The card's name and power limit are read in the same
run and written beside the numbers.
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

USERS = (1, 32, 256, 2_048, 32_768)
ITEMS = (256, 512, 1_000, 1_328, 2_000, 3_500, 5_000, 6_384)
KS = (16, 64, 128)
TOPS = (10, 100)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as e:
        return {"name": None, "error": str(e)}


def fused(n_items, top_n):
    return -(-n_items // 16) >= 2 * max(2 * top_n, top_n + 32)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_topn_exact_band.json"))
    args = ap.parse_args()

    from poismf_b200 import _lib
    from poismf_b200.device import DeviceFit
    _lib.require_gpu()
    os.environ.pop("POISMF_B200_TOPN_EXACT", None)
    res = {"card": card(), "dtype": "float32", "steps": args.steps, "warmup": args.warmup, "shapes": []}
    rng = np.random.default_rng(4)
    for k in KS:
        A = np.ascontiguousarray(rng.gamma(0.5, 0.5, size=(max(USERS), k)).astype(np.float32))
        for n_items in ITEMS:
            B = np.ascontiguousarray(rng.gamma(0.5, 0.5, size=(n_items, k)).astype(np.float32))
            fit = DeviceFit(max(USERS), n_items, k, np.float32)
            try:
                fit.set_factors(A, B)
                for top_n in TOPS:
                    if fused(n_items, top_n) or top_n > n_items:
                        continue
                    for n_users in USERS:
                        users = np.arange(n_users, dtype=np.uint64)
                        ms = {"default": [], "exact": []}
                        n_tc = 0
                        for rep in range(2):
                            for route in ("default", "exact"):
                                if route == "exact":
                                    os.environ["POISMF_B200_TOPN_EXACT"] = "1"
                                for _ in range(args.warmup):
                                    fit.topN(users=users, top_n=top_n, output_score=True)
                                _lib.topn_stats(reset=True)
                                ts = []
                                for _ in range(args.steps):
                                    t0 = time.perf_counter()
                                    fit.topN(users=users, top_n=top_n, output_score=True)
                                    ts.append(time.perf_counter() - t0)
                                if route == "default":
                                    n_tc += _lib.topn_stats(reset=True)[0]
                                os.environ.pop("POISMF_B200_TOPN_EXACT", None)
                                ms[route].append(1e3 * float(np.median(ts)))
                        total = 2 * args.steps * n_users
                        w = {"users": n_users, "items": n_items, "k": k, "top_n": top_n,
                             "route": "tensor_cores" if n_tc == total else "exact" if n_tc == 0 else "mixed",
                             "default_ms": round(float(np.mean(ms["default"])), 4),
                             "exact_ms": round(float(np.mean(ms["exact"])), 4),
                             "spread_ms": round(max(abs(ms[r][0] - ms[r][1]) for r in ms), 4)}
                        res["shapes"].append(w)
                        print(json.dumps(w), flush=True)
            finally:
                fit.close()
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"wrote": args.out, "card": res["card"]}))
    return 0


if __name__ == "__main__":
    sys.exit(main())
