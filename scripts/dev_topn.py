"""Batched topN wall time through the C ABI: tensor-core candidate scorer vs exact scorer."""
import os, sys, time
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from poismf_b200 import _lib, c_funs
rng = np.random.default_rng(1)
n_items, n_users, k, n_top = 160_000, 2048, 64, 100
A = np.ascontiguousarray(rng.gamma(0.5, 0.5, size=(n_users, k)).astype(np.float32))
B = np.ascontiguousarray(rng.gamma(0.5, 0.5, size=(n_items, k)).astype(np.float32))
lens = rng.integers(50, 350, n_users)
ptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
eix = np.concatenate([np.sort(rng.choice(n_items, int(m), replace=False)) for m in lens]).astype(np.uint64)
res = {}
for mode in ("tc", "exact", "tc", "exact"):
    os.environ.pop("POISMF_B200_TOPN_EXACT", None)
    if mode == "exact": os.environ["POISMF_B200_TOPN_EXACT"] = "1"
    _lib.topn_stats(reset=True)
    t0 = time.perf_counter()
    ix, sc = c_funs._topN_batch(A, B, excl_ptr=ptr, excl_ix=eix, top_n=n_top, output_score=True)
    dt = time.perf_counter() - t0
    res[mode] = (ix, sc)
    print(mode, f"{dt*1e3:.1f} ms  users/s {n_users/dt:.0f}  stats {_lib.topn_stats()}", flush=True)
print("scores identical:", np.array_equal(res["tc"][1], res["exact"][1]),
      " ids identical:", np.mean(res["tc"][0] == res["exact"][0]))
# larger batch: only the fused path (the exact one would need the score matrix in chunks)
os.environ.pop("POISMF_B200_TOPN_EXACT", None)
n_users2 = 32768
A2 = np.ascontiguousarray(rng.gamma(0.5, 0.5, size=(n_users2, k)).astype(np.float32))
for _ in range(2):
    _lib.topn_stats(reset=True)
    t0 = time.perf_counter()
    ix, sc = c_funs._topN_batch(A2, B, top_n=n_top, output_score=True)
    dt = time.perf_counter() - t0
    print(f"fused, {n_users2} users x {n_items} items: {dt*1e3:.1f} ms  users/s {n_users2/dt:.0f}  stats {_lib.topn_stats()}", flush=True)
