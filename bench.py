#!/usr/bin/env python
"""bench.py — poismf_b200 headline benchmark.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config c2|small|c1|c3s|c3|c4s|c5s]

Metric (BASELINE.json): nnz processed per second per alternating sweep.
A "step" is ONE alternating sweep (B half-sweep over CSC + A half-sweep over CSR) of the workload; at
N=1 the workload is BASELINE config #2 — Last.FM-360K-shaped synthetic, 359k users x 160k items, 17.5M
power-law draws, k=50, method=cg (maxupd 5, l2 1e4, limit_step), float32 (the reference's Python default,
poismf/__init__.py:240).  Other configs (not the driver's bench line): c3s / c3 Netflix-shaped tncg k=100,
c4s web-scale-shaped pg k=64 (1/10 scale in users, items and non-zeros), c5s batched topN (users/s).

  value    : nnz / device time per sweep, inputs resident in HBM (CUDA events on the launching stream, max
             over ranks); the K timed steps are sweeps 1..K of ONE fit from the initial factors
  e2e      : the same metric through the drop-in C ABI call run_poismf (numiter=1) with page-locked HOST
             buffers: H2D of CSR+CSC+factors and D2H of the factors inside the timed region
             (`e2e_pageable`: the same call on ordinary pageable numpy arrays, what the reference's callers pass)
  roofline : dominant launch of the sweep: algorithmic bytes of its rows / its average device time
  cpu_baseline : the reference's own C path (oracle/_ref, OpenMP, all host cores) on the SAME arrays, sweeps
             1..3 of one fit
  parity   : (N > 1) after the timed region every rank hashes its replicas and rank 0 repeats the sweeps
             on one GPU

--impl reference times only the reference's CPU implementation on the same arrays, sweeps 1..K of one fit
(rank 0; other ranks exit).

--dump-outputs DIR writes what the timed path returned after its last step (A and B after sweep K; for c5s the
ranked ids and scores) as DIR/<name>.npy, so that two builds can be compared output for output on the same
seeded inputs.  Outputs larger than DUMP_BYTES in all are cut to the same seeded sample of rows on every run.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    # name: dimA, dimB, nnz draws, k, method, hyper-parameters
    "c2": dict(dimA=359_000, dimB=160_000, nnz=17_500_000, k=50, method="cg",
               hp=dict(l2_reg=1e4, maxupd=5, limit_step=True),
               label="lastfm360k-shaped synthetic 359k x 160k, 17.5M power-law draws, k=50, cg"),
    "small": dict(dimA=45_000, dimB=20_000, nnz=2_200_000, k=50, method="cg",
                  hp=dict(l2_reg=1e4, maxupd=5, limit_step=True),
                  label="1/8-scale lastfm360k-shaped synthetic 45k x 20k, 2.2M draws, k=50, cg"),
    "c1": dict(dimA=100, dimB=1000, nnz=10_000, k=5, method="pg",
               hp=dict(l2_reg=1e9, maxupd=1, step_size=1e-7),
               label="README synthetic 100 x 1000, 1e4 nnz, k=5, pg"),
    # BASELINE config #3 (Netflix-shaped, tncg, k=100, maxupd = 15 k): full size and 1/10 of the users
    "c3": dict(dimA=480_000, dimB=17_700, nnz=100_000_000, k=100, method="tncg",
               hp=dict(l2_reg=1e3, maxupd=1500), alpha=(0.5, 0.7),
               label="netflix-shaped synthetic 480k x 17.7k, 100M power-law draws, k=100, tncg"),
    "c3s": dict(dimA=48_000, dimB=17_700, nnz=10_000_000, k=100, method="tncg",
                hp=dict(l2_reg=1e3, maxupd=1500), alpha=(0.5, 0.7),
                label="1/10-scale netflix-shaped synthetic 48k x 17.7k, 10M power-law draws, k=100, tncg"),
    # BASELINE config #4 (web-scale, pg, k=64, maxupd 1) at 1/10 of the users, items and non-zeros
    "c4s": dict(dimA=1_000_000, dimB=100_000, nnz=200_000_000, k=64, method="pg",
                hp=dict(l2_reg=1e9, maxupd=1, step_size=1e-7),
                label="1/10-scale web-scale synthetic 1M x 100k, 200M power-law draws, k=64, pg"),
}
TOPN = dict(users=32_768, items=1_000_000, k=64, top_n=100, excl=200,
            label="batched topN: 32k users x 1M items, k=64, top-100, ~200 excluded items per user")


DUMP_BYTES = 60 << 20


def dump_outputs(out_dir, arrays):
    """arrays: name -> float32/float64 array.  Every array keeps the same fraction of its rows (sorted, drawn with
    a fixed seed) so that together they fit in DUMP_BYTES."""
    os.makedirs(out_dir, exist_ok=True)
    frac = min(1.0, DUMP_BYTES / sum(a.nbytes for a in arrays.values()))
    for name, a in arrays.items():
        if frac < 1.0:
            rows = np.random.default_rng(0).choice(a.shape[0], int(a.shape[0] * frac), replace=False)
            a = a[np.sort(rows)]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def make_problem(cfg, dtype=np.float32):
    from poismf_b200.synth import init_factors, powerlaw_counts, readme_counts
    if cfg["dimA"] == 100:
        csr, csc = readme_counts(dtype=dtype)
    else:
        aa, ab = cfg.get("alpha", (0.6, 0.9))
        csr, csc = powerlaw_counts(cfg["dimA"], cfg["dimB"], cfg["nnz"], alpha_a=aa, alpha_b=ab, dtype=dtype, seed=1)
    A0, B0 = init_factors(cfg["dimA"], cfg["dimB"], cfg["k"], seed=1, dtype=dtype)
    return csr, csc, A0, B0


def team_name(code):
    if code == 200:
        return "lockstep"
    if code >= 100:
        return f"regtile{code - 100}w"
    return f"lanes{-code}" if code < 0 else ("block" if code == 1 else f"cluster{code}")


def algorithmic_bytes(nnz, rows, other, k, s):
    """SURVEY.md §8(d): bytes of one half-sweep = nnz*(k*s + s + 4) + rows*(2*k*s + 8) + other*k*s."""
    return nnz * (k * s + s + 4) + rows * (2 * k * s + 8) + other * k * s


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "25"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nme, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def run_reference(cfg, problem, sweeps, warmup_sweeps=0):
    """The reference's own CPU path (oracle/_ref, -O3 OpenMP build of /root/reference/src) on the SAME arrays
    as the device arm: sweeps 1..`sweeps` of ONE fit from the initial factors (what the device arm times).
    Returns (ms per sweep, info, (A, B) after the last sweep)."""
    from oracle.oracle import Ref, Restatement
    csr, csc, A0, B0 = problem
    nnz = int(csr[0].shape[0])
    cores = os.cpu_count() or 1
    if Ref.available(np.float32, fast=True):
        lib, kind = Ref(np.float32, fast=True), "reference"
    else:
        lib, kind, cores = Restatement(np.float32), "port", 1
    hp = dict(cfg["hp"])
    if warmup_sweeps:
        A, B = A0.copy(), B0.copy()
        lib.run_poismf(A, B, csr, csc, cfg["method"], numiter=warmup_sweeps, nthreads=cores, **hp)
    A, B = A0.copy(), B0.copy()
    t0 = time.perf_counter()
    lib.run_poismf(A, B, csr, csc, cfg["method"], numiter=sweeps, nthreads=cores, **hp)
    ms = 1e3 * (time.perf_counter() - t0) / sweeps
    build = ("-O3 x86-64-v3 OpenMP build of /root/reference/src + sequential BLAS" if kind == "reference"
             else "scalar restatement")
    info = {"value": nnz / (ms / 1e3), "unit": "nnz/s per sweep", "cores": cores, "kind": kind, "same_config": True,
            "sample": f"the full workload ({cfg['label']}: {nnz} stored nnz), sweeps 1..{sweeps} of one fit from the "
                      f"initial factors ({build})"}
    return ms, info, (A, B)


def topn_problem():
    rng = np.random.default_rng(5)
    t = TOPN
    A = np.ascontiguousarray(rng.gamma(0.5, 0.5, size=(t["users"], t["k"])).astype(np.float32))
    B = np.ascontiguousarray(rng.gamma(0.5, 0.5, size=(t["items"], t["k"])).astype(np.float32))
    lens = rng.poisson(t["excl"], t["users"])
    ptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    eix = rng.integers(0, t["items"], int(ptr[-1])).astype(np.uint64)
    return A, B, ptr, eix


def bench_topn(args, rank, world, local_rank):
    """c5s: users ranked per second through the batched topN entry (host buffers in and out: an e2e figure)."""
    import torch
    from poismf_b200 import _lib, c_funs
    from poismf_b200.sharding import user_ranges
    _lib.require_gpu()
    torch.cuda.set_device(local_rank)
    os.environ["POISMF_B200_DEVICE"] = str(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    t = TOPN
    A, B, ptr, eix = topn_problem()
    lo, hi = user_ranges(t["users"], world)[rank]
    users = np.arange(lo, hi, dtype=np.uint64)
    p64 = ptr.astype(np.int64)
    lptr = (p64[lo:hi + 1] - p64[lo]).astype(np.uint64)
    leix = np.ascontiguousarray(eix[p64[lo]:p64[hi]])

    # e2e: host buffers in and out.  N=1: the stateless batched entry (uploads A, B and the exclusion lists).
    # N>1: the sharded public API on a persistent backend — every rank uploads 1/N of the factor rows (stored
    # into all replicas over NVLink), ranks its share of the users against its replicas, reads its lists back
    from poismf_b200.device import DeviceFit
    be = None
    if world > 1:
        from poismf_b200.sharding import GpuBackend
        be = GpuBackend(None, None, A, B, rank, world, local_rank)

    def one():
        if dist is not None:
            dist.barrier()
        t0 = time.perf_counter()
        if be is None:
            c_funs._topN_batch(A, B, users=users, excl_ptr=lptr, excl_ix=leix, top_n=t["top_n"], output_score=True)
        else:
            be.reset(A, B)
            be.topN(t["top_n"], excl_ptr=ptr, excl_ix=eix, output_score=True, gather=False)
        return time.perf_counter() - t0
    for _ in range(max(args.warmup, 1)):
        one()
    _lib.topn_stats(reset=True)
    ts = [one() for _ in range(args.steps)]
    n_tc, n_redo = _lib.topn_stats(reset=True)
    ms_e2e = 1e3 * float(np.mean(ts))
    # value: the same ranking against factors RESIDENT in a fit handle (pmf_b200_topN_fitted: what follows a fit
    # on the device; every rank of a sharded fit holds full replicas): only ids and exclusion lists travel
    if be is None:
        fit = DeviceFit(t["users"], t["items"], t["k"], np.float32, device=local_rank)
        fit.set_factors(A, B)
    else:
        fit = be.fit

    last = []

    def one_resident():
        t0 = time.perf_counter()
        last[:] = fit.topN(users=users, excl_ptr=lptr, excl_ix=leix, top_n=t["top_n"], output_score=True)
        return time.perf_counter() - t0
    for _ in range(max(args.warmup, 1)):
        one_resident()
    if dist is not None:
        dist.barrier()
    ms = 1e3 * float(np.mean([one_resident() for _ in range(args.steps)]))
    if args.dump_outputs:      # this rank's users; ids are exact in float64
        ids, scores = last
        dump_outputs(os.path.join(args.dump_outputs, f"rank{rank}") if world > 1 else args.dump_outputs,
                     {"topn_ids": ids.astype(np.float64), "topn_scores": scores})
    if dist is not None:
        tt = torch.tensor([ms, ms_e2e], device="cuda", dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms, ms_e2e = float(tt[0].item()), float(tt[1].item())
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        # dense tf32 peak: half the measured bf16 cuBLAS figure (B200_PROFILING.md: 1.1 vs 2.25 PF nominal)
        peak = float(peaks.get("bf16_tflops", 1590.0)) / 2 * args.gpus          # all GPUs of the job
        flops = 2.0 * t["users"] * t["items"] * t["k"] * 2          # two scoring passes (threshold, candidates)
        h2d = (A.nbytes + B.nbytes) // world + users.nbytes + lptr.nbytes + leix.nbytes if world > 1 else \
            A.nbytes + B.nbytes + users.nbytes + lptr.nbytes + leix.nbytes
        d2h = users.shape[0] * t["top_n"] * 12
        line = {"metric": "users ranked/sec (batched topN)", "value": t["users"] / (ms / 1e3), "unit": "users/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "tf32 candidates + f32 exact re-score", "data": "synthetic",
                "config": {"workload": t["label"], "parallelism": f"users sharded x{args.gpus}, B replicated",
                           "value_call": "pmf_b200_topN_fitted: factors resident in a fit handle (HBM), ids + exclusion "
                                         "lists up, rankings + scores down"},
                "roofline": {"bound": "tensor", "achieved": flops / (ms / 1e3) / 1e12, "peak": peak, "unit": "TFLOP/s",
                             "frac": flops / (ms / 1e3) / 1e12 / peak, "traffic": None,
                             "note": "whole resident call (threshold pass on 1/4 of the item tiles counted as a full "
                                     "pass: 2 x 2 U n k flops) against half the measured bf16 cuBLAS peak of the job's GPUs"},
                "e2e": {"value": t["users"] / (ms_e2e / 1e3), "unit": "users/s", "ms_per_step": ms_e2e,
                        "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                        "call": ("pmf_b200_topN_batch: pageable host arrays A, B, exclusion lists in, rankings + scores out"
                                 if world == 1 else
                                 "GpuBackend.reset(A, B) + GpuBackend.topN(gather=False) on a persistent backend: every rank "
                                 "uploads 1/N of the factor rows (stored into all replicas over NVLink), ranks its users, "
                                 "reads its lists back (max over ranks; bytes are per rank)")},
                "topn_users_on_tensor_cores": int(n_tc), "topn_users_redone_exactly": int(n_redo)}
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=list(CONFIGS) + ["c5s"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (at most 60 MiB in all: "
                         "larger outputs as a fixed seeded sample of their rows)")
    ap.add_argument("--flags", type=int, default=0)
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "p2p-host", "nccl"],
                    help="N>1: refresh replicas by peer-memory stores from the row kernels, completion signalled on the "
                         "device (p2p) or by a host barrier (p2p-host), or by NCCL broadcasts")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.config == "c5s":
        if args.impl == "reference":
            if rank == 0:
                print(json.dumps({"impl": "reference", "unavailable": "c5s: the reference has no batched topN entry point"}))
            return 0
        return bench_topn(args, rank, world, local_rank)
    cfg = CONFIGS[args.config]
    warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    xdesc = {"p2p": "NVLink peer-memory stores fused into the row kernels, completion signalled on the device",
             "p2p-host": "NVLink peer-memory stores fused into the row kernels + host barrier",
             "nccl": "NCCL broadcasts"}[args.exchange]
    config_line = {"workload": cfg["label"], "method": cfg["method"], "k": cfg["k"], **cfg["hp"],
                   "l2_flush": "inputs larger than L2 (factors+CSR+CSC vs 126 MB)",
                   "parallelism": f"rows/cols sharded x{args.gpus}, replicas refreshed by {xdesc}" if args.gpus > 1 else "single GPU"}
    metric = "nnz processed/sec per alternating sweep"

    # ------------------------------------------------------------------ reference arm
    if args.impl == "reference":
        if rank != 0:
            return 0
        problem = make_problem(cfg)
        ms, info, (A, B) = run_reference(cfg, problem, args.steps, warmup_sweeps=min(args.warmup, 1))
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"A": A, "B": B})
        line = {"impl": "reference", "metric": metric, "value": info["value"],
                "unit": "nnz/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": config_line, "nnz": int(problem[0][0].shape[0]),
                "cpu_baseline": info,
                "e2e": {"value": info["value"], "unit": "nnz/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------ our arm
    import torch
    from poismf_b200 import FLAG_NO_LOCKSTEP, _lib, c_funs, make_params
    from poismf_b200.device import DeviceFit
    _lib.require_gpu()
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    L = _lib.lib()
    problem = make_problem(cfg)
    csr, csc, A0, B0 = problem
    nnz = int(csr[0].shape[0])
    dimA, dimB, k = cfg["dimA"], cfg["dimB"], cfg["k"]
    params = make_params(cfg["method"], numiter=1, flags=args.flags, **cfg["hp"])
    be = None

    if world == 1:
        fit = DeviceFit(dimA, dimB, k, np.float32, device=local_rank)
        stream = torch.cuda.Stream(device=local_rank)
        fit.set_stream(stream.cuda_stream)
        fit.set_csr_csc(csr, csc)
        reset = lambda: fit.set_factors(A0, B0)
        sweep = lambda: fit.sweeps(params)
        finish = lambda: None
        profiler = fit
    else:
        from poismf_b200.sharding import GpuBackend, ShardedSweep
        be = GpuBackend(csr, csc, A0, B0, rank, world, local_rank, exchange=args.exchange)
        stream = be.stream
        drv = ShardedSweep(be, dimA, dimB, np.float32)
        reset = lambda: be.reset(A0, B0)
        sweep = lambda: drv.run(params)
        finish = be.finish
        profiler = be.fit

    def barrier():
        finish()
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    reset()
    for _ in range(warmup):
        sweep()
    barrier()
    reset()
    launches0 = L.pmf_b200_kernel_launches()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        ev0.record(stream)
        for _ in range(args.steps):
            sweep()
        ev1.record(stream)
    barrier()
    ms_total = ev0.elapsed_time(ev1)
    launches = L.pmf_b200_kernel_launches() - launches0
    if args.dump_outputs:
        out = fit.get_factors() if world == 1 else be.factors(root=0)
        if rank == 0:
            dump_outputs(args.dump_outputs, {"A": out[0], "B": out[1]})
    # second pass over the same K sweeps with per-launch CUDA events (bins run one after the
    # other on the launching stream here; in the timed pass above they overlap on side streams)
    reset()
    profiler.set_profiling(True)
    barrier()
    pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        pe0.record(stream)
        for _ in range(args.steps):
            sweep()
        pe1.record(stream)
    barrier()
    ms_profiled_pass = pe0.elapsed_time(pe1)
    clocks = sampler.stop() if rank == 0 else None      # sampled over the timed pass and the per-launch pass
    prof = profiler.get_profile()
    profiler.set_profiling(False)
    if dist is not None:
        t = torch.tensor([ms_total], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    ms_step = ms_total / args.steps
    value = nnz / (ms_step / 1e3)

    # roofline of the dominant launch (by device time), rank 0's shard
    roof = None
    if prof:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        which = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
        top = max(prof, key=lambda p: p["ms"])
        s = 4
        # the opposite factor matrix's column-sum read is a separate kernel: not charged to the launch
        bytes_launch = top["nnz"] * (k * s + s + 4) + top["nrows"] * (2 * k * s + 8)
        avg_ms = top["ms"] / max(top["launches"], 1)
        achieved = bytes_launch / (avg_ms / 1e3) / 1e9 if avg_ms > 0 else 0.0
        sweep_bytes = algorithmic_bytes(nnz, dimA, dimB, k, s) + algorithmic_bytes(nnz, dimB, dimA, k, s)
        traffic = None
        try:   # DRAM bytes of this launch from the committed ncu --set full capture of the same command
            tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            traffic = tj.get(f"{args.config}_side{top['side']}_{team_name(top['block_team'])}_cap{top['cap']}")
        except Exception:
            pass
        roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "peak_source": which,
                "kernel": f"{team_name(top['block_team'])}<{cfg['method']}> side="
                          f"{'CSR(A)' if top['side'] == 0 else 'CSC(B)'} cap={top['cap']} rows={top['nrows']} nnz={top['nnz']}",
                "kernel_avg_ms": avg_ms, "kernel_share_of_step": top["ms"] / max(ms_profiled_pass, 1e-9),
                "serialized_ms_per_step": ms_profiled_pass / args.steps,
                "sweep_algorithmic_GBps": sweep_bytes / (ms_step / 1e3) / 1e9,
                "sweep_frac_of_peak": sweep_bytes / (ms_step / 1e3) / 1e9 / peak / max(args.gpus, 1),   # per GPU
                "bins": [{"side": p["side"], "team": team_name(p["block_team"]), "cap": p["cap"],
                          "rows": p["nrows"], "nnz": p["nnz"], "ms_per_sweep": p["ms"] / args.steps,
                          "GBps": (p["nnz"] * (k * s + s + 4) + p["nrows"] * (2 * k * s + 8)) / max(p["ms"] / args.steps, 1e-9) / 1e6}
                         for p in prof]}
        # SURVEY 8d: the solver re-reads every tile once per evaluation pass, out of registers / shared memory
        mu = int(cfg["hp"].get("maxupd", 1))
        passes = {"cg": 1 + 2 * mu, "pg": 2 * mu}.get(cfg["method"])
        if passes:
            roof["tile_passes_per_row_max"] = passes
            roof["onchip_tile_GBps_upper"] = 2 * nnz * k * s * passes / (ms_step / 1e3) / 1e9

    # every rank's own work per sweep (its bins' device times of the per-launch pass, by side): the shards' balance
    shard_work = None
    if world > 1 and prof:
        mine = torch.tensor([sum(p["ms"] for p in prof if p["side"] == sd) / args.steps for sd in (0, 1)],
                            device="cuda", dtype=torch.float64)
        allw = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allw, mine)
        shard_work = [[round(float(w[0]), 4), round(float(w[1]), 4)] for w in allw]

    # ---- N > 1: every rank hashes its replicas; rank 0 repeats the sweeps on one GPU
    parity = None
    if world > 1 and not args.no_parity:
        from poismf_b200.sharding import ShardedSweep
        n_chk = 2
        parity = {"sweeps": n_chk}
        for tag, fl in (("", args.flags | FLAG_NO_LOCKSTEP), ("lockstep_", args.flags)):
            pchk = make_params(cfg["method"], numiter=n_chk, flags=fl, **cfg["hp"])
            be.reset(A0, B0)
            ShardedSweep(be, dimA, dimB, np.float32).run(pchk)
            As, Bs = be.factors()
            digest = hashlib.sha256(As.tobytes() + Bs.tobytes()).hexdigest()
            alld = [None] * world
            dist.all_gather_object(alld, digest)
            same = len(set(alld)) == 1
            rel = llk_rel = None
            if rank == 0:
                one = DeviceFit(dimA, dimB, k, np.float32, device=local_rank)
                one.set_csr_csc(csr, csc); one.set_factors(A0, B0)
                one.sweeps(pchk); one.sync()
                A1, B1 = one.get_factors()
                one.close()
                rel = max(float(np.abs(As - A1).max() / max(np.abs(A1).max(), 1e-30)),
                          float(np.abs(Bs - B1).max() / max(np.abs(B1).max(), 1e-30)))
                try:
                    from oracle.oracle import Restatement
                    orc = Restatement(np.float32)
                    l1, ls = orc.llk(A1, B1, csr), orc.llk(As, Bs, csr)
                    llk_rel = abs(ls - l1) / abs(l1)
                except Exception:
                    pass
            parity[tag + "ranks_identical"] = bool(same)
            parity[tag + "vs_single_gpu_max_rel"] = rel
            parity[tag + "llk_rel"] = llk_rel
        parity["note"] = ("ranks_identical / vs_single_gpu_max_rel: per-row teams only (PMF_FLAG_NO_LOCKSTEP), whose bits do not "
                          "depend on the partition; lockstep_*: default flags, the heaviest rows' non-zeros are summed in an order "
                          "that depends on which heavy rows a rank holds (cg in float is chaotic in the rounding: compare llk)")

    # e2e: drop-in run_poismf with host buffers (rank 0 alone at N=1; the sharded public API otherwise)
    e2e = e2e_pageable = None
    if not args.no_e2e and world == 1:
        h2d = sum(a.nbytes for a in (csr[0], csr[1], csr[2], csc[0], csc[1], csc[2], A0, B0))
        d2h = A0.nbytes + B0.nbytes
        e_steps = max(3, min(args.steps, 5))
        hA, hB = A0.copy(), B0.copy()

        def one():
            hA[...] = A0; hB[...] = B0
            t0 = time.perf_counter()
            c_funs._run_poismf(csr[0], csr[2], csr[1], csc[0], csc[2], csc[1], hA, hB, method=cfg["method"],
                               limit_step=cfg["hp"].get("limit_step", False), l2_reg=cfg["hp"]["l2_reg"],
                               step_size=cfg["hp"].get("step_size", 1e-7), niter=1, maxupd=cfg["hp"]["maxupd"],
                               early_stop=False, reuse_prev=False, flags=args.flags)
            return time.perf_counter() - t0

        def timed(call):
            one()
            e_ms = 1e3 * float(np.mean([one() for _ in range(e_steps)]))
            return {"value": nnz / (e_ms / 1e3), "unit": "nnz/s", "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "ms_per_step": e_ms, "steps": e_steps, "call": call}
        e2e_pageable = timed("run_poismf(numiter=1) via C ABI, ordinary pageable numpy buffers (staged through page-locked "
                             "blocks by host threads), upload+plan+sweep+download")
        pin = []
        for arr in (csr[0], csr[1], csr[2], csc[0], csc[1], csc[2], hA, hB):
            t = torch.from_numpy(arr)
            try:
                torch.cuda.cudart().cudaHostRegister(t.data_ptr(), t.numel() * t.element_size(), 0)
                pin.append(t)
            except Exception:
                pass
        e2e = timed("run_poismf(numiter=1) via C ABI, host buffers (cudaHostRegister'ed), upload+plan+sweep+download")
        for t in pin:
            try:
                torch.cuda.cudart().cudaHostUnregister(t.data_ptr())
            except Exception:
                pass

    if not args.no_e2e and world > 1:
        # sharded public API end to end on the PERSISTENT backend (handles, peer mappings and epoch slots are
        # set up once per process group): every rank uploads ITS row/column shard and the replicated factors
        # from host memory, runs one sharded sweep, reads A,B back
        from poismf_b200.sharding import ShardedSweep
        ts = []
        h2d = d2h = 0
        outA, outB = np.empty_like(A0), np.empty_like(B0)
        pin = []             # page-locked host buffers, as in the N=1 leg (slices of them are page-locked too)
        for arr in (csr[0], csr[1], csr[2], csc[0], csc[1], csc[2], A0, B0, outA, outB):
            tt = torch.from_numpy(arr)
            try:
                torch.cuda.cudart().cudaHostRegister(tt.data_ptr(), tt.numel() * tt.element_size(), 0)
                pin.append(tt)
            except Exception:
                pass
        trace = bool(os.environ.get("POISMF_B200_BENCH_TRACE"))      # (every rank: finish() holds a barrier)
        for it in range(4):
            dist.barrier()
            t0 = time.perf_counter()
            be.load(csr, csc, A0, B0)
            t1 = time.perf_counter()
            ShardedSweep(be, dimA, dimB, np.float32).run(params)
            if trace:
                be.finish()
            t2 = time.perf_counter()
            be.factors(root=0, out=(outA, outB))
            t3 = time.perf_counter()
            dist.barrier()
            dt = time.perf_counter() - t0
            if trace and rank == 0:
                print(f"[e2e N={world}] load {1e3 * (t1 - t0):.2f} ms, sweep {1e3 * (t2 - t1):.2f} ms, factors "
                      f"{1e3 * (t3 - t2):.2f} ms, total {1e3 * dt:.2f} ms", file=sys.stderr)
            a0, a1 = be.rangesA[rank]; b0, b1 = be.rangesB[rank]
            h2d = ((A0.nbytes + B0.nbytes) // world + int(csr[1][a1] - csr[1][a0]) * 12 + int(csc[1][b1] - csc[1][b0]) * 12
                   + (a1 - a0 + b1 - b0) * 8)
            d2h = A0.nbytes + B0.nbytes if rank == 0 else 0
            if it > 0:
                ts.append(dt)
        for tt in pin:
            try:
                torch.cuda.cudart().cudaHostUnregister(tt.data_ptr())
            except Exception:
                pass
        t = torch.tensor([float(np.mean(ts))], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e_ms = 1e3 * float(t.item())
        e2e = {"value": nnz / (e_ms / 1e3), "unit": "nnz/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
               "ms_per_step": e_ms, "steps": len(ts),
               "call": "GpuBackend.load + ShardedSweep.run(numiter=1) + factors(root=0) on a persistent backend, host buffers "
                       "cudaHostRegister'ed: every rank "
                       "uploads its matrix shard and 1/N of the initial factors (stored into all replicas over NVLink), plan, "
                       "sweep with the fused exchange, rank 0 reads A and B back (max over ranks; bytes are per rank)"}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            _, cpu, _ = run_reference(cfg, problem, 3)
        except Exception as e:  # the oracle is optional infrastructure for this leg
            cpu = {"value": None, "unit": "nnz/s per sweep", "cores": 0, "kind": "unavailable", "sample": str(e)}

    if rank == 0:
        line = {"metric": metric, "value": value, "unit": "nnz/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": warmup, "ms_per_step": ms_step,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic", "config": config_line, "nnz": nnz, "gpu_launches": int(launches),
                "clocks": clocks, "roofline": roof, "cpu_baseline": cpu, "e2e": e2e}
        if e2e_pageable is not None:
            line["e2e_pageable"] = e2e_pageable
        if shard_work is not None:
            line["shard_work_ms"] = {"per_rank_A_B": shard_work,
                                     "note": "sum of a rank's own launches per sweep, serialised (per-launch pass)"}
        if parity is not None:
            line["parity"] = parity
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
