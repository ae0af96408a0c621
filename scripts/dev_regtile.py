"""Register-tile kernels with and without the lock-step path on one config: device time of the sweep, per-bin
times (serialised), log-likelihood after 1 and 3 sweeps, max factor difference.
    python scripts/dev_regtile.py [config] [method]"""
import os, sys
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bench import CONFIGS, make_problem, team_name
from poismf_b200 import FLAG_NO_LOCKSTEP, make_params
from poismf_b200.device import DeviceFit
from oracle.oracle import Restatement

name = sys.argv[1] if len(sys.argv) > 1 else "small"
cfg = dict(CONFIGS[name])
if len(sys.argv) > 2 and sys.argv[2] == "pg":
    cfg["method"] = "pg"; cfg["hp"] = dict(l2_reg=1e9, maxupd=1, step_size=1e-7)
csr, csc, A0, B0 = make_problem(cfg)
nnz = csr[0].shape[0]
orc = Restatement(np.float32)
res = {}
modes = os.environ.get("MODES", "regtile,nodense").split(",")
for mode in modes:
    fit = DeviceFit(cfg["dimA"], cfg["dimB"], cfg["k"], np.float32)
    st = torch.cuda.Stream(); fit.set_stream(st.cuda_stream); fit.set_csr_csc(csr, csc)
    p = make_params(cfg["method"], numiter=1, flags=FLAG_NO_LOCKSTEP if mode == "nodense" else 0, **cfg["hp"])
    ts = []
    for rep in range(5):
        fit.set_factors(A0, B0); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(st):
            e0.record(st); fit.sweeps(p); e1.record(st)
        torch.cuda.synchronize(); ts.append(e0.elapsed_time(e1))
    A1, B1 = fit.get_factors()
    fit.sweeps(p); fit.sweeps(p); fit.sync()
    A3, B3 = fit.get_factors()
    print(f"{mode}: ms/sweep {min(ts[1:]):.3f}  ({nnz / min(ts[1:]) * 1e-6:.3f} G nnz/s)  llk1 {orc.llk(A1, B1, csr):.6e} llk3 {orc.llk(A3, B3, csr):.6e}",
          "finite", bool(np.isfinite(A3).all() and np.isfinite(B3).all()), flush=True)
    fit.set_factors(A0, B0); fit.set_profiling(True)
    fit.sweeps(p); fit.sync()
    for b in fit.get_profile():
        if b["nnz"]:
            print(f"   side {b['side']} {team_name(b['block_team']):>11} cap {b['cap']:4d} rows {b['nrows']:7d} nnz {b['nnz']:9d} "
                  f"ms {b['ms']:.4f}  GB/s {b['nnz'] * (cfg['k'] * 4 + 8) / b['ms'] * 1e-6:8.1f}")
    fit.set_profiling(False)
    res[mode] = (A1, B1)
    fit.close()
for a in modes[1:]:
    dA = np.abs(res[modes[0]][0] - res[a][0]).max(); dB = np.abs(res[modes[0]][1] - res[a][1]).max()
    print(f"max |{modes[0]} - {a}| after one sweep: A", dA, "B", dB)
