"""Generate tests/golden/*.npz from the reference itself (oracle/_ref, strict build).

Run in the CPU container where /root/reference exists:
    make -C oracle ref && python tests/golden/make_golden.py
The fixtures pin the plain-C restatement (and through it the CUDA path) on boxes where
/root/reference is absent.  Inputs are NOT stored: they are regenerated from seeds by
poismf_b200.synth (numpy RandomState / default_rng streams are stable across versions).
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))
from conftest import CASES, FM_CASES, FS_CASES, FS_ROWS, fm_hyper, fm_problem, fs_row, hyper, problem  # noqa: E402
from oracle.oracle import Ref  # noqa: E402


def main():
    out = {}
    for dt in (np.float64, np.float32):
        ref = Ref(dt)
        for prob in ("readme", "ragged"):
            csr, csc, A0, B0, k = problem(prob, dt)
            out[f"{prob}/{np.dtype(dt).name}/csr_checksum"] = np.array(
                [csr[0].astype(np.float64).sum(), csr[2].astype(np.float64).sum(), csr[0].shape[0]])
            for case in CASES:
                method, kw = hyper(case, k)
                A, B = A0.copy(), B0.copy()
                rc = ref.run_poismf(A, B, csr, csc, method, **kw)
                assert rc == 0
                out[f"{prob}/{np.dtype(dt).name}/{case}/A"] = A
                out[f"{prob}/{np.dtype(dt).name}/{case}/B"] = B
        # factors_multiple (src/pred.c:66-199) on the README shape
        csr, B, Bsum, Amean, k = fm_problem("readme", dt)
        for case in FM_CASES:
            method, kw = fm_hyper(case, k)
            rc, A = ref.factors_multiple(B, Bsum, Amean, csr, method, **kw)
            assert rc == 0
            out[f"factors_multiple/{np.dtype(dt).name}/{case}"] = A
        # factors_single (src/pred.c:201-304): a few rows of the same problem, plus the empty row
        for case, kw in FS_CASES.items():
            rows = [ref.factors_single(*fs_row(csr, r), B, Bsum, Amean, **kw)[1] for r in FS_ROWS]
            rows.append(ref.factors_single(np.empty(0, dt), np.empty(0, np.uint64), B, Bsum, Amean, **kw)[1])
            out[f"factors_single/{np.dtype(dt).name}/{case}"] = np.stack(rows)
        # predict_multiple and topN known answers on the README factors
        csr, csc, A0, B0, k = problem("readme", dt)
        rng = np.random.default_rng(3)
        ixA = rng.integers(0, A0.shape[0], 257).astype(np.uint64)
        ixB = rng.integers(0, B0.shape[0], 257).astype(np.uint64)
        out[f"predict/{np.dtype(dt).name}"] = ref.predict_multiple(A0, B0, ixA, ixB)
        Brand = np.ascontiguousarray(rng.gamma(1, 1, size=B0.shape).astype(dt))
        rc, ix, sc = ref.topN(np.ascontiguousarray(A0[3]), Brand, 10)
        out[f"topn/{np.dtype(dt).name}/ix"] = ix
        out[f"topn/{np.dtype(dt).name}/score"] = sc
        excl = np.arange(0, 1000, 7, dtype=np.uint64)
        rc, ix, sc = ref.topN(np.ascontiguousarray(A0[3]), Brand, 10, exclude=excl)
        out[f"topn_excl/{np.dtype(dt).name}/ix"] = ix
        out[f"topn_excl/{np.dtype(dt).name}/score"] = sc
    for name in ("float64", "float32"):      # one file per dtype keeps each under 1 MB
        part = {key: v for key, v in out.items() if key.split("/")[1] == name}
        np.savez_compressed(os.path.join(HERE, f"reference_outputs_{name}.npz"), **part)
    print("wrote", len(out), "arrays")


if __name__ == "__main__":
    main()
