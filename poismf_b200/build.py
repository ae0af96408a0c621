"""Build libpoismf_b200.so (CUDA kernels + C ABI) and the host drop-in layer, in-tree.

    python -m poismf_b200.build            # incremental
    python -m poismf_b200.build --force

Everything is compiled for sm_100a only (-gencode arch=compute_100a,code=sm_100a).
The strict-numerics translation units get --fmad=false (see csrc/common.cuh).
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
HOST = os.path.join(HERE, "host")
OBJ = os.path.join(HERE, "_build")
LIB = os.path.join(HERE, "libpoismf_b200.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
HOSTCC = os.environ.get("PMF_HOSTCC", "/usr/bin/gcc")

EXTRA = os.environ.get("PMF_NVCC_EXTRA", "").split()
NVFLAGS = EXTRA + ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
           "--expt-extended-lambda", "--expt-relaxed-constexpr", "-Xcompiler", "-fPIC", "-Xcompiler", "-O2",
           "-Xcudafe", "--diag_suppress=177"]

UNITS = {
    "api.cu": [],
    "sweep_fast_pgcg.cu": [],
    "sweep_fast_tn.cu": [],
    "sweep_lockstep.cu": [],
    "sweep_regtile_cg.cu": [],
    "sweep_regtile_pg.cu": [],
    "sweep_strict_pgcg.cu": ["--fmad=false"],
    "sweep_strict_tn.cu": ["--fmad=false"],
}


def _newer(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def _headers():
    hs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    hs.append(os.path.join(HERE, "..", "include", "poismf_b200.h"))
    return hs


def _run(cmd):
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("build failed: " + " ".join(cmd) + "\n" + r.stdout + r.stderr)
    return r.stdout + r.stderr


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    hdrs = _headers()
    jobs = []
    objs = []
    for src, extra in UNITS.items():
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ, src.replace(".cu", ".o"))
        objs.append(o)
        if force or _newer(o, [s] + hdrs):
            jobs.append([NVCC] + NVFLAGS + extra + ["-c", s, "-o", o])
    if jobs:
        with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 4)) as ex:
            for out in ex.map(_run, jobs):
                if verbose and out.strip():
                    print(out)
    if force or jobs or _newer(LIB, objs):
        _run([NVCC, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a",
                                                     "-cudart", "shared", "-ldl"])
    # host drop-in layer: the reference's own prototypes (real_t / sparse_ix variants)
    host_src = os.path.join(HOST, "poismf_host.c")
    inc = os.path.join(HERE, "..", "include")
    if os.path.exists(host_src):
        for name, defs in (("double", []), ("float", ["-DUSE_FLOAT"]), ("double_int", ["-DPMF_INDEX_INT"])):
            out = os.path.join(HERE, f"libpoismf_host_{name}.so")
            if force or jobs or _newer(out, [host_src, LIB] + hdrs):
                _run([HOSTCC, "-std=c99", "-O2", "-fPIC", "-shared", "-I", inc, host_src] + defs +
                     ["-o", out, "-L", HERE, "-lpoismf_b200", "-Wl,-rpath,$ORIGIN"])
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
