"""CPU checks of the half-sweep's row planner (poismf_b200/csrc/row_plan.h): the bin ladder of every mode, where each
row length goes, the order of the row lists, the lock-step rows and their host tables, and the profile codes.  A small driver over the
header is compiled with the host C++ compiler; no CUDA call is made."""
import os
import shutil
import subprocess

import numpy as np
import pytest

import row_bins as rb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PG, CG, TNCG = 3, 2, 1
KS = (1, 3, 32, 33, 50, 64, 65, 100, 200, 256)

DRIVER = r"""
#include "row_plan.h"
#include <cstdio>
#include <cstdlib>
#include <cstring>
using namespace pmf;
static const char* kind_name[] = {"regtile", "warp", "cta", "cluster", "streaming"};
static PlanMode mode(int rs, int k, int method, bool strict, bool regtile)
{
    PlanMode m;
    const int V = 16 / rs;
    int units = (k + V - 1) / V;
    m.real_size = rs; m.ldf = units * V;
    if (units % 2 == 0) units++;
    m.kp = units * V; m.method = method; m.strict = strict; m.regtile = regtile;
    return m;
}
int main(int argc, char** argv)
{
    if (!strcmp(argv[1], "ladders")) {
        const int ks[] = {1, 3, 32, 33, 50, 64, 65, 100, 200, 256};
        const char* vn[5] = {"pg", "cg_cached", "cg_uncached", "cg_nolimit", "tncg"};
        const int vm[5] = {PMF_PG, PMF_CG, PMF_CG, PMF_CG, PMF_TNCG};
        for (int rs : {4, 8})
            for (int k : ks)
                for (int v = 0; v < 5; v++)
                    for (int s = 0; s < 2; s++) {
                        PlanMode m = mode(rs, k, vm[v], s, false);
                        m.regtile = rs == 4 && !s && m.ldf <= 64 && v <= 1;   // what HandleT::plan_mode decides
                        printf("%s %d %s %s:", rs == 4 ? "f32" : "f64", k, vn[v], s ? "strict" : "fast");
                        for (const BinShape& b : bin_ladder(m))
                            printf(" %s,%d,%d,%d,%d,%d,%zu", kind_name[(int)b.kind], b.lanes, b.threads, b.cap, b.acap,
                                   b.cluster, b.smem);
                        printf("\n");
                    }
        return 0;
    }
    if (!strcmp(argv[1], "tables")) {
        // tables <other_dim> <num_sms> <ldf>; stdin: n, n row lengths, then the lock-step rows
        std::vector<long long> ptr(1, 0);
        long long n = 0, v;
        if (scanf("%lld", &n) != 1) return 1;
        for (long long i = 0; i < n && scanf("%lld", &v) == 1; i++) ptr.push_back(ptr.back() + v);
        std::vector<int> rows;
        while (scanf("%lld", &v) == 1) rows.push_back((int)v);
        const LockstepTables t = lockstep_tables(ptr.data(), rows, (size_t)strtoull(argv[2], nullptr, 10), atoi(argv[3]),
                                                 atoi(argv[4]));
        printf("%d %d %d %d %d %zu %zu %zu %zu %zu\n", t.H, t.T, t.G, t.nnzH, t.nchunks, t.n_seg, t.n_dvec, t.n_hist,
               t.n_gpart, t.n_lsp);
        for (int x : t.i32) printf(" %d", x);
        printf("\n");
        for (long long x : t.hbeg) printf(" %lld", x);
        printf("\n");
        return 0;
    }
    // plan <real size> <k> <method> <strict> <regtile> <lockstep> <dense_min> <dense_min_total> <other_dim>,
    // row lengths on stdin
    PlanMode m = mode(atoi(argv[2]), atoi(argv[3]), atoi(argv[4]), atoi(argv[5]), atoi(argv[6]));
    m.lockstep = atoi(argv[7]); m.dense_min = atoll(argv[8]); m.dense_min_total = atoll(argv[9]);
    std::vector<long long> ptr(1, 0);
    long long n;
    while (scanf("%lld", &n) == 1) ptr.push_back(ptr.back() + n);
    const RowPlan p = plan_rows(m, ptr.data(), ptr.size() - 1, (size_t)strtoull(argv[10], nullptr, 10));
    printf("hmax %zu\n", lockstep_max_rows(m));
    for (const PlannedBin& b : p.bins) {
        printf("bin %s %d %d %d %d %lld %llu :", kind_name[(int)b.shape.kind], b.shape.lanes, b.shape.cap,
               b.shape.cluster, profile_code(b.shape), b.max_nnz, b.nnz);
        for (int r : b.rows) printf(" %d", r);
        printf("\n");
    }
    printf("empty :");
    for (int r : p.empty) printf(" %d", r);
    printf("\nlockstep :");
    for (int r : p.lockstep) printf(" %d", r);
    printf("\n");
    return 0;
}
"""


@pytest.fixture(scope="module")
def driver(tmp_path_factory):
    cxx = shutil.which("g++", path="/usr/bin:" + os.environ.get("PATH", "")) or shutil.which("c++")
    cuda_inc = "/usr/local/cuda/include"
    if cxx is None:
        pytest.skip("needs a host C++ compiler")
    d = tmp_path_factory.mktemp("row_plan")
    (d / "t.cpp").write_text(DRIVER)
    exe = d / "t"
    subprocess.run([cxx, "-std=c++17", "-O2", "-I", cuda_inc,
                    "-I", os.path.join(ROOT, "poismf_b200", "csrc"), str(d / "t.cpp"), "-o", str(exe)], check=True)
    return str(exe)


def _plan(driver, lengths, rs=4, k=32, method=CG, strict=False, regtile=False, lockstep=False, dense_min=4096,
          dense_min_total=250000, other=100000):
    args = [driver, "plan"] + [str(int(v)) for v in (rs, k, method, strict, regtile, lockstep, dense_min,
                                                      dense_min_total, other)]
    out = subprocess.run(args, input=" ".join(str(int(n)) for n in lengths), capture_output=True, text=True,
                         check=True).stdout.splitlines()
    plan = {"hmax": int(out[0].split()[1]), "bins": []}
    for line in out[1:]:
        head, rows = line.split(":")
        rows = [int(r) for r in rows.split()]
        f = head.split()
        if f[0] == "bin":
            plan["bins"].append(dict(kind=f[1], lanes=int(f[2]), cap=int(f[3]), cluster=int(f[4]), code=int(f[5]),
                                     max_nnz=int(f[6]), nnz=int(f[7]), rows=rows))
        else:
            plan[f[0]] = rows
    return plan


def test_golden_ladders(driver):
    """Every mode's ladder (kind, lanes, threads, cap, acap, cluster, dynamic smem) is the committed one."""
    with open(os.path.join(ROOT, "tests", "golden", "row_ladders.txt")) as f:
        want = [line.rstrip("\n") for line in f if not line.startswith("#")]
    got = subprocess.run([driver, "ladders"], capture_output=True, text=True, check=True).stdout.splitlines()
    assert len(got) == len(want) == 2 * len(KS) * 5 * 2
    for g, w in zip(got, want):
        assert g == w
    # strict numerics compile no 16-lane kernel: the cap-16 bin is a full warp's
    for line in got:
        if "strict" in line:
            assert line.split(": ")[1].startswith("warp,32,") and "warp,16," not in line


def _check_order(plan, lengths):
    for b in plan["bins"]:
        key = [(-lengths[r], r) for r in b["rows"]]
        assert key == sorted(key), b["kind"]                      # longest first, ties by ascending row id
        if b["rows"]:
            assert b["max_nnz"] == max(lengths[r] for r in b["rows"])
            assert b["nnz"] == sum(int(lengths[r]) for r in b["rows"])


@pytest.mark.parametrize("rs,k,method,strict,regtile", [
    (4, 32, PG, False, True),          # register tiles, CTA, clusters, streaming
    (4, 64, CG, False, True),
    (4, 65, CG, False, False),         # 16-lane warp teams, two-warp CTAs
    (4, 3, TNCG, True, False),         # strict: 32-lane teams, CTA bins, the global-memory CTA bin
    (8, 200, CG, False, False),
    (8, 256, TNCG, True, False),
])
def test_row_assignment(driver, rs, k, method, strict, regtile):
    """Every length 1..40 000 (twice, for ties) lands in the first bin whose cap x cluster holds it, or in the
    last bin; empty rows are listed; lists come longest first with ties by ascending row id."""
    lengths = np.concatenate([np.arange(0, 40001), np.arange(0, 40001)])
    np.random.default_rng(k).shuffle(lengths)
    plan = _plan(driver, lengths, rs, k, method, strict, regtile)
    bins = plan["bins"]
    assert plan["empty"] == sorted(np.flatnonzero(lengths == 0).tolist())
    assert plan["lockstep"] == []
    where = {}
    for i, b in enumerate(bins):
        for r in b["rows"]:
            assert r not in where
            where[r] = i
    assert len(where) + len(plan["empty"]) == lengths.shape[0]
    for r, i in where.items():
        n = lengths[r]
        first = next((j for j, b in enumerate(bins) if n <= b["cap"] * b["cluster"]), len(bins) - 1)
        assert i == min(first, len(bins) - 1), (n, i, first)
    assert bins[-1]["cap"] == 0 and bins[-1]["rows"]           # the last bin: tile in global memory
    assert bins[0]["kind"] == ("regtile" if regtile else "warp")
    if strict:
        assert all(b["kind"] in ("warp", "cta") for b in bins) and all(b["lanes"] != 16 for b in bins)
    _check_order(plan, lengths)


def test_row_order_past_counting_sort(driver):
    """A bin whose longest row has more than 2^22 non-zeros is sorted by comparison: same order."""
    lengths = np.array([5_000_000, 3, 4_500_000, 5_000_000, 0, 4_500_000, 70_000, 5_000_000])
    plan = _plan(driver, lengths, 4, 32, PG, False, True)
    last = plan["bins"][-1]
    assert last["kind"] == "streaming" and last["max_nnz"] > 2**22
    assert last["rows"] == [0, 3, 7, 2, 5, 6]
    _check_order(plan, lengths)


def _lockstep_case(n_heavy=400, heavy=(600, 1500), light=599, seed=0):
    rng = np.random.default_rng(seed)
    lengths = np.concatenate([rng.integers(heavy[0], heavy[1], n_heavy), rng.integers(0, light + 1, 2000),
                              np.full(40, 1200)])                     # ties among the heavy rows
    rng.shuffle(lengths)
    return lengths


def test_lockstep_rows(driver):
    """The heaviest rows with at least dense_min non-zeros, at most hmax of them, ties by row id, go to the lock-step
    path and to no bin."""
    for k, n_heavy in ((64, 400), (64, 100), (32, 1100)):
        lengths = _lockstep_case(n_heavy)
        plan = _plan(driver, lengths, 4, k, CG, False, True, lockstep=True, dense_min=600, dense_min_total=0)
        ldf = (k + 3) // 4 * 4
        hmax = min(1024, (232448 - 1024) // (ldf * 4) - 2 * 256 - 64)
        assert plan["hmax"] == hmax
        cand = sorted((-int(n), r) for r, n in enumerate(lengths) if n >= 600)
        want = [r for _, r in cand[:hmax]]
        assert plan["lockstep"] == want and len(want) == min(hmax, len(cand))
        binned = [r for b in plan["bins"] for r in b["rows"]]
        assert not set(binned) & set(want)
        assert len(binned) + len(want) + len(plan["empty"]) == lengths.shape[0]
        _check_order(plan, lengths)


def test_no_lockstep_rows(driver):
    """No lock-step rows below dense_min_total, without lock-step, outside cached cg on register tiles, or when the
    lock-step tables would overflow their 32-bit indices."""
    lengths = _lockstep_case()
    on = dict(rs=4, k=64, method=CG, regtile=True, lockstep=True, dense_min=600)
    rows = _plan(driver, lengths, **on, dense_min_total=0)["lockstep"]
    heavy = int(lengths[rows].sum())
    assert _plan(driver, lengths, **on, dense_min_total=heavy)["lockstep"] == rows
    assert _plan(driver, lengths, **on, dense_min_total=heavy + 1)["lockstep"] == []
    assert _plan(driver, lengths, **dict(on, lockstep=False), dense_min_total=0)["lockstep"] == []
    assert _plan(driver, lengths, **dict(on, regtile=False), dense_min_total=0)["lockstep"] == []
    assert _plan(driver, lengths, **dict(on, method=PG), dense_min_total=0)["lockstep"] == []
    # the T x H + 1 bounds of the (tile of the fixed matrix, heavy row) segments must fit an int32: T x H <= 2^31 - 2
    # (328 heavy rows at k = 64)
    tiles = (2**31 - 2) // 328
    assert _plan(driver, lengths, **on, dense_min_total=0, other=256 * tiles)["lockstep"]
    assert _plan(driver, lengths, **on, dense_min_total=0, other=256 * (tiles + 1))["lockstep"] == []
    one = np.zeros(100, dtype=np.int64)
    one[7] = 5000
    assert _plan(driver, one, **on, dense_min_total=0, other=256 * (2**31 - 2))["lockstep"] == [7]
    assert _plan(driver, one, **on, dense_min_total=0, other=256 * (2**31 - 2) + 1)["lockstep"] == []
    # the side's non-zeros >= 2^31 while the heavy rows' are not
    big = np.full(2400, 1_000_000)
    assert _plan(driver, big[:2000], **on, dense_min_total=0)["lockstep"]
    assert _plan(driver, big, **on, dense_min_total=0)["lockstep"] == []


def _tables(driver, lengths, rows, other, sms, ldf):
    out = subprocess.run([driver, "tables", str(other), str(sms), str(ldf)],
                         input=" ".join(str(int(v)) for v in [len(lengths), *lengths, *rows]),
                         capture_output=True, text=True, check=True).stdout.split("\n")
    return [int(v) for v in out[0].split()], [int(v) for v in out[1].split()], [int(v) for v in out[2].split()]


def _tables_ref(lengths, rows, other, sms, ldf):
    """numpy restatement of lockstep_tables: sizes, the int32 block hrow | hcol0 | chunk_ptr | chunk_h, hbeg, and the
    element counts of seg_ptr, dvec, gprev / dprev, gpart and lsp."""
    lengths, rows = np.asarray(lengths, dtype=np.int64), np.asarray(rows, dtype=np.int64)
    ptr = np.concatenate([[0], np.cumsum(lengths)])
    n = lengths[rows]
    H, T = len(rows), -(-other // 256)
    G = min(sms, T)
    hcol0 = np.concatenate([[0], np.cumsum(n)])
    chunks = -(-n // 2048)
    chunk_ptr = np.concatenate([[0], np.cumsum(chunks)])
    nchunks = int(chunk_ptr[-1])
    sizes = [H, T, G, int(hcol0[-1]), nchunks, T * H + 1, H * ldf, H * 64, G * H * ldf, nchunks * 20]
    i32 = np.concatenate([rows, hcol0, chunk_ptr, np.repeat(np.arange(H), chunks)])
    return sizes, i32.tolist(), ptr[rows].tolist()


@pytest.mark.parametrize("case", ["one_row", "many_rows", "chunk_edges", "odd_tiles", "few_tiles"])
def test_lockstep_tables(driver, case):
    """lockstep_tables gives the numpy restatement's tables and device array sizes: one heavy row, many rows, row
    lengths at multiples of the line-search chunk and one either side, fixed sides of no whole number of tiles, and
    fewer tiles than SMs (the gaxpy pass then runs one CTA per tile)."""
    rng = np.random.default_rng(len(case))
    lengths = rng.integers(0, 3000, 5000)
    other, sms, ldf = 160_000, 148, 52
    if case == "one_row":
        lengths[123] = 300_000
        rows = [123]
    elif case == "many_rows":
        lengths[rng.choice(5000, 400, replace=False)] = rng.integers(4096, 60_000, 400)
        rows = np.argsort(-lengths, kind="stable")[:400]
    elif case == "chunk_edges":
        edges = [m * 2048 + d for m in (1, 2, 3, 7) for d in (-1, 0, 1)] + [1, 2048 * 16]
        rows = rng.choice(5000, len(edges), replace=False)
        lengths[rows] = edges
    elif case == "odd_tiles":
        rows = np.argsort(-lengths, kind="stable")[:50]
        other, ldf = 100_001, 64
    else:
        rows = np.argsort(-lengths, kind="stable")[:30]
        other, ldf = 255 + 256 * 20, 16
    got = _tables(driver, lengths, rows, other, sms, ldf)
    want = _tables_ref(lengths, rows, other, sms, ldf)
    assert got == want
    if case == "few_tiles":
        assert got[0][2] == got[0][1] == 21
    if case == "chunk_edges":
        assert got[0][4] == sum(-(-e // 2048) for e in edges)


@pytest.mark.parametrize("rs,k,method,strict,regtile", [
    (4, 32, PG, False, True), (4, 65, CG, False, False), (8, 33, TNCG, True, False)])
def test_profile_codes(driver, rs, k, method, strict, regtile):
    """profile_code gives what tests/row_bins.bin_kind decodes for each kind."""
    plan = _plan(driver, [1], rs, k, method, strict, regtile)
    for b in plan["bins"]:
        got = rb.bin_kind({"block_team": b["code"], "cap": b["cap"]})
        want = {"regtile": f"regtile{b['lanes'] // 32}w:{b['cap']}", "warp": f"warp{b['lanes']}:{b['cap']}",
                "cta": f"cta:{b['cap']}", "cluster": f"cluster{b['cluster']}", "streaming": "streaming"}[b["kind"]]
        assert got == want
