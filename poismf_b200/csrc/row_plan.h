// poismf_b200 — the half-sweep's row planner: which kernel solves a row of n non-zeros.
//
// Host-only arithmetic, no CUDA call: HandleT::plan (api.cu) uploads what plan_rows decides, half_sweep
// launches one kernel per bin, and the launchers (sweep_inst.cuh, sweep_regtile.cuh) instantiate the kernel
// a BinShape names.  The lock-step rows go to LockstepPlan (lockstep.h), which uploads lockstep_tables.
#pragma once
#include <algorithm>
#include <cstddef>
#include <cstdint>
#include <utility>
#include <vector>

#include "../../include/poismf_b200.h"
#include "sweep_consts.h"

namespace pmf {

enum class BinKind { RegTile, Warp, Cta, Cluster, Streaming };

// register-tile kernels (regtile.cuh): {warps per row, tile rows per lane}, capacity 8 x warps x tile rows.
// sweep_regtile.cuh instantiates one kernel per entry.
struct RegTileShape { int nw, tpl; };
constexpr RegTileShape REGTILE_SHAPES[] = {{1, 2}, {1, 3}, {1, 4}, {2, 3}, {2, 4}, {4, 3}, {4, 4},
                                           {8, 3}, {8, 4}, {16, 3}, {16, 4}};

// the kernel and launch geometry of one bin
struct BinShape {
    BinKind kind = BinKind::Warp;
    int lanes = 32;         // lanes per team: 16 or 32 for Warp (several teams per CTA), else the CTA's threads
    int threads = 256;      // per CTA
    int cap = 0;            // staged tile capacity per CTA; 0 = tile stays in global memory
    int acap = 0;           // capacity of the per-non-zero arrays kept in shared memory
    int cluster = 1;        // CTAs per row
    size_t slice = 0;       // shared bytes per team
    size_t smem = 0;        // dynamic shared bytes per CTA
    int rt_nw = 0, rt_tpl = 0, rt_nc = 0;   // RegTile: warps per row, tile rows per lane, 16-byte chunks per lane
};

struct PlanMode {
    int real_size = 4;           // sizeof(real)
    int ldf = 0, kp = 0;         // factor row stride, tile row stride (reals)
    int method = PMF_CG;
    bool strict = false;
    bool regtile = false;        // the register-tile kernels take the rows they can hold (float32 fast pg, cached cg)
    bool lockstep = false;       // the heaviest rows of cg under the register-tile conditions go to the lock-step path
    long long dense_min = 4096;          // lock-step rows have at least this many non-zeros
    long long dense_min_total = 250000;  // ... and at least this many together
};

// pmf_b200_bin_profile::block_team: -lanes for a (sub-)warp team, CTAs per row for CTA and cluster teams,
// 100 + warps per row for register tiles, LOCKSTEP_PROFILE_CODE for the lock-step path
constexpr int LOCKSTEP_PROFILE_CODE = 200;
inline int profile_code(const BinShape& b)
{
    switch (b.kind) {
    case BinKind::RegTile: return 100 + b.rt_nw;
    case BinKind::Warp: return -b.lanes;
    default: return b.cluster;
    }
}

// The bins of a mode, ascending capacity: a row goes to the first bin whose cap x cluster holds it, or to the
// last bin, whose tile stays in global memory.
inline std::vector<BinShape> bin_ladder(const PlanMode& m)
{
    const int nvec = m.method == PMF_PG ? 3 : (m.method == PMF_CG ? 7 : TN_NUM_VECS);
    const size_t rs = (size_t)m.real_size, kp = (size_t)m.kp;
    // shared bytes of one team; (sub-)warp teams need no reduction scratch: their 640 bytes go to the tile instead
    auto slice_bytes = [&](int team_threads, int cap) {
        const size_t b = (team_threads > 32 ? 640 : 0) + (size_t)team_threads * 16 + nvec * kp * rs +
                         (size_t)4 * cap * rs + (size_t)cap * kp * rs;
        return (b + 15) / 16 * 16;
    };
    std::vector<BinShape> bins;
    if (m.regtile) {
        for (const RegTileShape& s : REGTILE_SHAPES) {
            BinShape b;
            b.kind = BinKind::RegTile;
            b.rt_nw = s.nw; b.rt_tpl = s.tpl; b.rt_nc = m.ldf <= 32 ? 2 : 4;
            b.cap = b.acap = 8 * s.nw * s.tpl;
            b.threads = b.lanes = 32 * s.nw;
            bins.push_back(b);
        }
    } else {
        // {lanes per row, tile capacity}.  Rows in flight per SM are bounded by shared memory (tile + solver
        // state per row), so capacities are graded finely; a full warp per row gives the shortest per-row
        // latency, which is what bounds throughput at that occupancy.  64 lanes = a two-warp CTA per row: from
        // ~64 non-zeros on, shared memory leaves fewer than 16 rows in flight per SM and one warp per row no
        // longer hides the latencies (measured on B200).  Strict numerics: warp teams only.
        static constexpr int teams[9][2] = {{16, 16}, {32, 24}, {32, 32}, {32, 40}, {32, 48},
                                            {64, 64}, {64, 80}, {64, 96}, {64, 128}};
        for (const auto& t : teams) {
            BinShape b;
            b.lanes = m.strict ? 32 : t[0];
            b.cap = b.acap = t[1];
            if (b.lanes > 32) {
                b.kind = BinKind::Cta;
                b.threads = b.lanes;
                b.slice = b.smem = slice_bytes(b.lanes, b.cap);
                if (b.smem <= SMEM_CTA_MAX) bins.push_back(b);
                continue;
            }
            b.kind = BinKind::Warp;
            b.slice = slice_bytes(b.lanes, b.cap);
            // teams per CTA: whatever keeps the most rows in flight per SM under the shared-memory
            // (228 KB / SM, 1 KB reserved per CTA) and register (80 per thread) budgets
            int best_teams = 0, best_rows = 0;
            for (int teams = 256 / b.lanes; teams >= 1; teams >>= 1) {
                const size_t smem = b.slice * teams;
                if (smem > SMEM_CTA_MAX) continue;
                const int by_smem = (int)(SMEM_PER_SM / (smem + SMEM_CTA_RESERVED));
                const int by_regs = 65536 / (teams * b.lanes * WARP_KERNEL_REGS);
                const int by_thr = 2048 / std::max(teams * b.lanes, 32);
                const int ctas = std::min(std::min(by_smem, by_regs), std::min(by_thr, 32));
                if (ctas * teams > best_rows) { best_rows = ctas * teams; best_teams = teams; }
            }
            if (best_teams == 0) continue;
            b.threads = std::max(best_teams * b.lanes, 32);
            b.smem = b.slice * (b.threads / b.lanes);
            bins.push_back(b);
        }
    }
    // CTA-per-row bins: largest capacity with 4, 2, 1 resident CTAs per SM.  The one-per-SM bins (and the
    // clusters below) run 512 threads per CTA: their rows are long enough to feed them, and per-row latency is
    // what bounds these bins.
    const int ctas[3] = {4, 2, 1};
    int last_cap = bins.empty() ? 0 : bins.back().cap;
    for (int c = 0; c < 3; c++) {
        const int thr = (ctas[c] == 1 && !m.strict) ? 512 : 256;
        const size_t budget = std::min(SMEM_CTA_MAX, SMEM_PER_SM / ctas[c] - SMEM_CTA_RESERVED);
        const size_t fixed = slice_bytes(thr, 0) + 16;
        if (budget <= fixed) continue;
        int cap = (int)((budget - fixed) / ((kp + 4) * rs));
        cap = cap / 4 * 4;
        if (cap <= last_cap) continue;
        BinShape b;
        b.kind = BinKind::Cta;
        b.cap = b.acap = cap;
        b.threads = b.lanes = thr;
        b.slice = b.smem = slice_bytes(thr, cap);
        bins.push_back(b);
        last_cap = cap;
    }
    if (!m.strict) {
        // cluster-per-row bins: G CTAs stage G slices of the tile (fast numerics only)
        const int thr = 512;
        const size_t fixed = slice_bytes(thr, 0) + GANG_XBYTES + 16;
        int gcap = (int)((SMEM_CTA_MAX - fixed) / ((kp + 4) * rs));
        gcap = gcap / 4 * 4;
        for (int g : {2, 4, 8, 16}) {
            if (gcap <= 0) break;
            BinShape b;
            b.kind = BinKind::Cluster;
            b.cluster = g;
            b.cap = b.acap = gcap;
            b.threads = b.lanes = thr;
            b.slice = b.smem = slice_bytes(thr, gcap) + GANG_XBYTES;
            bins.push_back(b);
        }
        BinShape b;     // beyond 16 resident slices: 16 CTAs, each streaming its slice from L2
        b.kind = BinKind::Streaming;
        b.cluster = 16;
        b.cap = 0;
        b.acap = 4096;   // 64 KB (float) of per-non-zero arrays on chip; two such CTAs share an SM
        b.threads = b.lanes = thr;
        b.slice = b.smem = slice_bytes(thr, 0) + GANG_XBYTES + (size_t)4 * b.acap * rs;
        bins.push_back(b);
    } else {   // strict numerics: everything longer stays on one CTA, tile in global memory / L2
        BinShape b;
        b.kind = BinKind::Cta;
        b.cap = b.acap = 0;
        b.threads = b.lanes = 256;
        b.slice = b.smem = slice_bytes(256, 0);
        bins.push_back(b);
    }
    return bins;
}

// the most rows the lock-step path takes: its gaxpy pass keeps two tiles of DN_TILE_ROWS rows, one accumulator row
// per heavy row and the per-group edge slots in one CTA's shared memory
inline size_t lockstep_max_rows(const PlanMode& m)
{
    const size_t row = (size_t)m.ldf * m.real_size;
    return std::min<size_t>(1024, (SMEM_CTA_MAX - 1024) / row - 2 * DN_TILE_ROWS - DN_GROUPS);
}

struct PlannedBin {
    BinShape shape;
    std::vector<int> rows;       // local row ids, longest first (ties: ascending id)
    long long max_nnz = 0;
    unsigned long long nnz = 0;
};

struct RowPlan {
    std::vector<PlannedBin> bins;   // bin_ladder(mode), with their rows
    std::vector<int> empty;         // rows without non-zeros
    std::vector<int> lockstep;      // rows of the lock-step path, heaviest first (ties: ascending id)
};

// Bins the rows [0, n_rows) of one side: ptr are its row pointers, other_dim the rows of the fixed factor matrix.
inline RowPlan plan_rows(const PlanMode& m, const long long* ptr, size_t n_rows, size_t other_dim)
{
    auto len = [ptr](size_t r) { return ptr[r + 1] - ptr[r]; };
    RowPlan plan;
    for (const BinShape& s : bin_ladder(m)) plan.bins.push_back({s, {}, 0, 0});

    if (m.lockstep && m.regtile && m.method == PMF_CG) {
        std::vector<std::pair<long long, int>> cand;
        for (size_t r = 0; r < n_rows; r++)
            if (len(r) >= m.dense_min) cand.push_back({-len(r), (int)r});
        std::sort(cand.begin(), cand.end());          // heaviest first, ties by row id
        if (cand.size() > lockstep_max_rows(m)) cand.resize(lockstep_max_rows(m));
        // the lock-step phase costs ~30 launches per half-sweep whatever its size: below ~250k non-zeros the
        // per-row cluster teams are cheaper (small shards of a multi-GPU fit, the user side of config #2)
        long long nnzH = 0;
        for (auto& c : cand) nnzH -= c.first;
        // the lock-step tables index non-zeros and the T x H + 1 bounds of the (tile, heavy row) segments with
        // 32-bit integers
        const long long T = ((long long)other_dim + DN_TILE_ROWS - 1) / DN_TILE_ROWS;
        const bool fits = nnzH < (1LL << 31) && T * (long long)cand.size() + 1 <= INT32_MAX && ptr[n_rows] < (1LL << 31);
        if (nnzH >= m.dense_min_total && fits)
            for (auto& c : cand) plan.lockstep.push_back(c.second);
    }
    std::vector<char> is_lockstep(plan.lockstep.empty() ? 0 : n_rows, 0);
    for (int r : plan.lockstep) is_lockstep[r] = 1;

    for (size_t r = 0; r < n_rows; r++) {
        const long long n = len(r);
        if (n == 0) { plan.empty.push_back((int)r); continue; }
        if (!is_lockstep.empty() && is_lockstep[r]) continue;
        size_t bi = 0;
        while (bi + 1 < plan.bins.size() && n > (long long)plan.bins[bi].shape.cap * plan.bins[bi].shape.cluster) bi++;
        PlannedBin& b = plan.bins[bi];
        b.rows.push_back((int)r);
        b.max_nnz = std::max(b.max_nnz, n);
        b.nnz += (unsigned long long)n;
    }
    for (PlannedBin& b : plan.bins) {
        if (b.rows.size() < 2) continue;
        // longest first; counting sort (row lengths inside a bin span a small range)
        const long long mx = b.max_nnz;
        if (mx <= (1 << 22)) {
            std::vector<int> cnt((size_t)mx + 2, 0);
            for (int r : b.rows) cnt[(size_t)(mx - len(r)) + 1]++;
            for (size_t i = 1; i < cnt.size(); i++) cnt[i] += cnt[i - 1];
            std::vector<int> sorted(b.rows.size());
            for (int r : b.rows) sorted[(size_t)cnt[(size_t)(mx - len(r))]++] = r;
            b.rows.swap(sorted);
        } else {
            std::stable_sort(b.rows.begin(), b.rows.end(), [&](int a, int c) { return len(a) > len(c); });
        }
    }
    return plan;
}

// The host side of a lock-step plan (sweep_lockstep.cu): the tables every lock-step kernel indexes and the element
// count of every device array, for the lock-step rows `rows` of a side with row pointers ptr, a fixed matrix of
// other_dim rows of ldf reals and num_sms SMs.  plan_rows keeps T x H + 1, the non-zeros and the side's non-zeros
// below 2^31; ldf <= 64 and H <= 65535 are the path's own bounds (lockstep.h).
struct LockstepTables {
    int H = 0;          // heavy rows
    int T = 0;          // tiles of DN_TILE_ROWS rows of the fixed matrix
    int G = 0;          // persistent CTAs of the gaxpy pass
    int nnzH = 0;       // non-zeros of the heavy rows
    int nchunks = 0;    // line-search chunks of DN_LS_CHUNK non-zeros, none across two rows
    std::vector<int> i32;          // one block: hrow [H] | hcol0 [H+1] | chunk_ptr [H+1] | chunk_h [nchunks]
    std::vector<long long> hbeg;   // [H] first non-zero of each heavy row in the side's arrays
    // device arrays: hbeg and the per-row scalars hold H entries; ent, sx, p, q and the sort's temporaries nnzH
    size_t n_seg = 0;       // seg_ptr: T x H + 1
    size_t n_dvec = 0;      // dvec: H x ldf
    size_t n_hist = 0;      // gprev, dprev: H x 64
    size_t n_gpart = 0;     // gpart: G x H x ldf
    size_t n_lsp = 0;       // lsp: nchunks x DN_TRIALS
};

inline LockstepTables lockstep_tables(const long long* ptr, const std::vector<int>& rows, size_t other_dim,
                                      int num_sms, int ldf)
{
    LockstepTables t;
    const int H = t.H = (int)rows.size();
    const long long T = ((long long)other_dim + DN_TILE_ROWS - 1) / DN_TILE_ROWS;
    t.T = (int)T;
    t.G = (int)std::min<long long>(num_sms, T);
    t.hbeg.resize(H);
    std::vector<int> hcol0(H + 1, 0), chunk_ptr(H + 1, 0);
    for (int h = 0; h < H; h++) {
        const long long n = ptr[rows[h] + 1] - ptr[rows[h]];
        t.hbeg[h] = ptr[rows[h]];
        hcol0[h + 1] = hcol0[h] + (int)n;
        chunk_ptr[h + 1] = chunk_ptr[h] + (int)((n + DN_LS_CHUNK - 1) / DN_LS_CHUNK);
    }
    t.nnzH = hcol0[H];
    t.nchunks = chunk_ptr[H];
    t.i32 = rows;
    t.i32.insert(t.i32.end(), hcol0.begin(), hcol0.end());
    t.i32.insert(t.i32.end(), chunk_ptr.begin(), chunk_ptr.end());
    for (int h = 0; h < H; h++) t.i32.insert(t.i32.end(), (size_t)(chunk_ptr[h + 1] - chunk_ptr[h]), h);
    t.n_seg = (size_t)T * H + 1;
    t.n_dvec = (size_t)H * ldf;
    t.n_hist = (size_t)H * 64;
    t.n_gpart = (size_t)t.G * H * ldf;
    t.n_lsp = (size_t)t.nchunks * DN_TRIALS;
    return t;
}

}  // namespace pmf
