// poismf_b200 — the heaviest rows of a half-sweep, solved in LOCK-STEP by the whole GPU.
//
// Power-law count matrices have a few rows (items of the CSC side, mostly) that touch a large
// fraction of the opposite factor matrix: the 65 heaviest items of the Last.FM-shaped synthetic
// hold 18 % of all non-zeros, the heaviest alone reaches 75 % of the users.  Giving such a row to
// one team (a cluster of 16 CTAs at most) leaves 9/10 of the GPU idle on the critical path and
// re-gathers hundreds of MB of factor rows through L2 on every tile pass.
//
// Here the H heaviest rows of a side advance through the cg iterations TOGETHER, and every phase
// of an iteration is one kernel over ALL their non-zeros:
//
//   * The non-zeros of the heavy rows are sorted once per matrix by (tile of the fixed matrix,
//     heavy row): a CTA walks a contiguous range of that order, so the factor rows it gathers come
//     from a few consecutive TILES of the fixed matrix (256 rows, 53 KB at k = 50).  A tile is
//     contiguous in memory: ONE TMA bulk copy (cp.async.bulk -> mbarrier) puts it in shared memory,
//     and every heavy row with non-zeros in the tile re-uses it: the fixed matrix crosses L2 -> SM
//     once per pass (72 MB for A at config #2) instead of once per non-zero (596 MB).
//   * dots pass   : <v_h, F_t> for the current vectors v (x or d); results go to per-non-zero arrays
//                   p / q kept in the row's own (compact CSC) order.
//   * gaxpy pass  : per-CTA accumulators G[h] in shared memory (no atomics: deterministic), folded
//                   over CTAs in a fixed order by the k-phase kernel.  The accepted step of the
//                   previous iteration is applied to p on the way (p += step q), so c_t = -x_t / p_t
//                   needs no pass of its own.  (Both passes: dense_walk_kernel below.)
//   * line search : O(n) as in solve_cg_cached: a streaming kernel over p, q, x evaluates all 20 trial
//                   steps (smax 4^-j) in one pass; the first acceptable one in sequence order wins,
//                   like the sequential search of nonnegcg.c:297-327.
//   * k phase     : one warp per heavy row does the direction update and every k-scalar.
//
// Same arithmetic as solve_cg_cached (fast numerics, float32, limit_step, w_mult == 1); the
// summation order over a row's non-zeros is fixed by the sort, so results are reproducible run to run.
#pragma once
#include "rowops.cuh"
#include "sweep_consts.h"

namespace pmf {

constexpr int DN_MAX_LS = 20, DN_MAX_NFEVAL = 150;

// ---- TMA bulk copy (cp.async.bulk, global -> shared, completion on an mbarrier) ---------------------
PMF_DEVINL unsigned dn_smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
PMF_DEVINL void dn_mbar_init(unsigned long long* bar, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(dn_smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
PMF_DEVINL void dn_tile_load(void* dst, const void* src, unsigned bytes, unsigned long long* bar)
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // earlier generic reads of dst are done (barrier)
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(dn_smem_u32(bar)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dn_smem_u32(dst)), "l"(src), "r"(bytes), "r"(dn_smem_u32(bar)) : "memory");
}
PMF_DEVINL void dn_mbar_wait(unsigned long long* bar, unsigned phase)
{
    unsigned ok;
    do {
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                     : "=r"(ok) : "r"(dn_smem_u32(bar)), "r"(phase) : "memory");
    } while (!ok);
}

struct DenseScal {          // per heavy row
    float fcur, regx, gprev_sq, step_applied;
    float gd, dsq, gg, lin, smax;
    float steps[DN_TRIALS];
    int active, it, nfe, pad;
};

struct DenseParams {
    int H, T, U, ldf, k, L;
    int nnzH, nchunks, G;               // G = CTAs of the gaxpy pass (= rows of gpart)
    int R;                              // rows of the fixed matrix F
    const float* F;                     // fixed factors
    float* M;                           // factors being updated (local row 0 of this side)
    const float* xv;                    // the side's non-zero values
    const float* csum;
    const int* hrow;                    // [H] local row ids, heaviest first
    const long long* hbeg;              // [H] first non-zero of the row in the side's arrays
    const int* hcol0;                   // [H+1] offsets of the rows in the compact per-non-zero arrays
    const uint2* ent;                   // [nnzH] sorted order: (byte offset of the row of F within its tile << 16 | heavy row
                                        //                       slot, index into the compact arrays p, q)
    const float* sx;                    // [nnzH] sorted order: the non-zero's value
    const int* seg_ptr;                 // [T*H+1] (tile, heavy row) segments of the sorted order
    const int* chunk_h;                 // [nchunks] heavy row of a line-search chunk
    const int* chunk_ptr;               // [H+1] first chunk of a heavy row
    float *p, *q;                       // [nnzH] <x,F_t>, <d,F_t>   (compact order)
    float *dvec;                        // [H][ldf] search directions
    float *gprev, *dprev;               // [H][64]
    float* gpart;                       // [G][H][ldf]
    float* lsp;                         // [nchunks][DN_TRIALS]
    DenseScal* sc;                      // [H]
    int* tile_counter;                  // dots passes: tiles are handed out dynamically (zeroed before the launch)
    HalfSweepConsts<float> hc;
    float* peerM[7];
    int npeers;
};

// ---- the two tile passes ---------------------------------------------------------------------------
// MODE 0: p_t = <x_h, F_t>   MODE 1: q_t = <d_h, F_t>   MODE 2: G[h] = sum_t c_t F_t, c_t = -x_t / p_t with p
// advanced by the step accepted in the previous iteration on the way.
//
// A persistent CTA walks a contiguous range of TILES of the fixed matrix.  Each tile (U consecutive
// rows: contiguous memory) is brought into shared memory by ONE TMA bulk copy, double-buffered so that
// the next tile lands while this one is used.  The tile's non-zeros — a contiguous range of the sorted
// order, 8 bytes per entry — are split EVENLY over the CTA's groups of 16 lanes, whatever segments they
// belong to.  A group takes 16 entries at a time: lane j loads (and, for the gaxpy pass, prepares the
// coefficient of) entry j, then the 16 entries are visited in turn with lane = 16-byte chunk of the
// factor row, so a whole row of the tile is one conflict-free LDS.128.
//   dots : per non-zero one LDS.128 + 4 FMA per lane; four non-zeros are folded across the 16 lanes
//          at once (transposing reduction: 5 shuffles) so that the sum of entry j ends in lane j, which
//          stores it; v_h stays in registers while h does not change
//   gaxpy: per non-zero one LDS.128 + 4 FMA per lane into a register accumulator, flushed to the CTA's
//          shared G[h] when the heavy row changes.  A run of one heavy row that STARTS inside a group's
//          range is added by that group alone; the run a group inherits from its predecessor goes to a
//          per-group edge slot, folded in group order after the barrier: no atomics, fixed order.
template <int MODE> struct DnWalk {
    static constexpr int threads = MODE == 2 ? 1024 : 256;     // gaxpy: one CTA per SM (its G[h] fill shared memory)
    static constexpr int groups = threads / 16;
    static constexpr int nbuf = MODE == 2 ? 2 : 1;             // dots: four CTAs per SM hide each other's tile copies
    static constexpr int min_ctas = MODE == 2 ? 1 : 4;
};
static_assert(DnWalk<2>::groups == DN_GROUPS, "the planner sizes the gaxpy pass with DN_GROUPS");

template <int MODE>
__global__ void __launch_bounds__(DnWalk<MODE>::threads, DnWalk<MODE>::min_ctas) dense_walk_kernel(const DenseParams P)
{
    constexpr int NBUF = DnWalk<MODE>::nbuf, NGROUPS = DnWalk<MODE>::groups;
    extern __shared__ __align__(128) unsigned char dn_smem[];
    __shared__ __align__(8) unsigned long long bar[2];
    __shared__ int edge_h[NGROUPS];
    const int ldf = P.ldf, L = P.L, H = P.H;
    const size_t tile_floats = (size_t)P.U * ldf;
    float* tiles = reinterpret_cast<float*>(dn_smem);
    float* Gacc = tiles + NBUF * tile_floats;                            // MODE 2: [H][ldf], then the edge slots
    float* edge_acc = Gacc + (size_t)H * ldf;
    int* hrow_s = reinterpret_cast<int*>(tiles + NBUF * tile_floats);   // MODE 0: rows of M holding the points
    if (MODE == 2) for (int i = threadIdx.x; i < H * ldf; i += blockDim.x) Gacc[i] = 0.f;
    if (MODE == 0) for (int i = threadIdx.x; i < H; i += blockDim.x) hrow_s[i] = P.hrow[i];
    const int tau0 = (int)((long long)P.T * blockIdx.x / gridDim.x), tau1 = (int)((long long)P.T * (blockIdx.x + 1) / gridDim.x);
    if (threadIdx.x == 0) { dn_mbar_init(&bar[0], 1); dn_mbar_init(&bar[1], 1); }
    __syncthreads();
    auto issue = [&](int tau, int b) {
        const int row0 = tau * P.U, nrows = min(P.U, P.R - row0);
        dn_tile_load(tiles + (size_t)b * tile_floats, P.F + (size_t)row0 * ldf, (unsigned)((size_t)nrows * ldf * sizeof(float)), &bar[b]);
    };
    if (NBUF == 2 && threadIdx.x == 0 && tau0 < tau1) issue(tau0, 0);
    const int lane = threadIdx.x & 31, cl = lane & 15, hbit = lane & 16;
    const int group = threadIdx.x >> 4;
    const bool chunk_ok = cl < L;
    const unsigned clo = chunk_ok ? (unsigned)cl * 16u : 0u;          // lanes beyond the row read chunk 0 (and discard)
    float* out = MODE == 0 ? P.p : P.q;
    int nload = 0;
    __shared__ int next_tile;
    for (int tau = tau0;; tau++) {
        if (NBUF == 2) {
            if (tau >= tau1) break;
        } else {
            // the dots passes accumulate nothing across tiles: tiles are drawn from a counter (no tail of idle CTAs)
            if (threadIdx.x == 0) next_tile = atomicAdd(P.tile_counter, 1);
            __syncthreads();
            tau = next_tile;
            __syncthreads();
            if (tau >= P.T) break;
        }
        const int n0 = P.seg_ptr[(size_t)tau * H], n1 = P.seg_ptr[(size_t)(tau + 1) * H];
        const int nb = n1 - n0;
        int b, phase;
        if (NBUF == 2) {
            b = (tau - tau0) & 1; phase = ((tau - tau0) >> 1) & 1;
            if (threadIdx.x == 0 && tau + 1 < tau1) issue(tau + 1, b ^ 1);   // that buffer was released by the last barrier
        } else {
            if (nb == 0) continue;
            b = 0; phase = nload & 1; nload++;
            if (threadIdx.x == 0) issue(tau, 0);
        }
        if (MODE == 2 && cl == 0) edge_h[group] = -1;
        // group g takes entries [r0, r1) of the tile's range; m is CTA-uniform
        const int m = (((nb + NGROUPS - 1) / NGROUPS) + 3) & ~3;
        const int r0 = n0 + min(nb, group * m), r1 = n0 + min(nb, (group + 1) * m);
        const unsigned tbase = dn_smem_u32(tiles + (size_t)b * tile_floats) + clo;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f), vv = acc;
        int hcur = -1;
        bool first = true;
        auto flush = [&]() {
            if (hcur < 0) return;
            if (chunk_ok) {
                if (first) {
                    *(reinterpret_cast<float4*>(edge_acc + (size_t)group * ldf) + cl) = acc;
                    if (cl == 0) edge_h[group] = hcur;
                } else {
                    float4* gq = reinterpret_cast<float4*>(Gacc + (size_t)hcur * ldf) + cl;
                    float4 v = *gq;
                    vaddto(v, acc);
                    *gq = v;
                }
            }
            first = false;
        };
        bool waited = false;
        // Entry loads run two batches ahead, the loads that depend on them (row state, p, q, value) one batch
        // ahead, so that their latency is covered by the visits of the current batch.
        // lane j of the group loads entry j of a batch.  Beyond the group's range its own last entry (for an
        // empty range: the tile's last entry) stands in with a zero coefficient / no output, so that the
        // inner loop has nothing to test and no heavy row gets a second writer.
        struct Dep { int active; float step, pt, qt, x; };
        const int last_valid = (r1 > r0 ? r1 : n1) - 1;
        auto load_ent = [&](int u) {
            const int mine = r0 + u + cl;
            return __ldg(P.ent + ((mine < r1 && u < m) ? mine : last_valid));
        };
        auto load_dep = [&](const uint2& e, int u) {
            Dep d;
            const DenseScal& S = P.sc[e.x & 0xffffu];
            d.active = S.active;
            d.step = 0.f; d.pt = 1.f; d.qt = 0.f; d.x = 0.f;
            if (MODE == 2) {
                const int mine = r0 + u + cl;
                d.step = S.step_applied;
                d.pt = P.p[e.y];
                d.qt = P.q[e.y];
                d.x = __ldg(P.sx + ((mine < r1 && u < m) ? mine : last_valid));
            }
            return d;
        };
        uint2 e0 = make_uint2(0u, 0u), e1 = e0;
        Dep d0 = {};
        if (nb > 0) { e0 = load_ent(0); d0 = load_dep(e0, 0); e1 = load_ent(16); }
        for (int u = 0; u < m && nb > 0; u += 16) {
            const uint2 e = e0;
            const Dep d = d0;
            e0 = e1;
            if (u + 16 < m) d0 = load_dep(e0, u + 16);
            if (u + 32 < m) e1 = load_ent(u + 32);
            const int mine = r0 + u + cl;
            const bool real = mine < r1;
            const unsigned off = e.x >> 16;
            const int h = (int)(e.x & 0xffffu);
            unsigned cp = e.y;
            float c = 0.f;
            if (MODE == 2) {
                if (real && d.active) {
                    float pt = d.pt;
                    if (d.step != 0.f) { pt = fmaf(d.step, d.qt, pt); P.p[cp] = pt; }
                    c = -d.x / pt;
                }
            } else if (!real || !d.active) cp = 0xffffffffu;
            if (!waited) { dn_mbar_wait(&bar[b], (unsigned)phase); waited = true; }
            if (MODE == 2) {
#pragma unroll 4
                for (int j = 0; j < 16; j++) {
                    const int hj = __shfl_sync(0xffffffffu, h, hbit | j);
                    const unsigned oj = __shfl_sync(0xffffffffu, off, hbit | j);
                    const float cj = __shfl_sync(0xffffffffu, c, hbit | j);
                    if (hj != hcur) { flush(); hcur = hj; acc = make_float4(0.f, 0.f, 0.f, 0.f); }
                    float4 f;
                    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(f.x), "=f"(f.y), "=f"(f.z), "=f"(f.w) : "r"(tbase + oj));
                    vfma(acc, cj, f);
                }
            } else {
#pragma unroll
                for (int s4 = 0; s4 < 4; s4++) {
                    float pend[4];
#pragma unroll
                    for (int v = 0; v < 4; v++) {
                        const int j = 4 * s4 + v;
                        const int hj = __shfl_sync(0xffffffffu, h, hbit | j);
                        const unsigned oj = __shfl_sync(0xffffffffu, off, hbit | j);
                        {   // v_h is re-read (predicated, no branch) when the heavy row changes
                            const float* vb = (MODE == 0 ? P.M + (size_t)hrow_s[hj] * ldf : P.dvec + (size_t)hj * ldf) + (clo >> 2);
                            asm volatile("{ .reg .pred p; setp.ne.s32 p, %5, %6;\n"
                                         "  @p ld.global.v4.f32 {%0,%1,%2,%3}, [%4]; }"
                                         : "+f"(vv.x), "+f"(vv.y), "+f"(vv.z), "+f"(vv.w) : "l"(vb), "r"(hj), "r"(hcur));
                            hcur = hj;
                        }
                        float4 f;
                        asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(f.x), "=f"(f.y), "=f"(f.z), "=f"(f.w) : "r"(tbase + oj));
                        pend[v] = vdot4(f, vv, 0.f);
                    }
                    // fold the four partial dot products over the 16 lanes; the sum of entry 4 s4 + v ends in
                    // the lanes with (b1 b0) = v, of which lane 4 s4 + v is the one that loaded the entry
                    const bool b1 = (cl & 2) != 0, b0 = (cl & 1) != 0;
                    if (!chunk_ok) { pend[0] = 0.f; pend[1] = 0.f; pend[2] = 0.f; pend[3] = 0.f; }
                    float k0 = b1 ? pend[2] : pend[0], k1 = b1 ? pend[3] : pend[1];
                    const float s0 = b1 ? pend[0] : pend[2], s1 = b1 ? pend[1] : pend[3];
                    k0 += __shfl_xor_sync(0xffffffffu, s0, 2);
                    k1 += __shfl_xor_sync(0xffffffffu, s1, 2);
                    float kk = b0 ? k1 : k0;
                    const float ss = b0 ? k0 : k1;
                    kk += __shfl_xor_sync(0xffffffffu, ss, 1);
                    kk += __shfl_xor_sync(0xffffffffu, kk, 4);
                    kk += __shfl_xor_sync(0xffffffffu, kk, 8);
                    if ((cl >> 2) == s4 && cp != 0xffffffffu) out[cp] = kk;
                }
            }
        }
        if (!waited) dn_mbar_wait(&bar[b], (unsigned)phase);
        if (MODE == 2) {
            flush();
            __syncthreads();
            {   // edge slots: runs of one heavy row sit in consecutive groups; the first group of a run
                // folds the run's slots in group order (fixed order, no two writers of one G[h])
                const int h = edge_h[group];
                if (h >= 0 && (group == 0 || edge_h[group - 1] != h) && chunk_ok) {
                    float4* gq = reinterpret_cast<float4*>(Gacc + (size_t)h * ldf) + cl;
                    float4 v = *gq;
                    for (int g = group; g < NGROUPS && edge_h[g] == h; g++)
                        vaddto(v, *(reinterpret_cast<const float4*>(edge_acc + (size_t)g * ldf) + cl));
                    *gq = v;
                }
            }
        }
        __syncthreads();                            // everybody is done with this tile's buffer
    }
    if (MODE == 2) {
        float4* outp = reinterpret_cast<float4*>(P.gpart + (size_t)blockIdx.x * H * ldf);
        for (int i = threadIdx.x; i < H * L; i += blockDim.x) outp[i] = reinterpret_cast<const float4*>(Gacc)[i];
    }
}

// ---- sums over a row's non-zeros of x log(p + s_j q) for the trial steps s_j ----------------------
// mode 0: the objective at the point itself (one sum: x log p); mode 1: DN_TRIALS trial steps
__global__ void __launch_bounds__(256) dense_ls_kernel(const DenseParams P, int mode)
{
    __shared__ float red[8][DN_TRIALS];
    const int ch = blockIdx.x;
    const int h = P.chunk_h[ch];
    if (!P.sc[h].active) return;
    const int first = P.hcol0[h] + (ch - P.chunk_ptr[h]) * DN_LS_CHUNK;
    const int last = min(first + DN_LS_CHUNK, P.hcol0[h + 1]);
    const float* xr = P.xv + P.hbeg[h] - P.hcol0[h];          // compact index -> the side's values
    float s[DN_TRIALS], acc[DN_TRIALS];
#pragma unroll
    for (int j = 0; j < DN_TRIALS; j++) { s[j] = mode ? P.sc[h].steps[j] : 0.f; acc[j] = 0.f; }
    for (int t = first + threadIdx.x; t < last; t += blockDim.x) {
        const float x = xr[t], pt = P.p[t];
        if (mode) {
            const float qt = P.q[t];
#pragma unroll
            for (int j = 0; j < DN_TRIALS; j++) acc[j] += xlogp(x, fmaf(s[j], qt, pt));
        } else acc[0] += xlogp(x, pt);
    }
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int j = 0; j < DN_TRIALS; j++) {
        if (mode || j == 0) {
            float v = acc[j];
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if (lane == 0) red[w][j] = v;
        }
    }
    __syncthreads();
    if (threadIdx.x < DN_TRIALS && (mode || threadIdx.x == 0)) {
        float v = 0.f;
        for (int ww = 0; ww < 8; ww++) v += red[ww][threadIdx.x];
        P.lsp[(size_t)ch * DN_TRIALS + threadIdx.x] = v;
    }
}

// ---- f0 = <csum,x> + l2 |x|^2 - w sum x log p   (nonnegcg.c:191): one warp per heavy row -------------
__global__ void __launch_bounds__(128) dense_init_kernel(const DenseParams P)
{
    const int h = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (h >= P.H) return;
    DenseScal& S = P.sc[h];
    float ls = 0.f;
    for (int ch = P.chunk_ptr[h] + lane; ch < P.chunk_ptr[h + 1]; ch += 32) ls += P.lsp[(size_t)ch * DN_TRIALS];
    ls = warp_sum(ls);                                                                              // fixed order
    const float* x = P.M + (size_t)P.hrow[h] * P.ldf;
    float reg = 0.f, sq = 0.f;
    for (int i = lane; i < P.k; i += 32) { const float xi = x[i]; reg = fmaf(P.csum[i], xi, reg); sq = fmaf(xi, xi, sq); }
    reg = warp_sum(reg); sq = warp_sum(sq);
    const float regx = fmaf(P.hc.l2, sq, reg), fcur = regx - ls * P.hc.w;
    for (int i = lane; i < 64; i += 32) { P.gprev[h * 64 + i] = 0.f; P.dprev[h * 64 + i] = 0.f; }
    if (lane == 0) {
        S.fcur = fcur; S.regx = regx; S.gprev_sq = 0.f; S.step_applied = 0.f;
        S.it = 0; S.nfe = 1;
        S.active = (is_bad(fcur) || P.hc.maxupd == 0) ? 0 : 1;
    }
}
// every row is active while the first passes compute p and f0
__global__ void dense_reset_kernel(const DenseParams P)
{
    const int h = blockIdx.x * blockDim.x + threadIdx.x;
    if (h < P.H) { P.sc[h].active = 1; P.sc[h].step_applied = 0.f; }
}

// ---- direction and k-scalars (nonnegcg.c:231-288), one CTA per heavy row ------------------------------
// The per-CTA partial gradients are folded in a fixed order (warp w takes partials w, w+8, ...; lanes are
// components: coalesced), then warp 0 does the k-phase with lane l owning components l and l+32.
__global__ void __launch_bounds__(256) dense_k_kernel(const DenseParams P)
{
    __shared__ float part[8][64];
    const int h = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    DenseScal& S = P.sc[h];
    if (!S.active) return;
    const int k = P.k, ldf = P.ldf;
    {
        float s0 = 0.f, s1 = 0.f, t0 = 0.f, t1 = 0.f;
        int b = warp;
        for (; b + 8 < P.G; b += 16) {                       // two partials in flight per lane (fixed pairing)
            const float* gp = P.gpart + ((size_t)b * P.H + h) * ldf;
            const float* gq = P.gpart + ((size_t)(b + 8) * P.H + h) * ldf;
            if (lane < ldf) { s0 += gp[lane]; t0 += gq[lane]; }
            if (lane + 32 < ldf) { s1 += gp[lane + 32]; t1 += gq[lane + 32]; }
        }
        for (; b < P.G; b += 8) {
            const float* gp = P.gpart + ((size_t)b * P.H + h) * ldf;
            if (lane < ldf) s0 += gp[lane];
            if (lane + 32 < ldf) s1 += gp[lane + 32];
        }
        part[warp][lane] = s0 + t0; part[warp][lane + 32] = s1 + t1;
    }
    __syncthreads();
    if (warp != 0) return;
    const HalfSweepConsts<float>& hc = P.hc;
    const float* xrow = P.M + (size_t)P.hrow[h] * ldf;
    float xo[2], cs[2], go[2], gpo[2], dpo[2], dn[2];
#pragma unroll
    for (int i = 0; i < 2; i++) {
        const int comp = lane + 32 * i;
        const bool own = comp < k;
        xo[i] = own ? xrow[comp] : 0.f;
        cs[i] = own ? P.csum[comp] : 0.f;
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < 8; w++) s += part[w][comp];
        go[i] = own ? fmaf(hc.two_l2, xo[i], cs[i]) + s : 0.f;
        gpo[i] = P.gprev[h * 64 + comp]; dpo[i] = P.dprev[h * 64 + comp];
    }
    const int it = S.it;
    float theta = 0.f, beta = 0.f;
    if (it > 0) {
#pragma unroll
        for (int i = 0; i < 2; i++)
            if (!(xo[i] <= 0.f)) { theta = fmaf(go[i], dpo[i], theta); beta = fmaf(go[i], go[i] - gpo[i], beta); }
        theta = warp_sum(theta) / S.gprev_sq;
        beta = warp_sum(beta) / S.gprev_sq;
    }
    float gd = 0.f, dsq = 0.f, gg = 0.f, lin = 0.f, m = 1.f;
#pragma unroll
    for (int i = 0; i < 2; i++) {
        const float xi = xo[i], gi = go[i];
        float di = (xi <= 0.f && gi >= 0.f) ? 0.f : -gi;
        if (it > 0 && !(xi <= 0.f)) di += beta * dpo[i] - theta * (gi - gpo[i]);
        dn[i] = di;
        gd = fmaf(gi, di, gd); dsq = fmaf(di, di, dsq); gg = fmaf(gi, gi, gg);
        lin = fmaf(fmaf(hc.two_l2, xi, cs[i]), di, lin);
        if (di < 0.f) { const float r = -xi / di; m = (r < m) ? r : m; }
    }
    gd = warp_sum(gd); dsq = warp_sum(dsq); gg = warp_sum(gg); lin = warp_sum(lin);
    m = warp_min(m);
#pragma unroll
    for (int i = 0; i < 2; i++) {
        const int comp = lane + 32 * i;
        if (comp < ldf) P.dvec[(size_t)h * ldf + comp] = dn[i];
        P.gprev[h * 64 + comp] = go[i]; P.dprev[h * 64 + comp] = dn[i];
    }
    if (lane == 0) {
        S.gd = gd; S.dsq = dsq; S.gg = gg; S.lin = lin; S.smax = m;
        float sj = m;
#pragma unroll
        for (int j = 0; j < DN_TRIALS; j++) { S.steps[j] = sj; sj *= 0.25f; }
        if (fabsf(gd) <= 1e-2f) S.active = 0;                                                 // :264-269
    }
}

// ---- pick the first acceptable trial (nonnegcg.c:297-327), move the row; one warp per heavy row ------
__global__ void __launch_bounds__(128) dense_choose_kernel(const DenseParams P)
{
    const int h = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (h >= P.H) return;
    DenseScal& S = P.sc[h];
    if (!S.active) return;
    const HalfSweepConsts<float>& hc = P.hc;
    const float c_ls = 0.01f;
    const float fcur = S.fcur, regx = S.regx, dsq = S.dsq, lin = S.lin, l2dd = hc.l2 * S.dsq;
    auto freg = [&](float sj) { return fmaf(sj, fmaf(sj, l2dd, lin), regx); };
    // lane j: sum of the line-search pass for trial j, its objective.  The row's chunk partials are summed by
    // all 32 lanes (lane = chunk mod 32, then a shuffle tree): a fixed order, whatever the launch
    float tot = 0.f;
    {
        const int c0 = P.chunk_ptr[h], c1 = P.chunk_ptr[h + 1];
        for (int j = 0; j < DN_TRIALS; j++) {
            float v = 0.f;
            for (int ch = c0 + lane; ch < c1; ch += 32) v += P.lsp[(size_t)ch * DN_TRIALS + j];
            v = warp_sum(v);
            if (lane == j) tot = v;
        }
    }
    const float sj = lane < DN_TRIALS ? S.steps[lane] : 0.f;
    const float fj = freg(sj) - tot * hc.w;
    const bool okj = lane < DN_TRIALS && !is_bad(fj) && fj <= fcur - c_ls * sj * dsq;
    const unsigned okmask = __ballot_sync(0xffffffffu, okj);
    // sequential semantics: trials 0, 1, ... each failed one counts a function evaluation
    int nfe = S.nfe;
    const int first = okmask ? __ffs(okmask) - 1 : DN_MAX_LS;
    const int fails_allowed = DN_MAX_NFEVAL - nfe;          // the fails_allowed-th failure stops the solver
    bool accepted = false, stop = false;
    int last_eval;                                           // trial whose objective is the last one computed
    if (first < fails_allowed && first < DN_MAX_LS) { accepted = true; nfe += first; last_eval = first; }
    else if (fails_allowed <= DN_MAX_LS && fails_allowed <= first) { stop = true; nfe += fails_allowed; last_eval = fails_allowed - 1; }
    else { nfe += DN_MAX_LS; last_eval = DN_MAX_LS - 1; }
    if (stop) {                                              // :317-320: leave the row where it is
        if (lane == 0) { S.active = 0; S.nfe = nfe; }
        return;
    }
    const float step = __shfl_sync(0xffffffffu, sj, last_eval);
    const float fnew = __shfl_sync(0xffffffffu, fj, last_eval);
    if (accepted) {
        float* xrow = P.M + (size_t)P.hrow[h] * P.ldf;
        for (int i = lane; i < P.k; i += 32) {
            const float v = fmaf(step, P.dvec[(size_t)h * P.ldf + i], xrow[i]);
            const float xn = (v >= hc.clip_thr) ? v : 0.f;
            xrow[i] = xn;
            for (int q = 0; q < P.npeers; q++) P.peerM[q][(size_t)P.hrow[h] * P.ldf + i] = xn;
        }
    }
    if (lane == 0) {
        if (accepted) S.regx = freg(step);
        S.step_applied = accepted ? step : 0.f;
        S.fcur = fnew;                                         // :328 (Q4: even when no trial passed)
        S.gprev_sq = S.gg;                                     // :332
        S.nfe = nfe;
        S.it = S.it + 1;
        if (S.it >= (hc.maxupd <= 0 ? INT32_MAX : hc.maxupd)) S.active = 0;
    }
}

// ---- plan-time helpers ---------------------------------------------------------------------------
// key (tile, heavy row) and position of every non-zero of the heavy rows
__global__ void dense_keys_kernel(const int* __restrict__ ind, const int* __restrict__ hrow_of_cp, const long long* hbeg,
                                  const int* hcol0, int nnzH, int H, int U, unsigned* keys, int* pos)
{
    for (int cp = blockIdx.x * blockDim.x + threadIdx.x; cp < nnzH; cp += gridDim.x * blockDim.x) {
        const int h = hrow_of_cp[cp];
        const long long ps = hbeg[h] + (cp - hcol0[h]);
        keys[cp] = (unsigned)(ind[ps] / U) * (unsigned)H + (unsigned)h;
        pos[cp] = (int)ps;
    }
}
__global__ void dense_fill_slot_kernel(const int* hcol0, int H, int* hrow_of_cp)
{
    const int h = blockIdx.y;
    for (int cp = hcol0[h] + blockIdx.x * blockDim.x + threadIdx.x; cp < hcol0[h + 1]; cp += gridDim.x * blockDim.x)
        hrow_of_cp[cp] = h;
}
__global__ void dense_unpack_kernel(const unsigned* __restrict__ keys, const int* __restrict__ spos, const int* __restrict__ ind,
                                    const float* __restrict__ xv, const long long* hbeg, const int* hcol0, int nnzH, int H, int U,
                                    int ldf, uint2* ent, float* sx)
{
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < nnzH; t += gridDim.x * blockDim.x) {
        const unsigned h = keys[t] % (unsigned)H;
        const int pos = spos[t];
        ent[t] = make_uint2(((unsigned)(ind[pos] % U) * (unsigned)(ldf * 4) << 16) | h, (unsigned)(hcol0[h] + (int)((long long)pos - hbeg[h])));
        sx[t] = xv[pos];
    }
}
// seg_ptr[s] = first sorted position whose key >= s
__global__ void dense_segments_kernel(const unsigned* __restrict__ keys, int nnzH, int nseg, int* seg_ptr)
{
    for (int s = blockIdx.x * blockDim.x + threadIdx.x; s <= nseg; s += gridDim.x * blockDim.x) {
        int lo = 0, hi = nnzH;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (keys[mid] < (unsigned)s) lo = mid + 1; else hi = mid;
        }
        seg_ptr[s] = lo;
    }
}

}  // namespace pmf
