// poismf_b200 — tensor-core candidate scorer for batched topN (sm_100a: tcgen05 + TMEM).
//
// topN's scoring step, scores[u, j] = <A[u], B[j]>, is the one dense contraction of the path
// (/root/reference/src/topN.c:215-224 does it as one GEMV per user).  Batched over users it is a
// GEMM; `score_pipe_tf32_kernel` runs it on the 5th-generation tensor cores in TF32: warp-specialised
// persistent CTAs, operands by TMA (128-byte-swizzled 2-D boxes), a ring of shared-memory stages, accumulators
// double-buffered in TMEM, eight epilogue warps — described in front of the kernel.  With too few items for
// the fused select below, `score_tiles_tf32_kernel` writes the TF32 score matrix for a segmented sort instead.
//
// TF32 scores are only used to pick CANDIDATES: the caller keeps the best 2N+ per user, re-scores
// them exactly in FP32 (same left-to-right sums as the reference) and proves from the TF32 error
// bound that no other item can enter the top N; users for which the proof fails are redone by the
// exact scorer.  Rankings are therefore those of the exact path.
//
// The select is fused into the scorer's epilogue so that the U x n score matrix never exists
// (SURVEY.md 8d).  Two passes over the tiles, the GEMM being far cheaper than any sort of n scores:
//   pass 1 (MODE_GROUPMAX)  per user, the maximum of every group of 16 consecutive items — of every S-th item
//           tile only (S = 4, 2 or 1)
//           -> tau[u] = the M-th largest of these group maxima: a lower bound of the M-th largest over all
//              items, so at least M items score >= tau[u], and about S M of them do;
//   pass 2 (MODE_EMIT)      all tiles; items with score >= tau[u] are appended to the user's candidate list,
// then the (<= 4096) candidates are ordered by (score desc, id asc) and the best M go to the exact
// re-scoring.  Excluded items are masked in the epilogue from a per-user bitmap.
#pragma once
#include <cuda.h>
#include "common.cuh"

namespace pmf {
namespace tc {

constexpr int TM = 128;   // users per tile  (UMMA M)
constexpr int TN = 128;   // items per tile  (UMMA N)
constexpr int GROUP = 16;        // items per group maximum
constexpr int CAND_CAP = 4096;   // candidates per user that are ordered (>= GROUP * 256)
constexpr int CAND_SLACK = 4;    // the per-CTA regions of a user hold CAND_SLACK x CAND_CAP slots together
constexpr int CAND_TOP = 256;    // candidates handed to the exact re-scoring (>= M)
enum { MODE_GROUPMAX = 1, MODE_EMIT = 2 };

// order-preserving key of a non-negative score; masked entries (negative) sort below everything
PMF_DEVINL uint32_t score_key(float s) { return s < 0.f ? 0u : __float_as_uint(s) + 1u; }
PMF_DEVINL float key_score(uint32_t key) { return key == 0u ? -RealTraits<float>::huge() : __uint_as_float(key - 1u); }

PMF_DEVINL uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// Shared-memory matrix descriptor (K-major, no swizzle), sm_100 format: start address >> 4 in bits
// [0,14), leading byte offset >> 4 in [16,30), stride byte offset >> 4 in [32,46), version 1 in [46,48).
PMF_DEVINL uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes)
{
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFFu);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
    d |= (uint64_t)1 << 46;
    return d;
}

// Instruction descriptor for kind::tf32: D = F32 (bits [4,6) = 1), A = B = TF32 (bits [7,10), [10,13) = 2),
// both K-major (bits 15, 16 = 0), N >> 3 in [17,23), M >> 4 in [24,29).
constexpr uint32_t make_idesc_tf32(int M, int N)
{
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

PMF_DEVINL void mbar_init(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
PMF_DEVINL void mbar_wait(uint64_t* bar, uint32_t phase)
{
    asm volatile(
        "{\n\t"
        ".reg .pred P1;\n\t"
        "LAB_WAIT:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1, %2;\n\t"
        "@P1 bra DONE;\n\t"
        "bra LAB_WAIT;\n\t"
        "DONE:\n\t"
        "}" ::"r"(smem_u32(bar)), "r"(phase), "r"(0x989680u)
        : "memory");
}
PMF_DEVINL void umma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
PMF_DEVINL void umma_commit(uint64_t* bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
PMF_DEVINL void tmem_ld32(uint32_t taddr, uint32_t (&r)[32])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// Stage `rows_valid` rows (row stride ldf floats, kpad <= padded k) of a factor matrix as one UMMA
// operand tile.  Eight consecutive threads write eight consecutive tile rows of one K-chunk: a
// conflict-free 128-byte shared-memory line per quarter-warp.
PMF_DEVINL void stage_operand(float4* s, const float* __restrict__ G, size_t row0, size_t rows_total, int ldf, int kpad,
                              int tile_rows)
{
    const int nkc = kpad / 4, rblocks = tile_rows / 8;
    for (int q = threadIdx.x >> 3; q < rblocks * nkc; q += blockDim.x >> 3) {
        const int rb = q % rblocks, kc = q / rblocks;
        const int row = rb * 8 + (threadIdx.x & 7);
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        const size_t gr = row0 + row;
        if (gr < rows_total && kc * 4 < ldf) v = __ldg(reinterpret_cast<const float4*>(G + gr * ldf + kc * 4));
        s[kc * tile_rows + row] = v;
    }
}

// What the epilogue of a tile does with its scores
struct TileOut {
    const uint32_t* excl_bits; size_t excl_words;   // bitmap of excluded items, excl_words 32-bit words per user (or null)
    float* gmax; size_t ngroups;             // MODE_GROUPMAX: gmax[u, j / GROUP]
    const float* tau;                        // MODE_EMIT: per-user threshold ...
    float* cand_sc; int* cand_id; int* cand_cnt;   // ... and candidate lists (CAND_CAP slots per user)
    // the scorer splits a user's slots into `cand_regions` regions of `cand_cap` slots, one per CTA
    // along the items (each written by exactly one thread: no atomics); cand_cnt is [user][region]
    int cand_regions, cand_cap;
};

// The TF32 score matrix of a chunk of users, for the segmented-sort select (items too few for the fused one):
// scores[u, j] and ids[u, j] = j, row stride n.  One CTA per 128 users x 128 items tile, both operand tiles
// staged K-major in shared memory by generic loads in the canonical no-swizzle UMMA layout (8-row x 16-byte
// core matrices; for tile row r and 16-byte K-chunk c the chunk sits at (c * 128 + r) * 16 bytes, i.e.
// stride-byte-offset 128 B between 8-row groups, leading-byte-offset 2048 B between K-chunks); one thread
// issues k/8 `tcgen05.mma.cta_group::1.kind::tf32` (M = N = 128, K = 8) into 128 TMEM columns and commits onto
// an mbarrier; the four warps read their 32 TMEM lanes back with `tcgen05.ld.32x32b.x32`.
// grid = (ceil(n/TN), ceil(U/TM)), 128 threads, kpad * 1024 bytes of dynamic shared memory.
__global__ void __launch_bounds__(128) score_tiles_tf32_kernel(const float* __restrict__ Asel, int U,
                                                               const float* __restrict__ B, size_t n, int ldf,
                                                               int kpad, float* __restrict__ scores,
                                                               int* __restrict__ ids)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float4* sA = reinterpret_cast<float4*>(smem_raw);
    float4* sB = sA + (size_t)(kpad / 4) * TM;
    __shared__ __align__(8) uint64_t mbar;
    __shared__ uint32_t tmem_base_s;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const size_t j0 = (size_t)blockIdx.x * TN;
    const int u0 = blockIdx.y * TM;

    if (warp == 0) {   // 128 TMEM columns (fp32 accumulators of the 128 x 128 tile)
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)),
                     "r"((uint32_t)TN)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 0) mbar_init(&mbar, 1);
    stage_operand(sA, Asel, (size_t)u0, (size_t)U, ldf, kpad, TM);
    stage_operand(sB, B, j0, n, ldf, kpad, TN);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy stores -> visible to the tensor core
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = tmem_base_s;

    if (tid == 0) {
        constexpr uint32_t idesc = make_idesc_tf32(TM, TN);
        const uint32_t a0 = smem_u32(sA), b0 = smem_u32(sB);
        for (int kb = 0; kb < kpad / 8; kb++) {   // K = 8 (two 16-byte chunks) per instruction
            const uint64_t da = make_smem_desc(a0 + (uint32_t)kb * 2u * TM * 16u, TM * 16u, 128u);
            const uint64_t db = make_smem_desc(b0 + (uint32_t)kb * 2u * TN * 16u, TN * 16u, 128u);
            umma_tf32(tmem, da, db, idesc, kb > 0 ? 1u : 0u);
        }
        umma_commit(&mbar);
    }
    mbar_wait(&mbar, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

    // epilogue: warp w owns TMEM lanes 32w .. 32w+31 (= tile rows), 32 columns at a time
    const int u = u0 + warp * 32 + lane;
    for (int c = 0; c < TN / 32; c++) {
        uint32_t r[32];
        tmem_ld32(tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)(c * 32), r);
        if (u >= U) continue;
        const size_t jc = j0 + c * 32;
        float* srow = scores + (size_t)u * n + jc;
        int* irow = ids + (size_t)u * n + jc;
#pragma unroll
        for (int i = 0; i < 32; i++)
            if (jc + i < n) { srow[i] = __uint_as_float(r[i]); irow[i] = (int)(jc + i); }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"((uint32_t)TN) : "memory");
}

// ---- the scorer: persistent CTAs, operands by TMA, accumulators double-buffered in TMEM ------
// One CTA keeps TWO user tiles (256 users: the A operands, loaded once) and walks a contiguous range of item
// tiles; every item tile brought on chip is used by both (half the L2 -> SM traffic of one tile per CTA).
// Operands arrive by TMA (`cp.async.bulk.tensor.2d`, SASS UTMALDG): the factor matrices are described to the
// TMA unit as 2-D tensors (k floats x rows) and fetched in boxes of 32 floats x 128 rows with the 128-byte
// swizzle, i.e. whole 128-byte lines of 128 factor rows per request, landing in the K-major SWIZZLE_128B
// layout the tensor core reads (descriptor: 8-row groups 1024 bytes apart, start address advanced by 32 bytes
// per K = 8 step inside the swizzle atom); rows beyond the matrix and floats beyond k are zero-filled by the
// TMA unit.  Item tiles go through a ring of PIPE_STAGES shared-memory stages guarded by mbarriers (expect_tx /
// complete_tx); the accumulators of consecutive item tiles alternate between two TMEM buffers of 2 x 128
// columns, so the epilogue of tile i-1 (TMEM -> registers -> group maxima / candidates) runs while the tensor
// core works on tile i:
// Warp roles (320 threads), coupled only through mbarriers:
//     warp 9 (one lane) : for each tile: wait stage_free[s] -> expect_tx + TMA boxes -> full[s]
//     warp 8 (one lane) : wait full[s], wait tmem_free[b] -> 2 x (k/8) tcgen05.mma into buffer b
//                         -> tcgen05.commit to stage_free[s] and to mma_done[b]
//     warps 0..7        : wait mma_done[b] -> TMEM -> registers (arrive on tmem_free[b] as soon as the last load
//                         has landed) -> group maxima / candidates
constexpr int PIPE_STAGES = 3;       // at most (5 stages measured slower: 9.8 vs 8.1 ms per pass at c5s); fewer when k is large
constexpr int PIPE_UT = 2;           // user tiles per CTA
constexpr int PIPE_BOXK = 32;        // floats per TMA box along k (128 bytes: the swizzle span)
constexpr int PIPE_THREADS = 320;    // 8 epilogue warps, the MMA warp, the TMA warp

// TMEM -> registers without the wait, and the wait carrying the registers as operands (so that no use of them can
// be scheduled above it): the load of the next 32 columns is in flight while the current ones are reduced
PMF_DEVINL void tmem_ld32_async(uint32_t taddr, uint32_t (&r)[32])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}
PMF_DEVINL void tmem_ld_wait(uint32_t (&r)[32])
{
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                   "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]),
                   "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]),
                   "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
                 :: "memory");
}

PMF_DEVINL void pipe_wait(uint64_t* bar, uint32_t phase)
{
    unsigned ok, spins = 0;
    do {
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                     : "=r"(ok) : "r"(smem_u32(bar)), "r"(phase) : "memory");
        if (!ok && ++spins > (1u << 26)) __trap();        // a lost copy must not hang the device
    } while (!ok);
}
PMF_DEVINL void pipe_expect(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
PMF_DEVINL void tma_box(void* smem_dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
                 : "memory");
}
// K-major SWIZZLE_128B operand: rows 128 bytes apart, 8-row groups 1024 bytes apart (SBO), LBO unused (1),
// descriptor version 1, layout type 2 (sm_100 encoding)
PMF_DEVINL uint64_t make_smem_desc_sw128(uint32_t saddr)
{
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFFu);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024u >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}

// grid = (item-tile chunks, pairs of user tiles), PIPE_THREADS threads, dynamic shared memory
// pipe_smem_bytes(kpad) = (PIPE_UT + stages) * nbox * 16 KB + 1 KB with nbox = ceil(kpad / 32).
// Epilogue: warp w reads TMEM lanes 32 (w % 4) .. +31 (its quarter; = tile rows = users) of user tile w / 4.
template <int MODE>
__global__ void __launch_bounds__(PIPE_THREADS) score_pipe_tf32_kernel(const __grid_constant__ CUtensorMap mapA,
                                                              const __grid_constant__ CUtensorMap mapB, int U, size_t n,
                                                              int kpad, int tile_stride, int nstages, TileOut out)
{
    extern __shared__ __align__(1024) unsigned char smem_dyn[];
    // the 128-byte swizzle works on 1024-byte atoms: align the operand area whatever the static variables take
    unsigned char* smem_raw = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
    __shared__ __align__(8) uint64_t full[PIPE_STAGES], stage_free[PIPE_STAGES], mma_done[2], tmem_free[2], a_full;
    __shared__ uint32_t tmem_base_s;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int nbox = (kpad + PIPE_BOXK - 1) / PIPE_BOXK;
    const uint32_t box_bytes = (uint32_t)TM * PIPE_BOXK * 4u;          // 16 KB
    const uint32_t tile_bytes = (uint32_t)nbox * box_bytes;
    unsigned char* sA = smem_raw;
    unsigned char* sB = smem_raw + (size_t)PIPE_UT * tile_bytes;
    const int u00 = blockIdx.y * (PIPE_UT * TM);
    // the CTA's i-th item tile is tile (blockIdx.x + i gridDim.x) * tile_stride: the CTAs along x interleave over
    // the items (popular items at low ids spread evenly over them), and with tile_stride > 1 only every
    // tile_stride-th tile is visited (the threshold pass works on a sample of the items)
    const size_t ntiles = (n + TN - 1) / TN;
    const size_t nvisit = (ntiles + tile_stride - 1) / tile_stride;
    const int nt = nvisit > blockIdx.x ? (int)((nvisit - blockIdx.x + gridDim.x - 1) / gridDim.x) : 0;
    auto visit = [&](int i) { return (size_t)blockIdx.x + (size_t)i * gridDim.x; };      // index among the visited tiles

    if (warp == 0) {   // two buffers of PIPE_UT accumulators of 128 columns: all 512 columns
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)),
                     "r"((uint32_t)(2 * PIPE_UT * TN))
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 0) {
        mbar_init(&a_full, 1);
        for (int s = 0; s < PIPE_STAGES; s++) { mbar_init(&full[s], 1); mbar_init(&stage_free[s], 1); }
        mbar_init(&mma_done[0], 1); mbar_init(&mma_done[1], 1);
        mbar_init(&tmem_free[0], 8); mbar_init(&tmem_free[1], 8);      // one arrival per epilogue warp
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = tmem_base_s;

    constexpr uint32_t idesc = make_idesc_tf32(TM, TN);
    if (warp == 9) {                 // ---- TMA producer ----
        if (lane == 0 && nt > 0) {
            pipe_expect(&a_full, PIPE_UT * tile_bytes);
            for (int ut = 0; ut < PIPE_UT; ut++)
                for (int bx = 0; bx < nbox; bx++)
                    tma_box(sA + (size_t)ut * tile_bytes + (size_t)bx * box_bytes, &mapA, bx * PIPE_BOXK, u00 + ut * TM, &a_full);
            for (int i = 0; i < nt; i++) {
                const int s = i % nstages;
                if (i >= nstages) pipe_wait(&stage_free[s], (uint32_t)((i / nstages - 1) & 1));
                pipe_expect(&full[s], tile_bytes);
                for (int bx = 0; bx < nbox; bx++)
                    tma_box(sB + (size_t)s * tile_bytes + (size_t)bx * box_bytes, &mapB, bx * PIPE_BOXK, (int)(visit(i) * tile_stride * TN), &full[s]);
            }
        }
    } else if (warp == 8) {          // ---- MMA issuer ----
        if (lane == 0 && nt > 0) {
            const uint32_t a0 = smem_u32(sA), b00 = smem_u32(sB);
            pipe_wait(&a_full, 0);
            for (int i = 0; i < nt; i++) {
                const int s = i % nstages, b = i & 1;
                pipe_wait(&full[s], (uint32_t)((i / nstages) & 1));
                if (i >= 2) pipe_wait(&tmem_free[b], (uint32_t)(((i >> 1) - 1) & 1));
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint64_t db0 = make_smem_desc_sw128(b00 + (uint32_t)s * tile_bytes);
                for (int ut = 0; ut < PIPE_UT; ut++) {
                    const uint64_t da0 = make_smem_desc_sw128(a0 + (uint32_t)ut * tile_bytes);
                    const uint32_t acc = tmem + (uint32_t)((b * PIPE_UT + ut) * TN);
                    for (int kb = 0; kb < kpad / 8; kb++) {   // K = 8 (32 bytes inside the swizzle atom) per instruction
                        const uint64_t koff = (uint64_t)(((uint32_t)(kb >> 2) * box_bytes + (uint32_t)(kb & 3) * 32u) >> 4);
                        umma_tf32(acc, da0 + koff, db0 + koff, idesc, kb > 0 ? 1u : 0u);
                    }
                }
                umma_commit(&stage_free[s]);
                umma_commit(&mma_done[b]);
            }
        }
    } else {                         // ---- epilogue warps ----
    const int quarter = warp & 3, ut_mine = warp >> 2;       // TMEM lane quarter, user tile
    const int u = u00 + ut_mine * TM + quarter * 32 + lane;
    const float NEG = -RealTraits<float>::huge();
    const float tau = (MODE == MODE_EMIT && u < U) ? out.tau[u] : 0.f;
    uint4 ex_next = make_uint4(0u, 0u, 0u, 0u);
    if (out.excl_bits && u < U && nt > 0)
        ex_next = __ldg(reinterpret_cast<const uint4*>(out.excl_bits + (size_t)u * out.excl_words + ((visit(0) * tile_stride * TN) >> 5)));
    int n_mine = 0;                                          // MODE_EMIT: candidates this thread has found
    const size_t region = ((size_t)(u < U ? u : 0) * out.cand_regions + blockIdx.x) * out.cand_cap;
        for (int j = 0; j < nt; j++) {
            pipe_wait(&mma_done[j & 1], (uint32_t)((j >> 1) & 1));
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const size_t j0 = visit(j) * tile_stride * TN;
            const uint4 ex = ex_next;                        // this user's exclusion bits of the tile's 128 items
            if (out.excl_bits && u < U && j + 1 < nt)        // (the next tile's are fetched a tile ahead)
                ex_next = __ldg(reinterpret_cast<const uint4*>(out.excl_bits + (size_t)u * out.excl_words +
                                                               ((visit(j + 1) * tile_stride * TN) >> 5)));
            float gm[8];                                     // MODE_GROUPMAX: the 8 group maxima of the 128 columns
            const uint32_t tcol = tmem + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(((j & 1) * PIPE_UT + ut_mine) * TN);
            uint32_t ra[32], rb[32];
            tmem_ld32_async(tcol, ra);
#pragma unroll
            for (int c = 0; c < 4; c++) {
                uint32_t (&r)[32] = (c & 1) ? rb : ra;
                tmem_ld_wait(r);
                if (c < 3) tmem_ld32_async(tcol + (uint32_t)((c + 1) * 32), (c & 1) ? ra : rb);
                else {      // the tile is in registers: its TMEM buffer may take tile j + 2
                    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                    __syncwarp();
                    if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&tmem_free[j & 1])) : "memory");
                }
                const size_t jc = j0 + c * 32;
                uint32_t valid = ~(c == 0 ? ex.x : (c == 1 ? ex.y : (c == 2 ? ex.z : ex.w)));
                if (jc + 32 > n) valid &= (jc >= n) ? 0u : ((1u << (unsigned)(n - jc)) - 1u);
                if (MODE == MODE_GROUPMAX) {
#pragma unroll
                    for (int g = 0; g < 32 / GROUP; g++) {
                        float m = NEG;
                        if (((valid >> (g * GROUP)) & 0xffffu) == 0xffffu) {      // nothing masked: plain maximum
#pragma unroll
                            for (int q = 0; q < GROUP; q++) m = fmaxf(m, __uint_as_float(r[g * GROUP + q]));
                        } else {
#pragma unroll
                            for (int q = 0; q < GROUP; q++)
                                if ((valid >> (g * GROUP + q)) & 1u) m = fmaxf(m, __uint_as_float(r[g * GROUP + q]));
                        }
                        gm[c * 2 + g] = m;
                    }
                } else if (u < U) {
                    float mx = NEG;                         // most 32-column blocks hold no candidate at all
#pragma unroll
                    for (int q = 0; q < 32; q++) mx = fmaxf(mx, __uint_as_float(r[q]));
                    if (mx >= tau) {
                        // rare path, kept compact (an unrolled predicated emission is ~25 KB of code and stalls the
                        // instruction fetch): a bit per candidate column, then a loop over the set bits that picks
                        // the value out of the registers with a 5-level select tree
                        uint32_t hit = 0;
#pragma unroll
                        for (int q = 0; q < 32; q++) hit |= (__uint_as_float(r[q]) >= tau ? 1u : 0u) << q;
                        hit &= valid;
                        while (hit) {
                            const int q = __ffs((int)hit) - 1;
                            hit &= hit - 1;
                            uint32_t t[16];
#pragma unroll
                            for (int e = 0; e < 16; e++) t[e] = (q & 1) ? r[2 * e + 1] : r[2 * e];
#pragma unroll
                            for (int e = 0; e < 8; e++) t[e] = (q & 2) ? t[2 * e + 1] : t[2 * e];
#pragma unroll
                            for (int e = 0; e < 4; e++) t[e] = (q & 4) ? t[2 * e + 1] : t[2 * e];
#pragma unroll
                            for (int e = 0; e < 2; e++) t[e] = (q & 8) ? t[2 * e + 1] : t[2 * e];
                            const uint32_t vb = (q & 16) ? t[1] : t[0];
                            if (n_mine < out.cand_cap) {       // this thread owns the region: plain stores
                                out.cand_sc[region + n_mine] = __uint_as_float(vb);
                                out.cand_id[region + n_mine] = (int)(jc + q);
                            }
                            n_mine++;
                        }
                    }
                }
            }
            if (MODE == MODE_GROUPMAX && u < U) {           // 8 consecutive group maxima: two 16-byte stores when they fit
                const size_t gi = visit(j) * (TN / GROUP);          // groups are numbered along the VISITED tiles
                float* dst = out.gmax + (size_t)u * out.ngroups + gi;
                if (gi + 8 <= out.ngroups && ((reinterpret_cast<uintptr_t>(dst) & 15) == 0)) {
                    reinterpret_cast<float4*>(dst)[0] = make_float4(gm[0], gm[1], gm[2], gm[3]);
                    reinterpret_cast<float4*>(dst)[1] = make_float4(gm[4], gm[5], gm[6], gm[7]);
                } else
                    for (int g = 0; g < 8; g++) if (gi + g < out.ngroups) dst[g] = gm[g];
            }
        }
        if (MODE == MODE_EMIT && u < U) out.cand_cnt[(size_t)u * out.cand_regions + blockIdx.x] = n_mine;
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"((uint32_t)(2 * PIPE_UT * TN)) : "memory");
}

// operand stages that fit next to the two user tiles (227 KB per CTA; k <= 64: 3, k <= 96: 2, k <= 128: 1) and
// the dynamic shared memory of the launch (+1 KB for the alignment)
inline int pipe_stages(int kpad)
{
    const size_t tile = (size_t)((kpad + PIPE_BOXK - 1) / PIPE_BOXK) * TM * PIPE_BOXK * 4;
    const size_t room = (size_t)226 * 1024 - 1024 - PIPE_UT * tile;
    return (int)std::max<size_t>(1, std::min<size_t>(PIPE_STAGES, room / tile));
}
inline size_t pipe_smem_bytes(int kpad)
{
    const size_t tile = (size_t)((kpad + PIPE_BOXK - 1) / PIPE_BOXK) * TM * PIPE_BOXK * 4;
    return (size_t)(PIPE_UT + pipe_stages(kpad)) * tile + 1024;
}

// a factor matrix [rows x ldf floats] as a 2-D tensor for the TMA unit, fetched in boxes of 32 floats x 128 rows
// with the 128-byte swizzle
inline int make_operand_map(CUtensorMap* map, const float* base, size_t rows, int ldf)
{
    typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                 const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                 CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static EncodeFn fn = nullptr;
    if (!fn) {
        void* f = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess || !f) return 1;
        fn = (EncodeFn)f;
    }
    const cuuint64_t gdim[2] = {(cuuint64_t)ldf, (cuuint64_t)rows};
    const cuuint64_t gstride[1] = {(cuuint64_t)ldf * sizeof(float)};
    const cuuint32_t box[2] = {(cuuint32_t)PIPE_BOXK, (cuuint32_t)TM};
    const cuuint32_t estr[2] = {1u, 1u};
    return fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
              CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS ? 0 : 1;
}

// Exact re-scoring + final ordering of the per-user candidates.  One CTA (128 threads) per user.
//   cand_ids / cand_approx : the first M entries of the user's approx-sorted row (stride n)
// The M candidates are re-scored with the reference's left-to-right non-contracted sum, ordered by
// (score desc, id asc) with a bitonic network in shared memory, and the first n_top written out.
// flag[u] = 1 when the TF32 error bound cannot exclude an item outside the candidates.
__global__ void __launch_bounds__(128) rescore_select_kernel(const float* __restrict__ Asel, const float* __restrict__ B,
                                                             int k, int ldf, const int* __restrict__ cand_ids,
                                                             const float* __restrict__ cand_approx, size_t n, int M,
                                                             int n_avail_is_M, int n_top, float rel_bound,
                                                             long long* __restrict__ out_ids,
                                                             float* __restrict__ out_scores, int* __restrict__ flag)
{
    __shared__ float ss[256];
    __shared__ int si[256];
    __shared__ float a[256];
    const int u = blockIdx.x, tid = threadIdx.x;
    for (int c = tid; c < k; c += blockDim.x) a[c] = Asel[(size_t)u * ldf + c];
    __syncthreads();
    const float NEG = -RealTraits<float>::huge();
    for (int c = tid; c < 256; c += blockDim.x) {
        float s = NEG; int id = 0x7fffffff;
        if (c < M) {
            const float ap = cand_approx[(size_t)u * n + c];
            if (ap > NEG) {
                id = cand_ids[(size_t)u * n + c];
                const float* b = B + (size_t)id * ldf;
                float acc = 0;
                for (int i = 0; i < k; i++) acc = add_rn(acc, mul_rn(a[i], b[i]));
                s = acc;
            }
        }
        ss[c] = s; si[c] = id;
    }
    __syncthreads();
    for (int len = 2; len <= 256; len <<= 1)
        for (int j = len >> 1; j > 0; j >>= 1) {
            for (int t = tid; t < 128; t += blockDim.x) {
                const int lo = 2 * t - (t & (j - 1)), hi = lo + j;
                const bool desc_block = ((lo & len) == 0);
                const float s0 = ss[lo], s1 = ss[hi];
                const int i0 = si[lo], i1 = si[hi];
                const bool before = (s0 > s1) || (s0 == s1 && i0 < i1);   // lo already precedes hi
                if (before != desc_block) { ss[lo] = s1; ss[hi] = s0; si[lo] = i1; si[hi] = i0; }
            }
            __syncthreads();
        }
    for (int c = tid; c < n_top; c += blockDim.x) {
        out_ids[(size_t)u * n_top + c] = si[c];
        if (out_scores) out_scores[(size_t)u * n_top + c] = ss[c];
    }
    if (tid == 0) {
        int bad = 0;
        if (!n_avail_is_M) {
            // every item outside the candidates has TF32 score <= a_min, hence exact score <= a_min * (1 + rel_bound)
            const float a_min = cand_approx[(size_t)u * n + (M - 1)];
            const float e_n = ss[n_top - 1];
            if (!(a_min == NEG) && !(e_n > a_min * (1.0f + rel_bound))) bad = 1;
        }
        flag[u] = bad;
    }
}

// bits[u, j] = 1 for every item j in user (user0 + u)'s exclusion list.  grid = (x, users of the chunk)
template <class IX>
__global__ void exclusion_bitmap_kernel(uint32_t* __restrict__ bits, size_t words, const IX* __restrict__ excl_ptr,
                                        const IX* __restrict__ excl_ix, size_t user0, size_t n)
{
    const size_t u = blockIdx.y;
    const size_t beg = (size_t)excl_ptr[user0 + u], end = (size_t)excl_ptr[user0 + u + 1];
    for (size_t t = beg + blockIdx.x * (size_t)blockDim.x + threadIdx.x; t < end; t += (size_t)gridDim.x * blockDim.x) {
        const size_t j = (size_t)excl_ix[t];
        if (j < n) atomicOr(bits + u * words + (j >> 5), 1u << (j & 31));
    }
}

// tau[u] = the M-th largest of the user's group maxima, in two reads of the row (it is HBM traffic that this
// kernel costs: 250 KB per user at 1M items).  Read 1: a 4096-bin histogram of the top 12 key bits (exponent + 4
// mantissa bits); a block-wide suffix sum finds the bin that holds the M-th largest.  Read 2: that bin's keys
// (a few hundred) are collected in shared memory and a radix select on their low 19 bits finishes there.
// A bin with more keys than the list holds falls back to the bin's lower edge — a smaller threshold, i.e. more
// candidates, never fewer.  One CTA of 256 threads per user.
constexpr int SEL_BINS = 4096, SEL_LIST = 4096, SEL_SHIFT = 19;
__global__ void __launch_bounds__(256) select_threshold_kernel(const float* __restrict__ gmax, size_t ngroups, int M,
                                                               float* __restrict__ tau)
{
    __shared__ unsigned int hist[SEL_BINS];
    __shared__ unsigned int part[256];
    __shared__ uint32_t list[SEL_LIST];
    __shared__ uint32_t s_prefix;
    __shared__ int s_want, s_cnt;
    const float* g = gmax + (size_t)blockIdx.x * ngroups;
    const int tid = threadIdx.x;
    for (int i = tid; i < SEL_BINS; i += 256) hist[i] = 0u;
    if (tid == 0) s_cnt = 0;
    __syncthreads();
    for (size_t i = tid; i < ngroups; i += 256) atomicAdd(&hist[score_key(g[i]) >> SEL_SHIFT], 1u);
    __syncthreads();
    unsigned int mine = 0;                                  // thread t owns bins [16 t, 16 t + 16)
    for (int b = 0; b < 16; b++) mine += hist[16 * tid + b];
    part[tid] = mine;
    __syncthreads();
    for (int off = 1; off < 256; off <<= 1) {               // part[t] = keys in the bins of threads >= t
        const unsigned int v = tid + off < 256 ? part[tid + off] : 0u;
        __syncthreads();
        part[tid] += v;
        __syncthreads();
    }
    const unsigned int above = part[tid] - mine;
    if (above < (unsigned)M && (unsigned)M <= above + mine) {      // the M-th largest lies in my bins
        int want = M - (int)above, b = 15;
        for (; b > 0; b--) {
            const int c = (int)hist[16 * tid + b];
            if (c >= want) break;
            want -= c;
        }
        s_prefix = (uint32_t)(16 * tid + b) << SEL_SHIFT;
        s_want = want;
    }
    __syncthreads();
    uint32_t prefix = s_prefix;
    const unsigned int in_bin = hist[prefix >> SEL_SHIFT];
    if (in_bin > (unsigned)SEL_LIST) {
        if (tid == 0) tau[blockIdx.x] = key_score(prefix);
        return;
    }
    for (size_t i = tid; i < ngroups; i += 256) {
        const uint32_t key = score_key(g[i]);
        if ((key >> SEL_SHIFT) == (prefix >> SEL_SHIFT)) list[atomicAdd(&s_cnt, 1)] = key;
    }
    __syncthreads();
    const int cnt = s_cnt;
    uint32_t mask = ~0u << SEL_SHIFT;
    for (int round = 0; round < 3; round++) {               // low 19 bits: digits of 8, 8 and 3 bits
        const int shift = round == 0 ? 11 : (round == 1 ? 3 : 0);
        const uint32_t dmask = round == 2 ? 7u : 255u;
        hist[tid] = 0u;
        __syncthreads();
        for (int i = tid; i < cnt; i += 256) {
            const uint32_t key = list[i];
            if ((key & mask) == prefix) atomicAdd(&hist[(key >> shift) & dmask], 1u);
        }
        __syncthreads();
        if (tid == 0) {     // walk the digits from the top until `want` keys have been passed
            int want = s_want, d = (int)dmask;
            for (; d > 0; d--) {
                const int c = (int)hist[d];
                if (c >= want) break;
                want -= c;
            }
            s_prefix = prefix | ((uint32_t)d << shift);
            s_want = want;
        }
        __syncthreads();
        prefix = s_prefix;
        mask |= dmask << shift;
        __syncthreads();
    }
    if (tid == 0) tau[blockIdx.x] = key_score(prefix);
}

// Order one user's candidates by (score desc, id asc) and keep the best CAND_TOP (padded with -huge).
// overflow[u] = 1 when more than CAND_CAP items reached the threshold (ties at tau): redo exactly.
__global__ void __launch_bounds__(512) sort_candidates_kernel(const float* __restrict__ cand_sc,
                                                              const int* __restrict__ cand_id,
                                                              const int* __restrict__ cand_cnt, int regions, int cap,
                                                              float* __restrict__ top_sc, int* __restrict__ top_id,
                                                              int* __restrict__ overflow)
{
    __shared__ float ss[CAND_CAP];
    __shared__ int si[CAND_CAP];
    __shared__ int s_off[65];                        // where each region's candidates go (regions <= 64)
    const int u = blockIdx.x, tid = threadIdx.x;
    const float NEG = -RealTraits<float>::huge();
    if (tid == 0) {
        int off = 0, ovf = 0;
        for (int r = 0; r < regions; r++) {
            const int c = cand_cnt[(size_t)u * regions + r];
            s_off[r] = off;
            off += c < cap ? c : cap;
            ovf |= c > cap;
            if (off > CAND_CAP) { off = CAND_CAP; ovf = 1; }      // more than can be ordered here: exact fallback
        }
        s_off[regions] = off;
        overflow[u] = ovf;
    }
    __syncthreads();
    const int m = s_off[regions];                    // <= CAND_CAP
    int len_pad = CAND_TOP;                          // sort only as much as is filled (power of two)
    while (len_pad < m) len_pad <<= 1;
    for (int c = m + tid; c < len_pad; c += blockDim.x) { ss[c] = NEG; si[c] = 0x7fffffff; }
    for (int r = 0; r < regions; r++) {
        const int o = s_off[r], c = s_off[r + 1] - o;
        const size_t base = ((size_t)u * regions + r) * cap;
        for (int t = tid; t < c; t += blockDim.x) { ss[o + t] = cand_sc[base + t]; si[o + t] = cand_id[base + t]; }
    }
    __syncthreads();
    for (int len = 2; len <= len_pad; len <<= 1)
        for (int j = len >> 1; j > 0; j >>= 1) {
            for (int t = tid; t < len_pad / 2; t += blockDim.x) {
                const int lo = 2 * t - (t & (j - 1)), hi = lo + j;
                const bool desc_block = ((lo & len) == 0);
                const float s0 = ss[lo], s1 = ss[hi];
                const int i0 = si[lo], i1 = si[hi];
                const bool before = (s0 > s1) || (s0 == s1 && i0 < i1);
                if (before != desc_block) { ss[lo] = s1; ss[hi] = s0; si[lo] = i1; si[hi] = i0; }
            }
            __syncthreads();
        }
    for (int c = tid; c < CAND_TOP; c += blockDim.x) {
        top_sc[(size_t)u * CAND_TOP + c] = ss[c];
        top_id[(size_t)u * CAND_TOP + c] = si[c];
    }
}

__global__ void any_negative_kernel(const float* __restrict__ x, size_t n, int* __restrict__ flag)
{
    int f = 0;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        f |= (x[i] < 0.f);
    if (f) atomicOr(flag, 1);
}

// flag |= 1 when an id lies outside [0, n)  (the batched entry's check of the exclusion lists: millions of ids
// that are on the device anyway; a negative id of a signed type is a huge size_t)
template <class IX>
__global__ void any_id_out_of_range_kernel(const IX* __restrict__ ids, size_t count, size_t n, int* __restrict__ flag)
{
    int f = 0;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < count; i += (size_t)gridDim.x * blockDim.x)
        f |= ((size_t)ids[i] >= n);
    if (f) atomicOr(flag, 1);
}

}  // namespace tc
}  // namespace pmf
