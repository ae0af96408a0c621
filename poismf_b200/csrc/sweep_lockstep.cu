// poismf_b200 — the lock-step path for the heaviest cg rows of a side (lockstep.h): building its device plan and
// launching one half-sweep of the kernels of dense_rows.cuh.
#include <algorithm>
#include <vector>

#include <cub/cub.cuh>

#include "dense_rows.cuh"
#include "devpool.h"
#include "lockstep.h"

namespace pmf {

#define LS_CK(call) do { const cudaError_t e_ = (call); if (e_ != cudaSuccess) return e_; } while (0)

LockstepPlan::LockstepPlan() : P(new DenseParams()) {}
LockstepPlan::~LockstepPlan() = default;

void LockstepPlan::release()
{
    timings.clear();
    for (void* b : blocks) dfree(b);
    blocks.clear();
    H = 0; nnzH = 0;
}

cudaError_t LockstepPlan::build(const std::vector<int>& rows, const long long* h_ptr, const int* ind, const float* xv,
                                size_t other_dim, int k, int ldf, int num_sms_, std::vector<void*>& deferred,
                                cudaStream_t st, std::atomic<uint64_t>& launches)
{
    release();
    const LockstepTables t = lockstep_tables(h_ptr, rows, other_dim, num_sms_, ldf);
    if (ldf > 64 || t.H > 65535) return cudaErrorInvalidValue;
    // count elements of *ptr, owned by `owner`: the plan's `blocks` (a part-way failure leaves them for the caller's
    // release()) or, for the sort's temporaries, `deferred`
    auto alloc = [](std::vector<void*>& owner, auto** ptr, size_t count) {
        const cudaError_t e = dmalloc(ptr, std::max<size_t>(count * sizeof(**ptr), 16));
        if (e == cudaSuccess) owner.push_back((void*)*ptr);
        return e;
    };
    const int U = DN_TILE_ROWS;
    DenseParams& D = *P;
    D = DenseParams();
    D.H = t.H; D.T = t.T; D.U = U; D.ldf = ldf; D.k = k; D.L = ldf / 4;
    D.nnzH = t.nnzH; D.nchunks = t.nchunks; D.G = t.G; D.R = (int)other_dim;
    D.xv = xv;
    int *tables, *seg_ptr;
    long long* hbeg;
    uint2* ent;
    float* sx;
    LS_CK(alloc(blocks, &tables, t.i32.size()));
    LS_CK(alloc(blocks, &hbeg, t.H));
    LS_CK(alloc(blocks, &ent, t.nnzH));
    LS_CK(alloc(blocks, &sx, t.nnzH));
    LS_CK(alloc(blocks, &seg_ptr, t.n_seg));
    LS_CK(alloc(blocks, &D.p, t.nnzH));
    LS_CK(alloc(blocks, &D.q, t.nnzH));
    LS_CK(alloc(blocks, &D.dvec, t.n_dvec));
    LS_CK(alloc(blocks, &D.gprev, t.n_hist));
    LS_CK(alloc(blocks, &D.dprev, t.n_hist));
    LS_CK(alloc(blocks, &D.gpart, t.n_gpart));
    LS_CK(alloc(blocks, &D.lsp, t.n_lsp));
    LS_CK(alloc(blocks, &D.sc, t.H));
    LS_CK(alloc(blocks, &tile_counters, DN_TILE_COUNTERS));
    D.hrow = tables; D.hcol0 = tables + t.H; D.chunk_ptr = D.hcol0 + t.H + 1; D.chunk_h = D.chunk_ptr + t.H + 1;
    D.hbeg = hbeg; D.ent = ent; D.sx = sx; D.seg_ptr = seg_ptr;
    LS_CK(cudaMemcpyAsync(tables, t.i32.data(), t.i32.size() * sizeof(int), cudaMemcpyHostToDevice, st));
    LS_CK(cudaMemcpyAsync(hbeg, t.hbeg.data(), (size_t)t.H * sizeof(long long), cudaMemcpyHostToDevice, st));
    LS_CK(cudaMemsetAsync(D.q, 0, (size_t)t.nnzH * sizeof(float), st));
    // sort the heavy rows' non-zeros by (tile of the fixed matrix, heavy row); stable: ascending position inside
    const int nnz = t.nnzH;
    int *slot, *pos, *spos;
    unsigned *k1, *k2;
    unsigned char* tmp;
    for (int** q : {&slot, &pos, &spos}) LS_CK(alloc(deferred, q, nnz));
    for (unsigned** q : {&k1, &k2}) LS_CK(alloc(deferred, q, nnz));
    const int nseg = (int)(t.n_seg - 1);
    int bits = 1;
    while (bits < 32 && (1LL << bits) < nseg) bits++;
    size_t tb = 0;
    LS_CK(cub::DeviceRadixSort::SortPairs(nullptr, tb, k1, k2, pos, spos, nnz, 0, bits, st));
    LS_CK(alloc(deferred, &tmp, tb));
    const int grid = num_sms_ * 8;
    dense_fill_slot_kernel<<<dim3(8, t.H), 256, 0, st>>>(D.hcol0, t.H, slot);
    dense_keys_kernel<<<grid, 256, 0, st>>>(ind, slot, hbeg, D.hcol0, nnz, t.H, U, k1, pos);
    LS_CK(cub::DeviceRadixSort::SortPairs(tmp, tb, k1, k2, pos, spos, nnz, 0, bits, st));
    dense_unpack_kernel<<<grid, 256, 0, st>>>(k2, spos, ind, xv, hbeg, D.hcol0, nnz, t.H, U, ldf, ent, sx);
    dense_segments_kernel<<<grid, 256, 0, st>>>(k2, nnz, nseg, seg_ptr);
    launches.fetch_add(5, std::memory_order_relaxed);
    LS_CK(cudaGetLastError());
    H = t.H; nnzH = (unsigned long long)nnz; num_sms = num_sms_;
    return cudaSuccess;
}

// ~5 launches per cg iteration, all on `st`
cudaError_t LockstepPlan::run(float* M, float* const* peers, int npeers, size_t row_begin, const float* F,
                              const float* csum, const HalfSweepConsts<float>& hc, cudaStream_t st,
                              std::atomic<uint64_t>& launches)
{
    DenseParams& D = *P;
    const int ldf = D.ldf;
    D.M = M + row_begin * (size_t)ldf; D.F = F; D.csum = csum; D.hc = hc;
    D.npeers = npeers;
    for (int q = 0; q < 7; q++) D.peerM[q] = q < npeers ? peers[q] + row_begin * (size_t)ldf : nullptr;
    const size_t tile_bytes = (size_t)DN_TILE_ROWS * ldf * sizeof(float);
    const size_t smem_dots = tile_bytes + (size_t)H * sizeof(int);
    const size_t smem_g = 2 * tile_bytes + (size_t)(H + DN_GROUPS) * ldf * sizeof(float);
    LS_CK(ensure_smem((const void*)dense_walk_kernel<0>, smem_dots));
    LS_CK(ensure_smem((const void*)dense_walk_kernel<1>, smem_dots));
    LS_CK(ensure_smem((const void*)dense_walk_kernel<2>, smem_g));
    const int hg = (H + 3) / 4;
    const int gd = (int)std::min<long long>(4 * num_sms, D.T);   // dots passes: four persistent CTAs per SM
    const int ring = DN_TILE_COUNTERS;
    LS_CK(cudaMemsetAsync(tile_counters, 0, ring * sizeof(int), st));
    int n_dots = 0;
    dense_reset_kernel<<<(H + 127) / 128, 128, 0, st>>>(D);
    D.tile_counter = tile_counters + (n_dots++ % ring);
    dense_walk_kernel<0><<<gd, DnWalk<0>::threads, smem_dots, st>>>(D);
    dense_ls_kernel<<<D.nchunks, 256, 0, st>>>(D, 0);
    dense_init_kernel<<<hg, 128, 0, st>>>(D);
    launches.fetch_add(4, std::memory_order_relaxed);
    const long long maxiter = hc.maxupd <= 0 ? (1LL << 40) : hc.maxupd;
    for (long long it = 0; it < maxiter; it++) {
        dense_walk_kernel<2><<<D.G, DnWalk<2>::threads, smem_g, st>>>(D);
        dense_k_kernel<<<H, 256, 0, st>>>(D);
        if (n_dots % ring == 0) LS_CK(cudaMemsetAsync(tile_counters, 0, ring * sizeof(int), st));   // all used up
        D.tile_counter = tile_counters + (n_dots++ % ring);
        dense_walk_kernel<1><<<gd, DnWalk<1>::threads, smem_dots, st>>>(D);
        dense_ls_kernel<<<D.nchunks, 256, 0, st>>>(D, 1);
        dense_choose_kernel<<<hg, 128, 0, st>>>(D);
        launches.fetch_add(5, std::memory_order_relaxed);
        if ((it & 7) == 7 && it + 1 < maxiter) {
            // long iteration budgets (factors_multiple's cg): stop enqueueing once every row is done
            std::vector<DenseScal> hs(H);
            LS_CK(cudaMemcpyAsync(hs.data(), D.sc, (size_t)H * sizeof(DenseScal), cudaMemcpyDeviceToHost, st));
            LS_CK(cudaStreamSynchronize(st));
            bool any = false;
            for (auto& q : hs) any = any || q.active;
            if (!any) break;
        }
    }
    return cudaGetLastError();
}

}  // namespace pmf
