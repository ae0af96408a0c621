// poismf_b200 — half-sweep kernels: a (sub-)warp per short row, a CTA per longer row, a
// thread-block cluster per heavy row.
//
// Replaces the OpenMP `parallel for schedule(dynamic)` row loops of the reference
// (/root/reference/src/poismf.c:159-187 pg, :296-321 cg, :352-397 tncg).
// Rows are binned by non-zero count on the host (plan_rows in row_plan.h); each bin is one
// launch of a persistent grid whose teams fetch rows from a list sorted by decreasing
// length (longest-processing-time-first) through an atomic counter.
#pragma once
#include "cluster_team.cuh"
#include "solver_pg_cg.cuh"
#include "solver_tn.cuh"
#include "sweep_consts.h"

namespace pmf {

template <class real> struct SideParams {
    real* M;               // factors being updated  [dim   x ldf]
    const real* F;         // fixed factors          [other x ldf]
    const real* xv;        // non-zero values of this side's compressed matrix
    const long long* ptr;  // row pointers (CSR for the A side, CSC for the B side)
    const int* ind;        // indices into F
    const real* csum;      // prepared column sums of F (+l1, pg: pre-scaled)
    const int* rows;       // rows of this launch, longest first
    int nrows;
    int* counter;          // dynamic fetch counter (zeroed before the launch)
    int k, kp, ldf;
    int cap;               // tile capacity (non-zeros) of a team's shared slice; 0: tile stays in global
    int acap;              // capacity of the per-non-zero arrays (x, <x,F>, coefficients, <d,F>) in the slice;
                           // == cap for staged bins; > 0 with cap == 0: tile streamed, arrays kept on chip
    int slice_bytes;       // shared bytes per team
    HalfSweepConsts<real> hc;
    real* gscratch;        // per-CTA global scratch for rows that are not staged (3*gs_stride reals)
    long long gs_stride;
    unsigned long long* n_unchanged;  // tncg early-stop counter (src/poismf.c:393-396)
    real* peerM[7];        // the same rows of M in the other GPUs' replicas (NVLink peer memory)
    int npeers;            // 0: single GPU, or replicas refreshed by a collective instead
};

PMF_DEVINL int num_vecs(int method)
{
    return method == M_PG ? 3 : (method == M_CG ? 7 : TN_NUM_VECS);
}

// Shared-memory slice of one team:
//   [team scratch 640 B][cluster exchange 2*272*8 B (gangs only)][gscr team*16 B][vectors NV*kp]
//   [xv,pa,pb,pc: 4*cap][tile cap*kp]
template <class real> struct Slice {
    void* team_scratch;
    void* xchg;
    real* gscr;
    real* vecs;
    real *xv, *pa, *pb, *pc;
    real* tile;
    PMF_DEVINL Slice(unsigned char* base, int team_size, int nvec, int kp, int cap, bool gang = false, int acap = -1)
    {
        if (acap < 0) acap = cap;
        team_scratch = base; if (team_size > 32) base += 640;   // (sub-)warp teams reduce by shuffles only
        xchg = base; if (gang) base += GANG_XBYTES;
        gscr = (real*)base; base += (size_t)team_size * 16;
        vecs = (real*)base; base += (size_t)nvec * kp * sizeof(real);
        xv = (real*)base; pa = xv + acap; pb = pa + acap; pc = pb + acap;
        base += (size_t)4 * acap * sizeof(real);
        tile = (real*)base;
    }
};

template <class real, int METHOD, bool STRICT, bool CACHED, class Team>
PMF_DEVINL void process_row(const Team& tm, const SideParams<real>& P, const Slice<real>& S,
                            int row, real* gscratch_cta)
{
    long long beg = P.ptr[row];
    int n = (int)(P.ptr[row + 1] - beg);
    if (Team::is_gang) {
        // this CTA's contiguous slice of the row's non-zeros
        const int chunk = (((n + (int)tm.csize_() - 1) / (int)tm.csize_()) + 3) & ~3;
        const int t0 = min(n, (int)tm.crank_() * chunk);
        const int t1 = min(n, t0 + chunk);
        beg += t0;
        n = t1 - t0;
    }
    const int k = P.k, kp = P.kp;
    RowView<real> rv;
    rv.F = P.F; rv.ind = P.ind + beg; rv.n = n; rv.k = k; rv.kp = kp; rv.ldf = P.ldf;
    rv.gscr = S.gscr;
    const int nvec = num_vecs(METHOD);
    // zero every vector (pads must be 0 and finite for the 16-byte dot loops)
    for (int i = tm.rank(); i < nvec * kp; i += tm.size()) S.vecs[i] = (real)0;
    if (P.cap > 0 && n <= P.cap) {
        rv.tile = S.tile; rv.xv = S.xv; rv.pa = S.pa; rv.pb = S.pb; rv.pc = S.pc;
        stage_tile(tm, P.F, rv.ind, P.xv + beg, n, P.ldf, kp, S.tile, S.xv, reinterpret_cast<int*>(S.pa));
    } else if (n <= P.acap) {
        // tile streamed from L2, but the per-non-zero arrays (read by every line-search trial) on chip
        rv.tile = nullptr; rv.xv = S.xv; rv.pa = S.pa; rv.pb = S.pb; rv.pc = S.pc;
        for (int t = tm.rank(); t < n; t += tm.size()) S.xv[t] = P.xv[beg + t];
        tm.sync();
    } else {
        rv.tile = nullptr; rv.xv = P.xv + beg;
        rv.pa = gscratch_cta; rv.pb = gscratch_cta + P.gs_stride; rv.pc = gscratch_cta + 2 * P.gs_stride;
        tm.sync();
    }
    real* V = S.vecs;
    real* x = V;                  // vector 0: the row being solved
    real* csum = V + kp;          // vector 1: column sums for this row
    real* Mrow = P.M + (size_t)row * P.ldf;
    for (int i = tm.rank(); i < k; i += tm.size()) x[i] = Mrow[i];
    if (P.hc.w == (real)1) {
        for (int i = tm.rank(); i < k; i += tm.size()) csum[i] = P.csum[i];
        tm.sync();
    } else {
        tm.sync();
        weighted_colsum<STRICT>(tm, rv, P.csum, P.hc, rv.pb, csum);
    }

    if (METHOD == M_PG) {
        solve_pg<STRICT>(tm, rv, P.hc, x, csum, V + 2 * kp);
    } else if (METHOD == M_CG) {
        CgVecs<real> vv;
        vv.x = x; vv.csum = csum;
        vv.g0 = V + 2 * kp; vv.g1 = V + 3 * kp; vv.d0 = V + 4 * kp; vv.d1 = V + 5 * kp; vv.xnew = V + 6 * kp;
        if (CACHED && !STRICT && P.hc.limit_step) solve_cg_cached(tm, rv, P.hc, vv);
        else solve_cg<STRICT>(tm, rv, P.hc, vv);
    } else {
        solve_tn<STRICT>(tm, rv, P.hc, V, Mrow, P.n_unchanged);
    }
    tm.sync();
    if (tm.owns_row()) {
        for (int i = tm.rank(); i < k; i += tm.size()) Mrow[i] = x[i];
        // fused exchange: the solved row goes straight into every peer's replica over NVLink
        for (int p = 0; p < P.npeers; p++) {
            real* prow = P.peerM[p] + (size_t)row * P.ldf;
            for (int i = tm.rank(); i < k; i += tm.size()) prow[i] = x[i];
        }
    }
    tm.sync();
}

// W lanes per row (W = 32: a warp per row; W = 16: two short rows side by side in one
// warp).  Each team owns one slice of the CTA's dynamic shared memory and fetches rows from
// the bin's list through an atomic counter.
template <class real, int METHOD, bool STRICT, bool CACHED, int W>
__global__ void __launch_bounds__(256, PMF_WARP_KERNEL_MIN_CTAS) rows_warp_kernel(const SideParams<real> P)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int team_id = threadIdx.x / W;
    Slice<real> S(smem + (size_t)team_id * P.slice_bytes, W, num_vecs(METHOD), P.kp, P.cap, false, P.acap);
    SubWarpTeam<W> tm(S.team_scratch);
    for (;;) {
        int idx = 0;
        if (tm.lane == 0) idx = atomicAdd(P.counter, 1);
        idx = tm.bcast0(idx);
        if (idx >= P.nrows) break;
        process_row<real, METHOD, STRICT, CACHED>(tm, P, S, P.rows[idx], (real*)nullptr);
    }
}

// THREADS = 256 (several CTAs per SM: registers capped at 80) or 512 (one CTA per SM)
template <class real, int METHOD, bool STRICT, bool CACHED, int THREADS>
__global__ void __launch_bounds__(THREADS, THREADS == 256 ? 3 : 1) rows_block_kernel(const SideParams<real> P)
{
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ int next_row;
    Slice<real> S(smem, blockDim.x, num_vecs(METHOD), P.kp, P.cap, false, P.acap);
    BlockTeam tm(S.team_scratch);
    real* gs = P.gscratch ? P.gscratch + (size_t)blockIdx.x * 3 * P.gs_stride : nullptr;
    for (;;) {
        __syncthreads();
        if (threadIdx.x == 0) next_row = atomicAdd(P.counter, 1);
        __syncthreads();
        const int idx = next_row;
        if (idx >= P.nrows) break;
        process_row<real, METHOD, STRICT, CACHED>(tm, P, S, P.rows[idx], gs);
    }
}

// One thread-block cluster per heavy row (fast numerics only: the cross-CTA fold changes
// the summation order).  Clusters draw rows from the bin's list, longest first.
// MINB = 1: resident slices (the CTA owns the SM's shared memory anyway); MINB = 2: streaming
// slices, registers capped at 64 so that the CTA can share an SM with the short-row kernels
template <class real, int METHOD, bool CACHED, int MINB>
__global__ void __launch_bounds__(512, MINB) rows_cluster_kernel(const SideParams<real> P)
{
    extern __shared__ __align__(16) unsigned char smem[];
    cg::cluster_group cl = cg::this_cluster();
    Slice<real> S(smem, blockDim.x, num_vecs(METHOD), P.kp, P.cap, true, P.acap);
    ClusterTeam tm(S.team_scratch, S.xchg);
    __shared__ int next_row;
    real* gs = P.gscratch ? P.gscratch + (size_t)blockIdx.x * 3 * P.gs_stride : nullptr;
    int* leader_slot = cl.map_shared_rank(&next_row, 0);
    for (;;) {
        // the cluster's rank-0 CTA draws the next row (longest first); peers read it over DSMEM
        if (cl.block_rank() == 0 && threadIdx.x == 0) next_row = atomicAdd(P.counter, 1);
        cl.sync();
        const int idx = *leader_slot;
        cl.sync();
        if (idx >= P.nrows) break;
        process_row<real, METHOD, false, CACHED>(tm, P, S, P.rows[idx], gs);
    }
    cl.sync();   // nobody leaves while a peer may still read its shared memory
}

}  // namespace pmf
