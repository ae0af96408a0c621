// poismf_b200 — a thread-block CLUSTER as the team of one heavy row.
//
// Power-law count matrices have rows whose gathered tile is far larger than one SM's
// shared memory (the heaviest items of the Last.FM-shaped synthetic have > 2e5
// non-zeros: 50 MB of factor rows).  Such a row is given to a cluster of G <= 16 CTAs:
//   * the row's non-zeros are cut into G contiguous slices, one per CTA; each CTA stages
//     ITS slice of the tile in its own shared memory (or streams it from L2 when even the
//     slice is too large),
//   * every CTA keeps a full replica of the solver's k-vectors and scalars and executes
//     the solver's control flow redundantly, so k-vector work needs no communication,
//   * the only exchanges are the sums over non-zeros (the log-likelihood term, and the
//     k-vector sum_t c_t F_t): each CTA publishes its partial in its own shared memory,
//     one hardware cluster barrier, then every CTA reads all G partials through
//     distributed shared memory and folds them in rank order — so all replicas get the
//     same bits and keep taking the same branches.
// Exchange slots are double-buffered by parity: one cluster barrier per reduction.
#pragma once
#include <cooperative_groups.h>
#include "common.cuh"
#include "sweep_consts.h"

namespace pmf {
namespace cg = cooperative_groups;

struct ClusterTeam : BlockOps {
    double* xbuf;       // 2 * GANG_XSLOTS doubles, viewed as `real`
    unsigned crank, csize;
    mutable int parity;
    PMF_DEVINL explicit ClusterTeam(void* scratch, void* exchange) : xbuf((double*)exchange), parity(0)
    {
        red = (double*)scratch;
        cg::cluster_group cl = cg::this_cluster();
        crank = cl.block_rank();
        csize = cl.num_blocks();
    }
    // ---- cluster-wide sums over the row's non-zeros -----------------------------
    static constexpr bool is_gang = true;
    PMF_DEVINL bool owns_row() const { return crank == 0; }
    PMF_DEVINL unsigned crank_() const { return crank; }
    PMF_DEVINL unsigned csize_() const { return csize; }
    template <class T> PMF_DEVINL T* slot() const { return reinterpret_cast<T*>(xbuf) + (size_t)parity * GANG_XSLOTS; }
    template <class T, int N> PMF_DEVINL void nnz_sum_n(T (&v)[N]) const
    {
        cg::cluster_group cl = cg::this_cluster();
        sum_n(v);                                               // CTA-local first
        T* mine = slot<T>();
        if (threadIdx.x == 0)
#pragma unroll
            for (int j = 0; j < N; j++) mine[j] = v[j];
        cl.sync();
#pragma unroll
        for (int j = 0; j < N; j++) v[j] = 0;
        for (unsigned r = 0; r < csize; r++) {                  // same order on every CTA
            const T* theirs = cl.map_shared_rank(mine, r);
#pragma unroll
            for (int j = 0; j < N; j++) v[j] += theirs[j];
        }
        parity ^= 1;
    }
    template <class T> PMF_DEVINL T nnz_sum(T v) const
    {
        T a[1] = {v};
        nnz_sum_n(a);
        return a[0];
    }
    // vec[0..n) <- sum over CTAs of their vec[0..n)  (vec is a CTA-local shared vector)
    template <class real> PMF_DEVINL void nnz_vec_sum(real* vec, int n) const
    {
        cg::cluster_group cl = cg::this_cluster();
        real* mine = slot<real>();
        for (int i = threadIdx.x; i < n; i += blockDim.x) mine[i] = vec[i];
        cl.sync();
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            real acc = 0;
            for (unsigned r = 0; r < csize; r++) acc += cl.map_shared_rank(mine, r)[i];
            vec[i] = acc;
        }
        parity ^= 1;
        __syncthreads();
    }
};

}  // namespace pmf
