// poismf_b200 — explicit instantiation of the half-sweep kernels for one
// (numerics mode, solver family) pair.  Included by four tiny .cu files so that
// the strict variants can be compiled with --fmad=false and the large tncg
// kernels build in parallel with the pg/cg ones.
//   PMF_INST_STRICT : 0/1      PMF_INST_TN : 0 (pg + cg) / 1 (tncg)
#pragma once
#include "kernels.cuh"
#include "launch.h"

namespace pmf {

// the kernel a (sub-)warp or CTA bin names; strict numerics compile 32-lane and 256-thread teams only
template <class real, int METHOD, bool STRICT, bool CACHED>
static cudaError_t launch_one(const BinShape& b, const LaunchArgs& a, const SideParams<real>& P)
{
    if (b.kind == BinKind::Cta) {
        if constexpr (!STRICT)
            if (b.threads == 512) return launch_persistent(rows_block_kernel<real, METHOD, STRICT, CACHED, 512>, b, a, P);
        return launch_persistent(rows_block_kernel<real, METHOD, STRICT, CACHED, 256>, b, a, P);
    }
    if (b.lanes == 16) {
        if constexpr (STRICT) return cudaErrorInvalidConfiguration;
        else return launch_persistent(rows_warp_kernel<real, METHOD, STRICT, CACHED, 16>, b, a, P);
    }
    return launch_persistent(rows_warp_kernel<real, METHOD, STRICT, CACHED, 32>, b, a, P);
}

#if !PMF_INST_STRICT
// ---- cluster-per-row launch (cudaLaunchKernelEx with a cluster dimension) ----
template <class real, int METHOD, bool CACHED>
static cudaError_t launch_gang_one(const BinShape& b, const LaunchArgs& a, const SideParams<real>& P)
{
    // streaming bins are compiled for 2 CTAs per SM (64 registers) so that they can share an SM with the
    // short-row kernels while they wait on L2
    auto kern = b.kind == BinKind::Streaming ? rows_cluster_kernel<real, METHOD, CACHED, 2>
                                             : rows_cluster_kernel<real, METHOD, CACHED, 1>;
    int nclusters = 1;
    cudaError_t e = ensure_smem((const void*)kern, b.smem);
    if (e == cudaSuccess) e = resident(&nclusters, (const void*)kern, b.threads, b.smem, b.cluster, a.num_sms);
    if (e != cudaSuccess) return e;
    nclusters = std::min({nclusters, a.needed, a.max_grid});
    cudaLaunchConfig_t lc = {};
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = b.cluster; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    lc.attrs = at; lc.numAttrs = 1;
    lc.gridDim = dim3((unsigned)(nclusters * b.cluster));
    lc.blockDim = dim3(b.threads); lc.dynamicSmemBytes = b.smem; lc.stream = a.stream;
    return cudaLaunchKernelEx(&lc, kern, P);
}
#if PMF_INST_TN
template <class real>
cudaError_t launch_gang_tn_fast(const BinShape& b, const LaunchArgs& a, const SideParams<real>& P)
{
    return launch_gang_one<real, M_TNCG, false>(b, a, P);
}
template cudaError_t launch_gang_tn_fast<float>(const BinShape&, const LaunchArgs&, const SideParams<float>&);
template cudaError_t launch_gang_tn_fast<double>(const BinShape&, const LaunchArgs&, const SideParams<double>&);
#else
template <class real>
cudaError_t launch_gang_pgcg_fast(const BinShape& b, const LaunchArgs& a, const SideParams<real>& P)
{
    if (P.hc.method == M_PG) return launch_gang_one<real, M_PG, false>(b, a, P);
    if (a.cached) return launch_gang_one<real, M_CG, true>(b, a, P);
    return launch_gang_one<real, M_CG, false>(b, a, P);
}
template cudaError_t launch_gang_pgcg_fast<float>(const BinShape&, const LaunchArgs&, const SideParams<float>&);
template cudaError_t launch_gang_pgcg_fast<double>(const BinShape&, const LaunchArgs&, const SideParams<double>&);
#endif
#endif

#if PMF_INST_TN
#define PMF_LAUNCH_NAME_(s) launch_rows_tn_##s
#else
#define PMF_LAUNCH_NAME_(s) launch_rows_pgcg_##s
#endif
#if PMF_INST_STRICT
#define PMF_LAUNCH_NAME PMF_LAUNCH_NAME_(strict)
#else
#define PMF_LAUNCH_NAME PMF_LAUNCH_NAME_(fast)
#endif

template <class real>
cudaError_t PMF_LAUNCH_NAME(const BinShape& b, const LaunchArgs& a, const SideParams<real>& P)
{
    constexpr bool S = PMF_INST_STRICT != 0;
#if PMF_INST_TN
    return launch_one<real, M_TNCG, S, false>(b, a, P);
#else
    if (P.hc.method == M_PG) return launch_one<real, M_PG, S, false>(b, a, P);
    if (!S && a.cached) return launch_one<real, M_CG, S, true>(b, a, P);
    return launch_one<real, M_CG, S, false>(b, a, P);
#endif
}
template cudaError_t PMF_LAUNCH_NAME<float>(const BinShape&, const LaunchArgs&, const SideParams<float>&);
template cudaError_t PMF_LAUNCH_NAME<double>(const BinShape&, const LaunchArgs&, const SideParams<double>&);

}  // namespace pmf
