// poismf_b200 — instantiation of the register-tile row kernels (regtile.cuh) for one method: one kernel per
// entry of REGTILE_SHAPES (row_plan.h) and chunk count.
//   PMF_RT_METHOD : M_PG or M_CG
#pragma once
#include <utility>
#include "regtile.cuh"
#include "launch.h"

namespace pmf {

template <int NC, int METHOD, size_t... I>
static cudaError_t rt_launch_nc(const BinShape& b, const LaunchArgs& a, const SideParams<float>& P,
                                std::index_sequence<I...>)
{
    cudaError_t e = cudaErrorInvalidConfiguration;
    ((b.rt_nw == REGTILE_SHAPES[I].nw && b.rt_tpl == REGTILE_SHAPES[I].tpl &&
      (e = launch_persistent(rows_regtile_kernel<NC, REGTILE_SHAPES[I].tpl, REGTILE_SHAPES[I].nw, METHOD>, b, a, P),
       true)) || ...);
    return e;
}

#if PMF_RT_METHOD == 3
cudaError_t launch_regtile_pg(const BinShape& b, const LaunchArgs& a, const SideParams<float>& P)
#else
cudaError_t launch_regtile_cg(const BinShape& b, const LaunchArgs& a, const SideParams<float>& P)
#endif
{
    constexpr int METHOD = PMF_RT_METHOD;
    constexpr auto shapes = std::make_index_sequence<sizeof(REGTILE_SHAPES) / sizeof(REGTILE_SHAPES[0])>();
    if (b.rt_nc == 2) return rt_launch_nc<2, METHOD>(b, a, P, shapes);
    if (b.rt_nc == 4) return rt_launch_nc<4, METHOD>(b, a, P, shapes);
    return cudaErrorInvalidConfiguration;
}

}  // namespace pmf
