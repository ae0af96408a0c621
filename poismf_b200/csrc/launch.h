// poismf_b200 — host-side launch interface of the row kernels, shared by api.cu and the kernel TUs.
#pragma once
#include <cuda_runtime.h>
#include <algorithm>
#include <map>
#include <mutex>
#include <tuple>
#include <utility>
#include <vector>
#include "row_plan.h"

namespace pmf {

// profiling: a start/stop event pair around each launch of a bin (or of the lock-step path)
struct Timings {
    std::vector<cudaEvent_t> ev;
    cudaError_t start(cudaStream_t st)
    {
        cudaEvent_t a = nullptr, b = nullptr;
        cudaError_t e = cudaEventCreate(&a);
        if (e == cudaSuccess && (e = cudaEventCreate(&b)) != cudaSuccess) cudaEventDestroy(a);
        if (e != cudaSuccess) return e;
        ev.push_back(a); ev.push_back(b);
        return cudaEventRecord(a, st);
    }
    cudaError_t stop(cudaStream_t st) { return cudaEventRecord(ev.back(), st); }
    int launches() const { return (int)(ev.size() / 2); }
    double ms() const
    {
        double sum = 0;
        for (size_t i = 0; i + 1 < ev.size(); i += 2) {
            float ms = 0;
            if (cudaEventElapsedTime(&ms, ev[i], ev[i + 1]) == cudaSuccess) sum += ms;
        }
        return sum;
    }
    void clear()
    {
        for (auto e : ev) cudaEventDestroy(e);
        ev.clear();
    }
};

template <class real> struct SideParams;

// what varies from one launch of a bin to the next
struct LaunchArgs {
    cudaStream_t stream;
    int needed;          // CTAs (clusters) needed to give every row its own team
    int max_grid;        // upper bound on the grid (global-scratch bin)
    int num_sms;
    bool cached;         // cg: re-use <x,F_t>, <d,F_t> in the line search (fast mode, limit_step)
};

// Occupancy queries and attribute calls cost far more than a launch, so both are cached.  Function attributes
// and occupancy are per device (a process may hold handles on several GPUs: pmf_b200_create(device),
// POISMF_B200_DEVICE), so the keys carry the current device.
inline int current_device()
{
    int d = 0;
    cudaGetDevice(&d);
    return d;
}

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize): the attribute is a per-kernel maximum, so it is only ever
// raised (bins of different tile capacity share one kernel)
inline cudaError_t ensure_smem(const void* kern, size_t bytes)
{
    static std::mutex mu;
    static std::map<std::pair<int, const void*>, size_t> current;
    std::lock_guard<std::mutex> lk(mu);
    size_t& cur = current[std::make_pair(current_device(), kern)];
    if (bytes <= cur) return cudaSuccess;
    const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e == cudaSuccess) cur = bytes;
    return e;
}

// *out = CTAs of `kern` resident per SM (cluster 1) or clusters resident on the device (cluster > 1) at this
// block size and dynamic shared memory; at least 1
inline cudaError_t resident(int* out, const void* kern, int threads, size_t smem, int cluster, int num_sms)
{
    static std::mutex mu;
    static std::map<std::tuple<int, const void*, int, size_t, int>, int> cache;
    std::lock_guard<std::mutex> lk(mu);
    const auto key = std::make_tuple(current_device(), kern, threads, smem, cluster);
    auto it = cache.find(key);
    if (it != cache.end()) { *out = it->second; return cudaSuccess; }
    int n = 0;
    if (cluster == 1) {
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kern, threads, smem) != cudaSuccess || n < 1) n = 1;
    } else {
        if (cluster > 8) {
            const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
            if (e != cudaSuccess) return e;
        }
        cudaLaunchConfig_t lc = {};
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = cluster; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        lc.attrs = at; lc.numAttrs = 1;
        lc.gridDim = dim3(cluster); lc.blockDim = dim3(threads); lc.dynamicSmemBytes = smem;
        if (cudaOccupancyMaxActiveClusters(&n, kern, &lc) != cudaSuccess || n < 1) {
            cudaGetLastError();
            n = std::max(num_sms / cluster / 2, 1);
        }
    }
    *out = cache[key] = n;
    return cudaSuccess;
}

// Persistent grid of one CTA per team or row: as many CTAs as can be resident (SMs x occupancy), never more than
// there are rows to hand out.
template <class real>
cudaError_t launch_persistent(void (*kern)(SideParams<real>), const BinShape& b, const LaunchArgs& a,
                              const SideParams<real>& P)
{
    int occ = 1;
    cudaError_t e = ensure_smem((const void*)kern, b.smem);
    if (e == cudaSuccess) e = resident(&occ, (const void*)kern, b.threads, b.smem, 1, a.num_sms);
    if (e != cudaSuccess) return e;
    const long long g = std::max(1LL, std::min<long long>({(long long)a.num_sms * occ, a.needed, a.max_grid}));
    kern<<<(unsigned)g, b.threads, b.smem, a.stream>>>(P);
    return cudaGetLastError();
}

template <class real> cudaError_t launch_rows_pgcg_fast(const BinShape&, const LaunchArgs&, const SideParams<real>&);
template <class real> cudaError_t launch_rows_pgcg_strict(const BinShape&, const LaunchArgs&, const SideParams<real>&);
template <class real> cudaError_t launch_rows_tn_fast(const BinShape&, const LaunchArgs&, const SideParams<real>&);
template <class real> cudaError_t launch_rows_tn_strict(const BinShape&, const LaunchArgs&, const SideParams<real>&);
// cluster-per-row kernels exist in fast numerics only
template <class real> cudaError_t launch_gang_pgcg_fast(const BinShape&, const LaunchArgs&, const SideParams<real>&);
template <class real> cudaError_t launch_gang_tn_fast(const BinShape&, const LaunchArgs&, const SideParams<real>&);
// register-tile kernels: fast numerics, float32, w_mult == 1; pg, and cg with limit_step + cached line search
cudaError_t launch_regtile_pg(const BinShape&, const LaunchArgs&, const SideParams<float>&);
cudaError_t launch_regtile_cg(const BinShape&, const LaunchArgs&, const SideParams<float>&);

}  // namespace pmf
