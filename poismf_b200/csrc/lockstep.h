// poismf_b200 — host interface of the lock-step path: the heaviest cg rows of a side, solved together by the whole
// GPU (dense_rows.cuh, DESIGN §4 (b)).  sweep_lockstep.cu builds a side's plan from the rows plan_rows picks and the
// tables of lockstep_tables (row_plan.h), runs its half-sweeps and releases it.
//
// Preconditions: float32 factors with ldf <= 64 (an entry packs the byte offset of a factor row within its tile into
// 16 bits; the per-row gradient history holds 64 reals) and at most 65535 rows (the row takes the other 16 bits).
// build() returns cudaErrorInvalidValue outside them.
#pragma once
#include <cuda_runtime.h>
#include <atomic>
#include <cstdint>
#include <memory>
#include <vector>
#include "launch.h"

namespace pmf {

struct DenseParams;
template <class real> struct HalfSweepConsts;

// One side's plan: the device arrays of its rows and the kernels' parameter block, whose plan-time fields build()
// sets once.  Callers synchronise the streams that used a plan before they release or rebuild it (devpool.h).
// Both calls add the kernels they launch to `launches`.
class LockstepPlan {
public:
    LockstepPlan();
    ~LockstepPlan();
    int rows() const { return H; }
    unsigned long long nnz() const { return nnzH; }
    Timings timings;    // profiling: one pair per half-sweep

    // rows: heaviest first; h_ptr: the side's host row pointers; ind, xv: its device column ids and values;
    // other_dim: rows of the fixed matrix.  The sort's temporaries go to `deferred`, for release once `st` is synchronised.
    cudaError_t build(const std::vector<int>& rows, const long long* h_ptr, const int* ind, const float* xv,
                      size_t other_dim, int k, int ldf, int num_sms, std::vector<void*>& deferred, cudaStream_t st,
                      std::atomic<uint64_t>& launches);
    // one half-sweep on `st`: M and the npeers peers' replicas are the matrix being updated, from its row 0, and the
    // side's rows start at row_begin; F is the fixed matrix
    cudaError_t run(float* M, float* const* peers, int npeers, size_t row_begin, const float* F, const float* csum,
                    const HalfSweepConsts<float>& hc, cudaStream_t st, std::atomic<uint64_t>& launches);
    void release();

private:
    int H = 0, num_sms = 0;
    unsigned long long nnzH = 0;
    std::unique_ptr<DenseParams> P;
    int* tile_counters = nullptr;
    std::vector<void*> blocks;   // every device allocation of the plan
};

}  // namespace pmf
