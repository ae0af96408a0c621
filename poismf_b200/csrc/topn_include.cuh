// poismf_b200 — batched top-N over per-user candidate ("include") lists (src/topN.c:112-284 with
// include_ix, for many users at once).
//
// Every user ranks a different set of items, so there is no shared operand tile and tensor cores do
// not apply: per candidate the kernels read one k-wide row of B (k * sizeof(real) bytes) for 2k flops,
// which makes this a gather bound by L2 / HBM bandwidth.  Scores are the sequential, unfused sums of
// score_items_kernel (acc = add_rn(acc, mul_rn(a[c], b[c])), c = 0..k-1): bitwise the reference's strict
// build.  The ranking is descending score, ties by ascending item id; scores are compared through an
// order-preserving unsigned transform (negative scores included).
//
//   path (a) include_select_smem_kernel: lists up to a shared-memory capacity, one CTA per user: score
//            into shared memory, bitonic sort of (key, id), write the first n_top.
//   path (b) include_score_long_kernel + two CUB segmented radix sorts + include_emit_long_kernel: longer
//            lists.  The first sort orders each segment by item id, the second (stable) by score.
#pragma once
#include <cstdint>

#include "common.cuh"

namespace pmf {
namespace incl {

template <class real> struct OrderKey;
template <> struct OrderKey<float> {
    using T = uint32_t;
    PMF_DEVINL static T of(float s)
    {
        const uint32_t b = __float_as_uint(s == 0.f ? 0.f : s);      // -0 ranks as +0 (they compare equal)
        return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
    }
    PMF_DEVINL static float back(T k) { return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k); }
};
template <> struct OrderKey<double> {
    using T = unsigned long long;
    PMF_DEVINL static T of(double s)
    {
        const T b = (T)__double_as_longlong(s == 0. ? 0. : s);
        return (b >> 63) ? ~b : (b | (1ull << 63));
    }
    PMF_DEVINL static double back(T k) { return __longlong_as_double((long long)((k >> 63) ? (k & ~(1ull << 63)) : ~k)); }
};

template <class real> struct Vec;
template <> struct Vec<float> { using T = float4; };
template <> struct Vec<double> { using T = double2; };

// <a, b> in the reference's order; b is a row of B padded to a multiple of 16 bytes, a is in shared memory
template <class real>
PMF_DEVINL real dot_row(const real* a, const real* __restrict__ b, int k)
{
    using V = typename Vec<real>::T;
    constexpr int W = RealTraits<real>::V;
    const V* bv = reinterpret_cast<const V*>(b);
    real acc = 0;
    int c = 0;
    for (; c + W <= k; c += W) {
        const V x = __ldg(bv + c / W);
        const real* e = reinterpret_cast<const real*>(&x);
#pragma unroll
        for (int i = 0; i < W; i++) acc = add_rn(acc, mul_rn(a[c + i], e[i]));
    }
    for (; c < k; c++) acc = add_rn(acc, mul_rn(a[c], __ldg(b + c)));
    return acc;
}

template <class real>
PMF_DEVINL void load_row(real* a, const real* __restrict__ arow, int k)
{
    for (int c = threadIdx.x; c < k; c += blockDim.x) a[c] = arow[c];
}

// bytes of shared memory before the sort arrays (the user's row, 16-byte aligned)
__host__ __device__ inline size_t row_bytes(int ldf, size_t elem) { return (ldf * elem + 15) / 16 * 16; }

constexpr int SMEM_THREADS = 256;

// Path (a).  One CTA per listed user (`users`: positions in the chunk, all with lists of at most `cap` items,
// a power of two; the host launches one length class at a time so that shared memory fits the class).
// `ptr` holds the chunk's list offsets (rebased to 0), `ix` the chunk's lists.
template <class real, class IX>
__global__ void __launch_bounds__(SMEM_THREADS, 4)
include_select_smem_kernel(const real* __restrict__ Asel, const real* __restrict__ B, int k, int ldf,
                           const long long* __restrict__ ptr, const IX* __restrict__ ix, const int* __restrict__ users,
                           int cap, int n_top, IX* __restrict__ out_ix, real* __restrict__ out_sc)
{
    using K = typename OrderKey<real>::T;
    extern __shared__ __align__(16) unsigned char sm_raw[];
    const int u = users[blockIdx.x];
    const long long beg = ptr[u], L = ptr[u + 1] - beg;
    real* a = reinterpret_cast<real*>(sm_raw);
    K* key = reinterpret_cast<K*>(sm_raw + row_bytes(ldf, sizeof(real)));
    uint32_t* id = reinterpret_cast<uint32_t*>(key + cap);
    int P = 1;
    while (P < L) P <<= 1;
    load_row(a, Asel + (size_t)u * ldf, k);
    __syncthreads();
    for (int t = threadIdx.x; t < P; t += blockDim.x) {
        if (t < L) {
            const size_t j = (size_t)ix[beg + t];
            key[t] = OrderKey<real>::of(dot_row(a, B + j * ldf, k));
            id[t] = (uint32_t)j;
        } else {
            key[t] = 0;                    // below every score (0 is the transform of a negative NaN only)
            id[t] = 0xffffffffu;           // and after every item id
        }
    }
    __syncthreads();
    // bitonic sort into (key descending, id ascending)
    for (int size = 2; size <= P; size <<= 1)
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int t = threadIdx.x; t < P / 2; t += blockDim.x) {
                const int i = 2 * t - (t & (stride - 1)), j = i + stride;
                const bool fwd = (i & size) == 0;
                const K ki = key[i], kj = key[j];
                const uint32_t ii = id[i], ij = id[j];
                const bool j_first = kj > ki || (kj == ki && ij < ii);
                if (j_first == fwd) { key[i] = kj; key[j] = ki; id[i] = ij; id[j] = ii; }
            }
            __syncthreads();
        }
    for (int t = threadIdx.x; t < n_top; t += blockDim.x) {
        out_ix[(size_t)u * n_top + t] = (IX)id[t];
        if (out_sc) out_sc[(size_t)u * n_top + t] = OrderKey<real>::back(key[t]);
    }
}

// Path (b), scoring.  grid.y: the chunk's long-list users (`users`: their positions in the chunk), their
// candidates land at seg[i] .. seg[i+1] of the sort buffers.
template <class real, class IX>
__global__ void __launch_bounds__(256)
include_score_long_kernel(const real* __restrict__ Asel, const real* __restrict__ B, int k, int ldf,
                          const long long* __restrict__ ptr, const IX* __restrict__ ix, const int* __restrict__ users,
                          const int* __restrict__ seg, uint32_t* __restrict__ id_out,
                          typename OrderKey<real>::T* __restrict__ key_out)
{
    extern __shared__ __align__(16) unsigned char sm_raw[];
    real* a = reinterpret_cast<real*>(sm_raw);
    const int u = users[blockIdx.y];
    const long long beg = ptr[u], L = ptr[u + 1] - beg;
    const size_t s0 = (size_t)seg[blockIdx.y];
    load_row(a, Asel + (size_t)u * ldf, k);
    __syncthreads();
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < L; t += (long long)gridDim.x * blockDim.x) {
        const size_t j = (size_t)ix[beg + t];
        id_out[s0 + t] = (uint32_t)j;
        key_out[s0 + t] = OrderKey<real>::of(dot_row(a, B + j * ldf, k));
    }
}

// Path (b), output: the first n_top of every sorted segment
template <class real, class IX>
__global__ void include_emit_long_kernel(const int* __restrict__ users, const int* __restrict__ seg,
                                         const uint32_t* __restrict__ id, const typename OrderKey<real>::T* __restrict__ key,
                                         int n_top, IX* __restrict__ out_ix, real* __restrict__ out_sc)
{
    const size_t u = (size_t)users[blockIdx.x], s0 = (size_t)seg[blockIdx.x];
    for (int t = threadIdx.x; t < n_top; t += blockDim.x) {
        out_ix[u * n_top + t] = (IX)id[s0 + t];
        if (out_sc) out_sc[u * n_top + t] = OrderKey<real>::back(key[s0 + t]);
    }
}

}  // namespace incl
}  // namespace pmf
