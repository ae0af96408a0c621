// poismf_b200 — small streaming kernels around the row solvers:
// index narrowing on upload, column sums (the "all items" term of the gradient,
// /root/reference/src/poismf.c:77-83,512-514,562-564), empty-row zeroing
// (:166-169,:308-311,:367-370) and predict_multiple (src/pred.c:42-64).
#pragma once
#include "common.cuh"

namespace pmf {

// host sparse_ix (size_t) -> device int32 indices (row pointers are widened to int64 on the host)
template <class SRC>
__global__ void narrow_indices_kernel(const SRC* __restrict__ src, int* __restrict__ dst, size_t n)
{
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        dst[i] = (int)src[i];
}
template <class real> struct ColsumFinal {
    real l1;        // added when > 0                       (:513-514)
    real scale1;    // pg, w==1: -step                      (:523-524, :573-574)
    real scale2;    // pg, w==1, A side only: -step again   (:577, quirk Q1)
    int nscale;     // 0, 1 or 2
};
template <class real> PMF_DEVINL real colsum_finish(real v, const ColsumFinal<real>& fin)
{
    if (fin.l1 > (real)0) v = add_rn(v, fin.l1);
    if (fin.nscale >= 1) v = mul_rn(v, fin.scale1);
    if (fin.nscale >= 2) v = mul_rn(v, fin.scale2);
    return v;
}

// dense host layout [n x k]  <->  device layout [n x ldf] (rows padded to 16 bytes, pads zero)
template <class real>
__global__ void pad_rows_kernel(const real* __restrict__ dense, real* __restrict__ padded, size_t n, int k, int ldf)
{
    const size_t total = n * (size_t)ldf;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t r = i / ldf; const int c = (int)(i - r * ldf);
        padded[i] = c < k ? dense[r * k + c] : (real)0;
    }
}
template <class real>
__global__ void unpad_rows_kernel(const real* __restrict__ padded, real* __restrict__ dense, size_t n, int k, int ldf)
{
    const size_t total = n * (size_t)k;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t r = i / k; const int c = (int)(i - r * k);
        dense[i] = padded[r * ldf + c];
    }
}

// Reference order: out[c] = ((M[0,c] + M[1,c]) + M[2,c]) + ...   one thread per column.
template <class real>
__global__ void colsum_seq_kernel(const real* __restrict__ M, size_t nrow, int k, int ldf,
                                  ColsumFinal<real> fin, real* __restrict__ out)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= k) return;
    real acc = 0;
    size_t r = 0;
    for (; r + 8 <= nrow; r += 8) {
        real v[8];
#pragma unroll
        for (int j = 0; j < 8; j++) v[j] = M[(r + j) * (size_t)ldf + c];
#pragma unroll
        for (int j = 0; j < 8; j++) acc = add_rn(acc, v[j]);
    }
    for (; r < nrow; r++) acc = add_rn(acc, M[r * (size_t)ldf + c]);
    out[c] = colsum_finish(acc, fin);
}

// Fast order: per-CTA partial sums over a strided set of rows (fully coalesced:
// the [nrow x ldf] matrix is one contiguous stream), then a fixed-order fold.
template <class real>
__global__ void __launch_bounds__(256) colsum_partial_kernel(const real* __restrict__ M, size_t nrow, int ldf,
                                                             real* __restrict__ partial)
{
    extern __shared__ __align__(16) unsigned char sm_raw[];
    real* sm = reinterpret_cast<real*>(sm_raw);
    const int rpb = blockDim.x / ldf;            // rows per CTA per iteration
    const int sub = threadIdx.x / ldf, c = threadIdx.x - sub * ldf;
    real acc0 = 0, acc1 = 0;
    if (sub < rpb) {
        size_t r = (size_t)blockIdx.x * rpb + sub;
        const size_t stride = (size_t)gridDim.x * rpb;
        for (; r + stride < nrow; r += 2 * stride) {
            acc0 += M[r * ldf + c];
            acc1 += M[(r + stride) * ldf + c];
        }
        if (r < nrow) acc0 += M[r * ldf + c];
    }
    sm[threadIdx.x] = acc0 + acc1;
    __syncthreads();
    if (threadIdx.x < ldf) {
        real tot = sm[threadIdx.x];
        for (int s = 1; s < rpb; s++) tot += sm[s * ldf + threadIdx.x];
        partial[(size_t)blockIdx.x * ldf + threadIdx.x] = tot;
    }
}
template <class real>
__global__ void colsum_fold_kernel(const real* __restrict__ partial, int nparts, int k, int ldf,
                                   ColsumFinal<real> fin, real* __restrict__ out)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= k) return;
    real acc = 0;
    for (int p = 0; p < nparts; p++) acc += partial[(size_t)p * ldf + c];
    out[c] = colsum_finish(acc, fin);
}

// every row of M [n x ldf] := mean [k] (pads zero), or zero without `mean`: the starting point of the rows
// of factors_multiple (src/pred.c:144-147)
template <class real>
__global__ void fill_rows_kernel(real* __restrict__ M, size_t n, int k, int ldf, const real* __restrict__ mean)
{
    const size_t total = n * (size_t)ldf;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % (size_t)ldf);
        M[i] = (mean && c < k) ? mean[c] : (real)0;
    }
}

template <class real>
__global__ void zero_rows_kernel(real* __restrict__ M, const int* __restrict__ rows, int nrows, int ldf)
{
    const size_t total = (size_t)nrows * ldf;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int r = (int)(i / ldf), c = (int)(i - (size_t)r * ldf);
        M[(size_t)rows[r] * ldf + c] = (real)0;
    }
}

// ---- device-side completion of the fused exchange (sharded fits) ----------------------------------------
// Every rank owns 8 epoch slots in peer-mapped memory.  After the kernels of half-sweep e (whose row
// epilogues stored the solved rows into every replica) a one-thread kernel writes e into slot `self` of
// every rank; before the kernels of half-sweep e+1 a one-warp kernel spins until all of ITS OWN slots
// have reached e.  The host never waits between half-sweeps.  (Waiting for ALL ranks also covers the
// write-after-read hazard: nobody overwrites rows of a matrix a slower rank is still reading.)
struct PeerSignals {
    unsigned long long* slot[8];     // slot[r]: rank r's epoch array (own entry included)
    int n_ranks, self;
};
__global__ void signal_epoch_kernel(PeerSignals S, unsigned long long epoch)
{
    __threadfence_system();
    for (int r = 0; r < S.n_ranks; r++) *reinterpret_cast<volatile unsigned long long*>(S.slot[r] + S.self) = epoch;
    __threadfence_system();
}
// `status` (device int, host-mapped copy checked by the caller) is set to 1 if a peer does not arrive
// within ~30 s: the fit then fails instead of hanging the GPU
__global__ void wait_epoch_kernel(const unsigned long long* own, int n_ranks, unsigned long long epoch, int* status)
{
    const int r = threadIdx.x;
    if (r < n_ranks) {
        const volatile unsigned long long* s = own + r;
        const long long t0 = clock64();
        while (*s < epoch) {
            __nanosleep(200);
            if (clock64() - t0 > 60000000000LL) { *status = 1; break; }
        }
    }
    __threadfence_system();
}

// out[i] = <A[ixA[i]], B[ixB[i]]>, summed left to right without contraction: the
// same bits as the reference's sequential dot.  One thread per pair; each thread
// streams its two factor rows with 16-byte loads (the path is a pure gather,
// 2*k*sizeof(real) bytes per output).
template <class real, class IX>
__global__ void predict_pairs_kernel(const real* __restrict__ A, const real* __restrict__ B,
                                     const IX* __restrict__ ixA, const IX* __restrict__ ixB,
                                     size_t n, int k, int ldf, real* __restrict__ out)
{
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const real* a = A + (ixA ? (size_t)ixA[i] : i) * ldf;       // no index arrays: row i of each (gathered) block
        const real* b = B + (ixB ? (size_t)ixB[i] : i) * ldf;
        real acc = 0;
        for (int c = 0; c < k; c++) acc = add_rn(acc, mul_rn(a[c], b[c]));
        out[i] = acc;
    }
}

// scores[u, j] = <A[user[u]], B[j]> (same left-to-right sum); excluded items get -inf later.
template <class real>
__global__ void score_items_kernel(const real* __restrict__ Arows, const real* __restrict__ B, size_t n, int k,
                                   int ldf, real* __restrict__ scores, int* __restrict__ ids)
{
    extern __shared__ __align__(16) unsigned char sm_raw[];
    real* a = reinterpret_cast<real*>(sm_raw);
    const real* arow = Arows + (size_t)blockIdx.y * ldf;
    for (int c = threadIdx.x; c < k; c += blockDim.x) a[c] = arow[c];
    __syncthreads();
    for (size_t j = blockIdx.x * (size_t)blockDim.x + threadIdx.x; j < n; j += (size_t)gridDim.x * blockDim.x) {
        const real* b = B + j * ldf;
        real acc = 0;
        for (int c = 0; c < k; c++) acc = add_rn(acc, mul_rn(a[c], b[c]));
        scores[(size_t)blockIdx.y * n + j] = acc;
        ids[(size_t)blockIdx.y * n + j] = (int)j;
    }
}
template <class real, class IX>
__global__ void mask_excluded_kernel(real* __restrict__ scores, size_t n, const IX* __restrict__ excl_ptr,
                                     const IX* __restrict__ excl_ix, size_t user0)
{
    const size_t u = blockIdx.y;
    const size_t beg = (size_t)excl_ptr[user0 + u], end = (size_t)excl_ptr[user0 + u + 1];
    for (size_t t = beg + blockIdx.x * (size_t)blockDim.x + threadIdx.x; t < end; t += (size_t)gridDim.x * blockDim.x)
        scores[u * n + (size_t)excl_ix[t]] = -RealTraits<real>::huge();
}
template <class real>
__global__ void gather_rows_kernel(const real* __restrict__ A, const long long* __restrict__ users, int nusers,
                                   int ldf, real* __restrict__ out)
{
    const size_t total = (size_t)nusers * ldf;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t u = i / ldf, c = i - u * ldf;
        out[i] = A[(size_t)users[u] * ldf + c];
    }
}

}  // namespace pmf
