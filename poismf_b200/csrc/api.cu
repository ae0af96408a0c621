// poismf_b200 — host side of libpoismf_b200.so: device handle, row planner,
// sweep driver and the C ABI declared in include/poismf_b200.h.
//
// The sweep driver restates run_poismf's outer loop (/root/reference/src/poismf.c:506-608)
// around device kernels: column sums -> (zero empty rows) -> binned row solvers,
// B side over CSC first, then A side over CSR, with pg's step halving between
// the two half-sweeps and tncg's early-stop bookkeeping.
#include <algorithm>
#include <atomic>
#include <csignal>
#include <ctime>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cmath>
#include <functional>
#include <map>
#include <mutex>
#include <string>
#include <type_traits>
#include <vector>

#include <cub/cub.cuh>
#include <nvtx3/nvToolsExt.h>

#include "../../include/poismf_b200.h"
#include "aux_kernels.cuh"
#include "devpool.h"
#include "ingest.cuh"
#include "staged_copy.h"
#include <chrono>
#include "kernels.cuh"
#include "launch.h"
#include "lockstep.h"
#include "topn_tc.cuh"
#include "topn_include.cuh"

using namespace pmf;

// ---------------------------------------------------------------------------
// errors, counters, interrupt flag
// ---------------------------------------------------------------------------
static thread_local std::string g_err;
static thread_local unsigned long long g_topn_stats[2] = {0, 0};   // users scored on tensor cores / redone exactly
static std::atomic<uint64_t> g_launches{0};
static volatile sig_atomic_t g_interrupted = 0;

static int fail(const char* fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    fprintf(stderr, "poismf_b200: %s\n", buf);
    return 1;
}
#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) return fail("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                                           __FILE__, __LINE__);                                    \
    } while (0)
#define LAUNCHED() (g_launches.fetch_add(1, std::memory_order_relaxed))

extern "C" const char* pmf_b200_last_error(void) { return g_err.c_str(); }
extern "C" uint64_t pmf_b200_kernel_launches(void) { return g_launches.load(); }
extern "C" int pmf_b200_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

// fn(real(), IX()) for the value type (PMF_F32: float, PMF_F64: double) and index width (8: uint64_t, 4: int)
// of a C call; `bad` is the error of any other pair
template <class F>
static int with_types(int dtype, int index_bytes, const char* bad, F&& fn)
{
    if (dtype == PMF_F32 && index_bytes == 8) return fn(float(), uint64_t());
    if (dtype == PMF_F32 && index_bytes == 4) return fn(float(), int());
    if (dtype == PMF_F64 && index_bytes == 8) return fn(double(), uint64_t());
    if (dtype == PMF_F64 && index_bytes == 4) return fn(double(), int());
    return fail("%s", bad);
}

// The device blocks of one call, released to the pool when it returns.  A call marks them settled once its
// last result is back on the host; one that returns before (an error, a failed check) may leave kernels
// using them, so the device is synchronised before they can go to another allocation.
struct DeviceBlocks {
    std::vector<void*> held;
    bool settled = false;
    template <class T> cudaError_t alloc(T** p, size_t bytes)
    {
        const cudaError_t e = dmalloc(p, bytes);
        if (e == cudaSuccess) held.push_back(*p);
        return e;
    }
    void adopt(void* p) { held.push_back(p); }
    ~DeviceBlocks()
    {
        if (!settled) cudaDeviceSynchronize();
        for (void* p : held) dfree(p);
    }
};

static inline int round_up(int v, int m) { return (v + m - 1) / m * m; }
static inline size_t round_up_sz(size_t v, size_t m) { return (v + m - 1) / m * m; }

// tile row stride: a multiple of 16 bytes whose 16-byte-unit count is odd, so that
// 16-byte accesses of consecutive lanes to consecutive tile rows hit distinct banks
static int tile_stride(int k, int V)
{
    int units = (k + V - 1) / V;
    if (units % 2 == 0) units++;
    return units * V;
}

// column sums of M [nrow x ldf] -> out [k], finished by `fin`, on `st`.  Both orders are fixed, so the sums are the
// same run to run and on every replica: strict = the reference's sequential order; else per-CTA partials over
// n_partial (at least) CTAs' strided rows, folded in CTA order.  `partial` holds n_partial x ldf reals.
template <class real>
static int launch_column_sums(const real* M, size_t nrow, int k, int ldf, const ColsumFinal<real>& fin, bool strict,
                              real* partial, int n_partial, real* out, cudaStream_t st)
{
    if (strict) {
        colsum_seq_kernel<real><<<(k + 63) / 64, 64, 0, st>>>(M, nrow, k, ldf, fin, out);
        LAUNCHED();
    } else {
        const int threads = 256;
        if (ldf > threads) return fail("k too large for the column-sum kernel");
        const int rpb = threads / ldf;
        int grid = (int)std::min<size_t>((size_t)n_partial, (nrow + rpb - 1) / rpb);
        grid = std::max(grid, 1);
        colsum_partial_kernel<real><<<grid, threads, threads * sizeof(real), st>>>(M, nrow, ldf, partial);
        LAUNCHED();
        colsum_fold_kernel<real><<<(k + 63) / 64, 64, 0, st>>>(partial, grid, k, ldf, fin, out);
        LAUNCHED();
    }
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail("column sums: %s", cudaGetErrorString(e));
    return 0;
}

// ---------------------------------------------------------------------------
// one orientation (CSR or CSC) of the count matrix on the device + its row plan
// ---------------------------------------------------------------------------
struct Bin : PlannedBin {
    int* d_rows = nullptr;         // device copy of `rows`
    Timings timings;
};

template <class real> struct Side {
    LockstepPlan lockstep;         // the heaviest rows (lockstep.h)
    real* xv = nullptr;
    long long* ptr = nullptr;
    int* ind = nullptr;
    size_t nnz = 0, row_begin = 0, n_rows = 0;
    std::vector<long long> h_ptr;
    std::vector<Bin> bins;
    int planned_method = -1;
    int* d_empty = nullptr;
    int n_empty = 0;
    int* d_all_rows = nullptr;
    real* gscratch = nullptr;
    long long gs_stride = 0;
    int gs_ctas = 0;
    // callers synchronise the streams that used these buffers first (devpool.h)
    void free_plan()
    {
        for (auto& b : bins) b.timings.clear();
        lockstep.release();
        if (d_all_rows) dfree(d_all_rows);
        if (gscratch) dfree(gscratch);
        d_all_rows = nullptr; gscratch = nullptr; d_empty = nullptr;
        bins.clear(); planned_method = -1;
    }
    void free_all()
    {
        free_plan();
        if (xv) dfree(xv);
        if (ptr) dfree(ptr);
        if (ind) dfree(ind);
        xv = nullptr; ptr = nullptr; ind = nullptr;
    }
};

struct pmf_b200_handle {
    int dtype = 0, device = 0;
    size_t dimA = 0, dimB = 0;
    int k = 0, kp = 0, ldf = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    bool have_stream = false;   // `stream` is valid (the legacy default stream is the null handle: never test the value)
    int num_sms = 148;
    virtual ~pmf_b200_handle() {}
    virtual int set_matrix(int side, const void* values, const void* indptr, const void* indices, size_t nnz,
                           int index_bytes, size_t row_begin, size_t n_rows) = 0;
    virtual int set_factors(const void* A, const void* B) = 0;
    virtual int get_factors(void* A, void* B) = 0;
    virtual int bind_factors(void* A, void* B) = 0;
    virtual int set_factor_rows(int which, const void* host, size_t row_begin, size_t n_rows) = 0;
    virtual void* factor_ptr(int which) = 0;
    virtual int half_sweep(int side, const pmf_b200_params& p, double step, double cdiv,
                           unsigned long long* n_unchanged) = 0;
    virtual int sweeps(const pmf_b200_params& p) = 0;
    virtual int run_dropin(void* A, void* B, const void* Xr, const void* Xr_indptr, const void* Xr_indices, size_t nnz_r,
                           const void* Xc, const void* Xc_indptr, const void* Xc_indices, size_t nnz_c, int index_bytes,
                           const pmf_b200_params& p, const std::function<void(const char*)>& lap, bool timing,
                           bool matrix_resident) = 0;
    virtual int factors_multiple(void* A_out, const void* Bsum, const void* Amean, const pmf_b200_params& p,
                                 int reuse_mean) = 0;
    virtual int ingest_coo(const void* rows, const void* cols, const void* vals, size_t n, int index_bytes) = 0;
    virtual int export_matrix(int side, void* values, void* indptr, void* indices, int index_bytes) = 0;
    virtual size_t side_nnz(int side) const = 0;
    virtual int ipc_export(int which, void* out) = 0;
    virtual int ipc_import(int which, const void* handles, int n_ranks, int self_rank) = 0;
    virtual int exchange_status() = 0;
    virtual bool has_peers() const = 0;        // peer replicas or epoch slots imported: part of a sharded fit
    virtual int get_profile(pmf_b200_bin_profile* out, int max_entries) = 0;
    virtual void clear_profile() = 0;
    bool profiling = false;
};

template <class real> struct HandleT : pmf_b200_handle {
    real *A = nullptr, *B = nullptr;
    bool ownA = false, ownB = false;
    Side<real> sides[2];
    real* csum = nullptr;       // k
    real* partial = nullptr;    // colsum partials
    int n_partial = 0;
    int* counters = nullptr;    // one per bin
    unsigned long long* d_unchanged = nullptr;
    // bins of one half-sweep are independent: they are launched on a few side streams so that
    // small or latency-bound bins overlap (fork from / join to the handle's stream with events)
    real* peer[2][7] = {};      // peers' replicas of A (0) and B (1), opened through CUDA IPC
    int npeers[2] = {0, 0};
    // device-side completion of the exchange: own epoch slots (raw cudaMalloc: exported), the ranks' slot arrays
    unsigned long long* sig = nullptr;
    int* sig_status = nullptr;
    PeerSignals sigs = {};
    void* sig_opened[7] = {};
    int n_sig_opened = 0;
    unsigned long long epoch = 0;
    bool exported[2] = {false, false};   // A / B handed to other processes: never recycled through the block cache
    static constexpr int NAUX = 6;
    cudaStream_t aux[NAUX] = {};
    cudaEvent_t ev_fork = nullptr, ev_join[NAUX] = {};
    // the stateless drop-in calls pipeline their transfers against the half-sweeps on this stream
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_copy = nullptr, ev_main = nullptr;
    std::vector<void*> deferred;   // staging buffers, released at the next synchronisation point
    static constexpr int V = RealTraits<real>::V;

    ~HandleT() override
    {
        cudaSetDevice(device);
        sync_all();
        sides[0].free_all(); sides[1].free_all();
        for (int w = 0; w < 2; w++)
            for (int q = 0; q < npeers[w]; q++) cudaIpcCloseMemHandle(peer[w][q]);
        for (int q = 0; q < n_sig_opened; q++) cudaIpcCloseMemHandle(sig_opened[q]);
        if (sig) cudaFree(sig);
        if (sig_status) cudaFree(sig_status);
        if (ownA && A) { if (exported[0]) DevPool::get().discard(A); else dfree(A); }
        if (ownB && B) { if (exported[1]) DevPool::get().discard(B); else dfree(B); }
        if (csum) dfree(csum);
        if (partial) dfree(partial);
        if (counters) dfree(counters);
        if (d_unchanged) dfree(d_unchanged);
        for (int i = 0; i < NAUX; i++) {
            if (aux[i]) cudaStreamDestroy(aux[i]);
            if (ev_join[i]) cudaEventDestroy(ev_join[i]);
        }
        if (ev_fork) cudaEventDestroy(ev_fork);
        if (ev_copy) cudaEventDestroy(ev_copy);
        if (ev_main) cudaEventDestroy(ev_main);
        if (copy_stream) cudaStreamDestroy(copy_stream);
        if (own_stream && stream) cudaStreamDestroy(stream);
    }

    // wait for everything this handle has enqueued, then release the staging buffers
    int sync_all()
    {
        cudaError_t e1 = have_stream ? cudaStreamSynchronize(stream) : cudaSuccess;
        cudaError_t e2 = copy_stream ? cudaStreamSynchronize(copy_stream) : cudaSuccess;
        for (void* q : deferred) dfree(q);
        deferred.clear();
        if (e1 != cudaSuccess) return fail("stream synchronize failed: %s", cudaGetErrorString(e1));
        if (e2 != cudaSuccess) return fail("stream synchronize failed: %s", cudaGetErrorString(e2));
        return 0;
    }

    // B_dev: bind this device matrix [dimB x ldf] as B instead of allocating one (a fold-in against resident factors)
    int init(real* B_dev = nullptr)
    {
        CK(cudaSetDevice(device));
        CK(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, device));
        ldf = round_up(k, V);
        kp = tile_stride(k, V);
        CK(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
        own_stream = true; have_stream = true;
        CK(dmalloc(&A, dimA * (size_t)ldf * sizeof(real)));
        ownA = true;
        CK(cudaMemsetAsync(A, 0, dimA * (size_t)ldf * sizeof(real), stream));
        if (B_dev) {
            B = B_dev;
        } else {
            CK(dmalloc(&B, dimB * (size_t)ldf * sizeof(real)));
            ownB = true;
            CK(cudaMemsetAsync(B, 0, dimB * (size_t)ldf * sizeof(real), stream));
        }
        CK(dmalloc(&csum, (size_t)kp * sizeof(real)));
        n_partial = num_sms * 4;
        CK(dmalloc(&partial, (size_t)n_partial * ldf * sizeof(real)));
        CK(dmalloc(&counters, 64 * sizeof(int)));   // one per bin (<= 12 + 3 + 5)
        CK(dmalloc(&d_unchanged, sizeof(unsigned long long)));
        for (int i = 0; i < NAUX; i++) {
            CK(cudaStreamCreateWithFlags(&aux[i], cudaStreamNonBlocking));
            CK(cudaEventCreateWithFlags(&ev_join[i], cudaEventDisableTiming));
        }
        CK(cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming));
        CK(cudaStreamCreateWithFlags(&copy_stream, cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&ev_copy, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&ev_main, cudaEventDisableTiming));
        return 0;
    }

    // enqueue the upload of one orientation on `st`; temporaries go to `deferred`
    template <class IX>
    int upload_side(Side<real>& S, const real* values, const IX* indptr, const IX* indices, size_t nnz, size_t n_rows,
                    cudaStream_t st)
    {
        S.h_ptr.resize(n_rows + 1);
        const long long base = (long long)indptr[0];
        for (size_t i = 0; i <= n_rows; i++) S.h_ptr[i] = (long long)indptr[i] - base;
        if ((size_t)S.h_ptr[n_rows] != nnz) return fail("set_matrix: indptr[n_rows]-indptr[0] != nnz");
        CK(dmalloc(&S.xv, std::max<size_t>(nnz, 1) * sizeof(real)));
        CK(dmalloc(&S.ind, std::max<size_t>(nnz, 1) * sizeof(int)));
        CK(dmalloc(&S.ptr, (n_rows + 1) * sizeof(long long)));
        CK(Stager::get().h2d(S.xv, values, nnz * sizeof(real), st));
        CK(cudaMemcpyAsync(S.ptr, S.h_ptr.data(), (n_rows + 1) * sizeof(long long), cudaMemcpyHostToDevice, st));
        // indices: upload at host width, narrow to int32 on the device
        if (sizeof(IX) == sizeof(int)) {
            CK(Stager::get().h2d(S.ind, indices, nnz * sizeof(int), st));
        } else {
            IX* tmp = nullptr;
            const size_t chunk = (size_t)1 << 27;   // bounded staging buffer (1 GiB of 8-byte ids)
            CK(dmalloc(&tmp, std::min(chunk, std::max<size_t>(nnz, 1)) * sizeof(IX)));
            deferred.push_back(tmp);
            for (size_t off = 0; off < nnz; off += chunk) {
                const size_t m = std::min(chunk, nnz - off);
                CK(Stager::get().h2d(tmp, indices + off, m * sizeof(IX), st));
                narrow_indices_kernel<IX><<<num_sms * 8, 256, 0, st>>>(tmp, S.ind + off, m);
                LAUNCHED();
                CK(cudaGetLastError());
            }
        }
        return 0;
    }
    int upload_matrix(int side, const void* values, const void* indptr, const void* indices, size_t nnz,
                      int index_bytes, size_t row_begin, size_t n_rows, cudaStream_t st)
    {
        if (side != 0 && side != 1) return fail("set_matrix: bad side");
        const size_t dim = side == PMF_SIDE_CSR ? dimA : dimB;
        if (row_begin + n_rows > dim) return fail("set_matrix: row range exceeds the dimension");
        Side<real>& S = sides[side];
        S.free_all();
        S.nnz = nnz; S.row_begin = row_begin; S.n_rows = n_rows;
        if (index_bytes == 8)
            return upload_side<uint64_t>(S, (const real*)values, (const uint64_t*)indptr, (const uint64_t*)indices, nnz, n_rows, st);
        if (index_bytes == 4)
            return upload_side<int>(S, (const real*)values, (const int*)indptr, (const int*)indices, nnz, n_rows, st);
        return fail("set_matrix: index_bytes must be 4 or 8");
    }

    int set_matrix(int side, const void* values, const void* indptr, const void* indices, size_t nnz,
                   int index_bytes, size_t row_begin, size_t n_rows) override
    {
        CK(cudaSetDevice(device));
        if (sync_all()) return 1;       // the side's old buffers may still be in use
        const int rc = upload_matrix(side, values, indptr, indices, nnz, index_bytes, row_begin, n_rows, stream);
        return sync_all() || rc;
    }

    // dense host rows are k reals, device rows ldf reals: one contiguous copy + a device repack
    // (a pitched cudaMemcpy2D of 200-byte rows is ~10x slower over PCIe)
    int copy_in(real* dev, const void* host, size_t n, cudaStream_t st)
    {
        if (ldf == k) { CK(Stager::get().h2d(dev, host, n * (size_t)k * sizeof(real), st)); return 0; }
        real* tmp = nullptr;
        CK(dmalloc(&tmp, std::max<size_t>(n * (size_t)k, 1) * sizeof(real)));
        deferred.push_back(tmp);
        CK(Stager::get().h2d(tmp, host, n * (size_t)k * sizeof(real), st));
        pad_rows_kernel<real><<<num_sms * 8, 256, 0, st>>>(tmp, dev, n, k, ldf);
        LAUNCHED();
        CK(cudaGetLastError());
        return 0;
    }
    int copy_out(void* host, const real* dev, size_t n, cudaStream_t st)
    {
        if (ldf == k) { CK(Stager::get().d2h(host, dev, n * (size_t)k * sizeof(real), st)); return 0; }
        real* tmp = nullptr;
        CK(dmalloc(&tmp, std::max<size_t>(n * (size_t)k, 1) * sizeof(real)));
        deferred.push_back(tmp);
        unpad_rows_kernel<real><<<num_sms * 8, 256, 0, st>>>(dev, tmp, n, k, ldf);
        LAUNCHED();
        CK(cudaGetLastError());
        CK(Stager::get().d2h(host, tmp, n * (size_t)k * sizeof(real), st));
        return 0;
    }
    int set_factors(const void* Ah, const void* Bh) override
    {
        CK(cudaSetDevice(device));
        int rc = 0;
        if (Ah) rc = copy_in(A, Ah, dimA, stream);
        if (Bh && !rc) rc = copy_in(B, Bh, dimB, stream);
        return sync_all() || rc;
    }
    // rows [row_begin, row_begin + n_rows) of A (which = 0) or B (1) from host memory into the own replica AND,
    // over NVLink, into every peer's: a sharded fit uploads each factor row once per box instead of once per GPU
    int set_factor_rows(int which, const void* host, size_t row_begin, size_t n_rows) override
    {
        CK(cudaSetDevice(device));
        if (which != 0 && which != 1) return fail("set_factor_rows: which must be 0 (A) or 1 (B)");
        const size_t dim = which == 0 ? dimA : dimB;
        if (row_begin + n_rows > dim) return fail("set_factor_rows: row range exceeds the dimension");
        real* M = (which == 0 ? A : B) + row_begin * (size_t)ldf;
        int rc = n_rows ? copy_in(M, host, n_rows, stream) : 0;
        for (int q = 0; q < npeers[which] && !rc && n_rows; q++)
            CK(cudaMemcpyAsync(peer[which][q] + row_begin * (size_t)ldf, M, n_rows * (size_t)ldf * sizeof(real),
                               cudaMemcpyDeviceToDevice, stream));
        return sync_all() || rc;
    }
    int get_factors(void* Ah, void* Bh) override
    {
        CK(cudaSetDevice(device));
        int rc = 0;
        if (Ah) rc = copy_out(Ah, A, dimA, stream);
        if (Bh && !rc) rc = copy_out(Bh, B, dimB, stream);
        return sync_all() || rc;
    }
    int bind_factors(void* Ad, void* Bd) override
    {
        CK(cudaSetDevice(device));
        if (sync_all()) return 1;
        if (Ad) { if (ownA && A) { if (exported[0]) DevPool::get().discard(A); else dfree(A); } A = (real*)Ad; ownA = false; }
        if (Bd) { if (ownB && B) { if (exported[1]) DevPool::get().discard(B); else dfree(B); } B = (real*)Bd; ownB = false; }
        return 0;
    }
    void* factor_ptr(int which) override { return which == 0 ? (void*)A : (void*)B; }

    // the planner's inputs for the parameters of a half-sweep (row_plan.h)
    PlanMode plan_mode(const pmf_b200_params& p) const
    {
        PlanMode m;
        m.real_size = sizeof(real); m.ldf = ldf; m.kp = kp;
        m.method = p.method;
        m.strict = (p.flags & PMF_FLAG_STRICT) != 0;
        // register-tile kernels (regtile.cuh) take the rows of up to 512 non-zeros when the fit is float32 in
        // fast numerics with w_mult == 1 and k <= 64: pg, and cg with limit_step and the cached line search
        m.regtile = std::is_same<real, float>::value && !m.strict && (real)p.w_mult == (real)1 && ldf <= 64 &&
                    (p.method == PMF_PG || (p.method == PMF_CG && p.limit_step && !(p.flags & PMF_FLAG_NO_CACHED)));
        m.lockstep = !(p.flags & PMF_FLAG_NO_LOCKSTEP);
        if (const char* e = getenv("POISMF_B200_DENSE_MIN")) m.dense_min = std::max(1LL, atoll(e));
        if (const char* e = getenv("POISMF_B200_DENSE_MIN_TOTAL")) m.dense_min_total = atoll(e);
        return m;
    }
    // row lists are uploaded on `st`; kernels that read them must be ordered after it
    int plan(Side<real>& S, const pmf_b200_params& p, cudaStream_t st)
    {
        const PlanMode m = plan_mode(p);
        const int key = m.method * 8 + (m.strict ? 1 : 0) + (m.regtile ? 2 : 0) + (m.lockstep ? 0 : 4);
        if (S.planned_method == key) return 0;
        if (S.planned_method >= 0) {    // re-planning for another method: the old lists may be in use
            if (sync_all()) return 1;
            S.free_plan();
        }
        if (build_plan(S, m, st)) {     // release what a part-way plan holds
            sync_all();
            S.free_plan();
            return 1;
        }
        S.planned_method = key;
        return 0;
    }
    int build_plan(Side<real>& S, const PlanMode& m, cudaStream_t st)
    {
        const size_t other = (&S == &sides[0]) ? dimB : dimA;
        RowPlan rp = plan_rows(m, S.h_ptr.data(), S.n_rows, other);
        if (!rp.lockstep.empty()) {
            const cudaError_t e = S.lockstep.build(rp.lockstep, S.h_ptr.data(), S.ind, (const float*)S.xv, other, k, ldf,
                                                   num_sms, deferred, st, g_launches);
            if (e != cudaSuccess) return fail("lock-step plan: %s", cudaGetErrorString(e));
        }
        size_t total = rp.empty.size();
        for (auto& b : rp.bins) total += b.rows.size();
        CK(dmalloc(&S.d_all_rows, std::max<size_t>(total, 1) * sizeof(int)));
        size_t off = 0;
        std::vector<Bin> bins;
        for (auto& pb : rp.bins) {
            Bin b{std::move(pb)};
            b.d_rows = S.d_all_rows + off;
            if (!b.rows.empty())
                CK(cudaMemcpyAsync(b.d_rows, b.rows.data(), b.rows.size() * sizeof(int), cudaMemcpyHostToDevice, st));
            off += b.rows.size();
            bins.push_back(std::move(b));
        }
        S.d_empty = S.d_all_rows + off;
        S.n_empty = (int)rp.empty.size();
        if (S.n_empty)
            CK(cudaMemcpyAsync(S.d_empty, rp.empty.data(), rp.empty.size() * sizeof(int), cudaMemcpyHostToDevice, st));
        const Bin& gb = bins.back();
        if (!gb.rows.empty()) {
            // per-CTA scratch for the three per-non-zero arrays of rows that are not staged
            const long long per_cta = (gb.max_nnz + gb.shape.cluster - 1) / gb.shape.cluster;
            S.gs_stride = (long long)round_up_sz((size_t)per_cta + 4, 4);
            // streaming clusters are compiled for two CTAs per SM: scratch for 2 x SMs CTAs
            S.gs_ctas = gb.shape.cluster > 1 ? 2 * num_sms
                                             : (int)std::min<size_t>(gb.rows.size(), (size_t)num_sms);
            CK(dmalloc(&S.gscratch, (size_t)S.gs_ctas * 3 * S.gs_stride * sizeof(real)));
        }
        S.bins.swap(bins);      // the row lists' host copies stay alive in S.bins until the next plan
        return 0;
    }

    // ---- column sums of the fixed factor matrix -------------------------------
    int column_sums(const real* F, size_t nrow, const ColsumFinal<real>& fin, bool strict)
    {
        return launch_column_sums(F, nrow, k, ldf, fin, strict, partial, n_partial, csum, stream);
    }

    // ---- one half-sweep ----------------------------------------------------------
    // side CSC: update local rows of B with A fixed (src/poismf.c:510-557)
    // side CSR: update local rows of A with B fixed (:561-604)
    int half_sweep(int side, const pmf_b200_params& p, double step_d, double cdiv_d,
                   unsigned long long* n_unchanged) override
    {
        return half_sweep_ex(side, p, step_d, cdiv_d, n_unchanged, nullptr, (real)1, -1);
    }
    // csum_host != nullptr: use these k column sums (already +l1 and, for pg, pre-scaled) instead of
    // summing the fixed matrix; maxupd_override >= 0 replaces p.maxupd (factors_multiple's cg)
    int half_sweep_ex(int side, const pmf_b200_params& p, double step_d, double cdiv_d,
                      unsigned long long* n_unchanged, const real* csum_host, real pre_scale,
                      long long maxupd_override)
    {
        CK(cudaSetDevice(device));
        struct NvtxScope { NvtxScope(const char* n) { nvtxRangePushA(n); } ~NvtxScope() { nvtxRangePop(); } };
        NvtxScope nvtx_hs(side == PMF_SIDE_CSR ? "poismf half-sweep A (CSR)" : "poismf half-sweep B (CSC)");
        Side<real>& S = sides[side];
        if (!S.ptr) return fail("half_sweep: matrix for side %d not set", side);
        if (p.method != PMF_PG && p.method != PMF_CG && p.method != PMF_TNCG) return fail("bad method");
        const bool strict = (p.flags & PMF_FLAG_STRICT) != 0;
        if (plan(S, p, stream)) return 1;
        const bool updA = side == PMF_SIDE_CSR;
        real* M = updA ? A : B;
        const real* F = updA ? B : A;
        const size_t other = updA ? dimB : dimA;

        const real l2 = (real)p.l2_reg, l1 = (real)p.l1_reg, w = (real)p.w_mult, step = (real)step_d;
        HalfSweepConsts<real> hc;
        hc.l2 = l2;
        hc.two_l2 = (real)(2. * (double)l2);
        hc.w = w;
        hc.wm1 = (real)((double)w - 1.);
        hc.step_w = step * w;
        hc.neg_step = -step;
        hc.cdiv = (real)cdiv_d;
        {   // (double)v >= 1e-15  <=>  v >= clip_thr  for every finite `real` v
            real c = (real)1e-15;
            if ((double)c < 1e-15) c = std::nextafter(c, (real)1);
            hc.clip_thr = c;
        }
        hc.maxupd = (int)std::min<size_t>(maxupd_override >= 0 ? (size_t)maxupd_override : p.maxupd, (size_t)INT32_MAX);
        hc.pre_scale = pre_scale;
        hc.limit_step = p.limit_step; hc.reuse_prev = p.reuse_prev;
        hc.early_stop = (p.method == PMF_TNCG && p.early_stop) ? 1 : 0;
        hc.method = p.method;

        // sharded fit with device-side completion: every rank's previous half-sweep must have landed
        if (sigs.n_ranks > 1 && epoch > 0) {
            wait_epoch_kernel<<<1, 32, 0, stream>>>(sig, sigs.n_ranks, epoch, sig_status);
            LAUNCHED();
        }
        ColsumFinal<real> fin;
        fin.l1 = l1; fin.scale1 = -step; fin.scale2 = -step; fin.nscale = 0;
        if (p.method == PMF_PG && w == (real)1) fin.nscale = updA ? 2 : 1;   // Q1: A side scaled twice
        if (csum_host) CK(cudaMemcpyAsync(csum, csum_host, (size_t)k * sizeof(real), cudaMemcpyHostToDevice, stream));
        else if (column_sums(F, other, fin, strict)) return 1;

        if (S.n_empty > 0) {
            const size_t total = (size_t)S.n_empty * ldf;
            const int grid = (int)std::min<size_t>((total + 255) / 256, (size_t)num_sms * 8);
            const int wm0 = updA ? 0 : 1;
            for (int q = -1; q < npeers[wm0]; q++) {      // own replica, then every peer's (fused exchange)
                real* base = (q < 0 ? M : peer[wm0][q]) + S.row_begin * (size_t)ldf;
                zero_rows_kernel<real><<<grid, 256, 0, stream>>>(base, S.d_empty, S.n_empty, ldf);
                LAUNCHED();
            }
        }
        CK(cudaMemsetAsync(counters, 0, 64 * sizeof(int), stream));
        if (hc.early_stop) CK(cudaMemsetAsync(d_unchanged, 0, sizeof(unsigned long long), stream));

        const bool overlap = !profiling;      // profiled bins run one after another, each timed on its own
        if (overlap) CK(cudaEventRecord(ev_fork, stream));
        int n_launched = 0;
        bool used[NAUX] = {};
        if (S.lockstep.rows() > 0) {                              // the heaviest rows: lock-step path, own stream
            cudaStream_t ls = stream;
            if (overlap) { ls = aux[0]; CK(cudaStreamWaitEvent(ls, ev_fork, 0)); used[0] = true; n_launched = 1; }
            if (profiling) CK(S.lockstep.timings.start(stream));
            cudaError_t e = cudaErrorInvalidValue;   // float32 only (row_plan.h)
            nvtxRangePushA("lock-step rows");
            if constexpr (std::is_same<real, float>::value)
                e = S.lockstep.run(M, peer[updA ? 0 : 1], npeers[updA ? 0 : 1], S.row_begin, F, csum, hc, ls, g_launches);
            nvtxRangePop();
            if (e != cudaSuccess) return fail("lock-step rows of side %d: %s", side, cudaGetErrorString(e));
            if (profiling) CK(S.lockstep.timings.stop(stream));
        }
        for (int bi = (int)S.bins.size() - 1; bi >= 0; bi--) {    // heaviest rows first
            const Bin& bin = S.bins[bi];
            const BinShape& b = bin.shape;
            if (bin.rows.empty()) continue;
            cudaStream_t ls = stream;
            if (overlap) {
                // (the lock-step chain keeps aux[0] to itself: a bin queued behind it would start when it ends)
                const int si = S.lockstep.rows() > 0 ? 1 + (n_launched - 1) % (NAUX - 1) : n_launched % NAUX;
                ls = aux[si];
                if (!used[si]) { CK(cudaStreamWaitEvent(ls, ev_fork, 0)); used[si] = true; }
            }
            n_launched++;
            SideParams<real> P;
            P.M = M + S.row_begin * (size_t)ldf;
            P.F = F; P.xv = S.xv; P.ptr = S.ptr; P.ind = S.ind; P.csum = csum;
            P.rows = bin.d_rows; P.nrows = (int)bin.rows.size();
            P.counter = counters + bi;
            P.k = k; P.kp = kp; P.ldf = ldf; P.cap = b.cap; P.slice_bytes = (int)b.slice;
            P.acap = b.acap;
            P.hc = hc;
            P.gscratch = b.cap == 0 ? S.gscratch : nullptr;   // rows beyond acap per CTA fall back to global arrays
            P.gs_stride = S.gs_stride;
            P.n_unchanged = d_unchanged;
            const int wm = updA ? 0 : 1;
            P.npeers = npeers[wm];
            for (int q = 0; q < 7; q++) P.peerM[q] = q < npeers[wm] ? peer[wm][q] + S.row_begin * (size_t)ldf : nullptr;
            LaunchArgs la;
            la.stream = ls;
            const int teams = b.kind == BinKind::Warp ? b.threads / b.lanes : 1;
            la.needed = (P.nrows + teams - 1) / teams;
            la.max_grid = b.cap == 0 ? S.gs_ctas / b.cluster : (1 << 30);
            la.num_sms = num_sms;
            la.cached = !strict && !(p.flags & PMF_FLAG_NO_CACHED);
            if (profiling) CK(S.bins[bi].timings.start(stream));
            static const char* const kind_name[] = {"regtile", "warp", "cta", "cluster", "streaming"};
            {
                char nm[96];
                snprintf(nm, sizeof nm, "bin %s cap %d rows %d", kind_name[(int)b.kind], b.cap, P.nrows);
                nvtxRangePushA(nm);
            }
            cudaError_t e = cudaErrorInvalidConfiguration;
            switch (b.kind) {
            case BinKind::RegTile:
                if constexpr (std::is_same<real, float>::value)
                    e = p.method == PMF_PG ? launch_regtile_pg(b, la, P) : launch_regtile_cg(b, la, P);
                break;
            case BinKind::Cluster:
            case BinKind::Streaming:
                e = p.method == PMF_TNCG ? launch_gang_tn_fast<real>(b, la, P) : launch_gang_pgcg_fast<real>(b, la, P);
                break;
            case BinKind::Warp:
            case BinKind::Cta:
                if (p.method == PMF_TNCG)
                    e = strict ? launch_rows_tn_strict<real>(b, la, P) : launch_rows_tn_fast<real>(b, la, P);
                else
                    e = strict ? launch_rows_pgcg_strict<real>(b, la, P) : launch_rows_pgcg_fast<real>(b, la, P);
                break;
            }
            LAUNCHED();
            nvtxRangePop();
            if (e != cudaSuccess)
                return fail("row kernel launch failed at side %d bin %d (%s, lanes %d cluster %d cap %d threads %d smem %zu): %s",
                            side, bi, kind_name[(int)b.kind], b.lanes, b.cluster, b.cap, b.threads, b.smem,
                            cudaGetErrorString(e));
            if (profiling) CK(S.bins[bi].timings.stop(stream));
        }
        if (overlap)
            for (int si = 0; si < NAUX; si++)
                if (used[si]) {
                    CK(cudaEventRecord(ev_join[si], aux[si]));
                    CK(cudaStreamWaitEvent(stream, ev_join[si], 0));
                }
        if (sigs.n_ranks > 1) {
            epoch++;
            signal_epoch_kernel<<<1, 1, 0, stream>>>(sigs, epoch);
            LAUNCHED();
        }
        if (hc.early_stop && n_unchanged) {
            CK(cudaMemcpyAsync(n_unchanged, d_unchanged, sizeof(unsigned long long), cudaMemcpyDeviceToHost, stream));
            CK(cudaStreamSynchronize(stream));
        }
        return 0;
    }
    // 1 if a peer failed to arrive at an exchange point (the fit's results are then invalid)
    int exchange_status() override
    {
        if (!sig_status) return 0;
        int v = 0;
        cudaMemcpy(&v, sig_status, sizeof v, cudaMemcpyDeviceToHost);
        return v;
    }
    bool has_peers() const override { return npeers[0] || npeers[1] || n_sig_opened; }

    int ipc_export(int which, void* out) override
    {
        CK(cudaSetDevice(device));
        if (which == 2) {          // the epoch slots of the device-side exchange completion
            if (!sig) {
                CK(cudaMalloc(&sig, 8 * sizeof(unsigned long long)));
                CK(cudaMemset(sig, 0, 8 * sizeof(unsigned long long)));
                CK(cudaMalloc(&sig_status, sizeof(int)));
                CK(cudaMemset(sig_status, 0, sizeof(int)));
            }
            cudaIpcMemHandle_t hd;
            CK(cudaIpcGetMemHandle(&hd, (void*)sig));
            memcpy(out, &hd, sizeof hd);
            return 0;
        }
        if ((which == 0 && !ownA) || (which == 1 && !ownB))
            return fail("ipc_export: factors are bound to caller memory; export needs handle-owned buffers");
        cudaIpcMemHandle_t hd;
        CK(cudaIpcGetMemHandle(&hd, which == 0 ? (void*)A : (void*)B));
        exported[which] = true;
        static_assert(sizeof(hd) == PMF_B200_IPC_HANDLE_BYTES, "IPC handle size");
        memcpy(out, &hd, sizeof hd);
        return 0;
    }
    int ipc_import(int which, const void* handles, int n_ranks, int self_rank) override
    {
        CK(cudaSetDevice(device));
        if (n_ranks < 1 || n_ranks > 8) return fail("ipc_import: 1..8 ranks");
        if (which == 2) {
            if (!sig) return fail("ipc_import: export the epoch slots first");
            for (int q = 0; q < n_sig_opened; q++) cudaIpcCloseMemHandle(sig_opened[q]);
            n_sig_opened = 0;
            sigs.n_ranks = n_ranks; sigs.self = self_rank;
            for (int r = 0; r < n_ranks; r++) {
                if (r == self_rank) { sigs.slot[r] = sig; continue; }
                cudaIpcMemHandle_t hd;
                memcpy(&hd, (const char*)handles + (size_t)r * sizeof hd, sizeof hd);
                void* ptr = nullptr;
                CK(cudaIpcOpenMemHandle(&ptr, hd, cudaIpcMemLazyEnablePeerAccess));
                sig_opened[n_sig_opened++] = ptr;
                sigs.slot[r] = (unsigned long long*)ptr;
            }
            return 0;
        }
        for (int q = 0; q < npeers[which]; q++) cudaIpcCloseMemHandle(peer[which][q]);
        npeers[which] = 0;
        for (int r = 0; r < n_ranks; r++) {
            if (r == self_rank) continue;
            cudaIpcMemHandle_t hd;
            memcpy(&hd, (const char*)handles + (size_t)r * sizeof hd, sizeof hd);
            void* ptr = nullptr;
            CK(cudaIpcOpenMemHandle(&ptr, hd, cudaIpcMemLazyEnablePeerAccess));
            peer[which][npeers[which]++] = (real*)ptr;
        }
        return 0;
    }

    void clear_profile() override
    {
        for (Side<real>& S : sides) {
            S.lockstep.timings.clear();
            for (Bin& b : S.bins) b.timings.clear();
        }
    }
    // the lock-step path of side 0, then of side 1, then the bins of side 0 and of side 1
    int get_profile(pmf_b200_bin_profile* out, int max_entries) override
    {
        cudaSetDevice(device);
        cudaStreamSynchronize(stream);
        int n = 0;
        auto put = [&](int sd, int code, int cap, int nrows, unsigned long long nnz, const Timings& t) {
            if (n >= max_entries) return;
            pmf_b200_bin_profile& o = out[n++];
            o.side = sd; o.block_team = code; o.cap = cap; o.nrows = nrows; o.nnz = nnz;
            o.launches = t.launches(); o.ms = t.ms();
        };
        for (int sd = 0; sd < 2; sd++) {
            const LockstepPlan& L = sides[sd].lockstep;
            if (L.rows() > 0) put(sd, LOCKSTEP_PROFILE_CODE, 0, L.rows(), L.nnz(), L.timings);
        }
        for (int sd = 0; sd < 2; sd++)
            for (const Bin& b : sides[sd].bins)
                if (!b.rows.empty()) put(sd, profile_code(b.shape), b.shape.cap, (int)b.rows.size(), b.nnz, b.timings);
        return n;
    }

    // ---- COO triplets -> both orientations, built on the device (ingest.cuh) ---------------------
    // What coo.tocsr() / coo.tocsc() give the reference (poismf/__init__.py:402-404): duplicates
    // summed, ids ascending within each row / column.
    size_t side_nnz(int side) const override { return sides[side].nnz; }
    template <class IX>
    int ingest_impl(const IX* rows, const IX* cols, const real* vals, size_t n)
    {
        typedef unsigned long long u64;
        if (n == 0) return fail("fit_coo: no entries");
        if (n > (size_t)INT32_MAX) return fail("fit_coo: more than 2^31-1 triplets; build CSR/CSC in parts");
        if (sync_all()) return 1;
        sides[0].free_all(); sides[1].free_all();
        IX *d_r = nullptr, *d_c = nullptr;
        real *v1 = nullptr, *v2 = nullptr;
        u64 *k1 = nullptr, *k2 = nullptr;
        int *d_flags = nullptr;        // [0] bad-id flag, [1] number of unique entries
        void* tmp = nullptr;
        auto defer = [&](void* q) { deferred.push_back(q); };
        CK(dmalloc(&d_r, n * sizeof(IX))); defer(d_r);
        CK(dmalloc(&d_c, n * sizeof(IX))); defer(d_c);
        CK(dmalloc(&v1, n * sizeof(real))); defer(v1);
        CK(dmalloc(&v2, n * sizeof(real))); defer(v2);
        CK(dmalloc(&k1, n * sizeof(u64))); defer(k1);
        CK(dmalloc(&k2, n * sizeof(u64))); defer(k2);
        CK(dmalloc(&d_flags, 2 * sizeof(int))); defer(d_flags);
        CK(cudaMemsetAsync(d_flags, 0, 2 * sizeof(int), stream));
        CK(Stager::get().h2d(d_r, rows, n * sizeof(IX), stream));
        CK(Stager::get().h2d(d_c, cols, n * sizeof(IX), stream));
        CK(Stager::get().h2d(v1, vals, n * sizeof(real), stream));
        const int grid = num_sms * 8;
        coo_keys_kernel<IX><<<grid, 256, 0, stream>>>(d_r, d_c, n, (u64)dimA, (u64)dimB, k1, d_flags);
        LAUNCHED();
        auto bits = [](size_t dim) { int b = 1; while (b < 32 && ((size_t)1 << b) < dim) b++; return b; };
        size_t b_sort1 = 0, b_red = 0, b_sort2 = 0;
        CK(cub::DeviceRadixSort::SortPairs(nullptr, b_sort1, k1, k2, v1, v2, (int)n, 0, 32 + bits(dimA), stream));
        CK(cub::DeviceReduce::ReduceByKey(nullptr, b_red, k2, k1, v2, v1, d_flags + 1, cub::Sum(), (int)n, stream));
        CK(cub::DeviceRadixSort::SortPairs(nullptr, b_sort2, k2, k1, v1, v2, (int)n, 0, 32 + bits(dimB), stream));
        const size_t tmp_bytes = std::max(std::max(b_sort1, b_red), std::max<size_t>(b_sort2, 16));
        CK(dmalloc(&tmp, tmp_bytes)); defer(tmp);
        size_t tb = tmp_bytes;
        // (row, col)-sorted, stable: duplicates stay in input order
        CK(cub::DeviceRadixSort::SortPairs(tmp, tb, k1, k2, v1, v2, (int)n, 0, 32 + bits(dimA), stream));
        LAUNCHED();
        tb = tmp_bytes;
        CK(cub::DeviceReduce::ReduceByKey(tmp, tb, k2, k1, v2, v1, d_flags + 1, cub::Sum(), (int)n, stream));
        LAUNCHED();
        int h_flags[2] = {0, 0};
        CK(cudaMemcpyAsync(h_flags, d_flags, sizeof h_flags, cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
        if (h_flags[0]) { sync_all(); g_err = "fit_coo: an id is outside [0, dim)"; return 2; }
        const size_t nnz = (size_t)h_flags[1];
        // unique (row, col) keys are in k1[0..nnz), their summed values in v1[0..nnz)
        auto build = [&](Side<real>& S, const u64* keys, const real* values, size_t nmajor) -> int {
            S.nnz = nnz; S.row_begin = 0; S.n_rows = nmajor;
            CK(dmalloc(&S.xv, std::max<size_t>(nnz, 1) * sizeof(real)));
            CK(dmalloc(&S.ind, std::max<size_t>(nnz, 1) * sizeof(int)));
            CK(dmalloc(&S.ptr, (nmajor + 1) * sizeof(long long)));
            CK(cudaMemcpyAsync(S.xv, values, nnz * sizeof(real), cudaMemcpyDeviceToDevice, stream));
            minor_ids_kernel<<<grid, 256, 0, stream>>>(keys, nnz, S.ind);
            LAUNCHED();
            key_offsets_kernel<<<grid, 256, 0, stream>>>(keys, nnz, nmajor, S.ptr);
            LAUNCHED();
            CK(cudaGetLastError());
            S.h_ptr.resize(nmajor + 1);
            CK(cudaMemcpyAsync(S.h_ptr.data(), S.ptr, (nmajor + 1) * sizeof(long long), cudaMemcpyDeviceToHost, stream));
            return 0;
        };
        if (build(sides[PMF_SIDE_CSR], k1, v1, dimA)) return 1;
        swap_keys_kernel<<<grid, 256, 0, stream>>>(k1, nnz, k2);
        LAUNCHED();
        tb = tmp_bytes;
        CK(cub::DeviceRadixSort::SortPairs(tmp, tb, k2, k1, v1, v2, (int)nnz, 0, 32 + bits(dimB), stream));
        LAUNCHED();
        if (build(sides[PMF_SIDE_CSC], k1, v2, dimB)) return 1;
        return sync_all();
    }
    int ingest_coo(const void* rows, const void* cols, const void* vals, size_t n, int index_bytes) override
    {
        CK(cudaSetDevice(device));
        if (index_bytes == 8) return ingest_impl<uint64_t>((const uint64_t*)rows, (const uint64_t*)cols, (const real*)vals, n);
        if (index_bytes == 4) return ingest_impl<int>((const int*)rows, (const int*)cols, (const real*)vals, n);
        return fail("fit_coo: index_bytes must be 4 or 8");
    }
    // device CSR / CSC back to host arrays at the caller's index width (tests, and callers that want
    // the conversion alone)
    int export_matrix(int side, void* values, void* indptr, void* indices, int index_bytes) override
    {
        CK(cudaSetDevice(device));
        Side<real>& S = sides[side];
        if (!S.ptr) return fail("export_matrix: side %d not set", side);
        if (index_bytes != 4 && index_bytes != 8) return fail("export_matrix: index_bytes must be 4 or 8");
        const int grid = num_sms * 8;
        CK(cudaMemcpyAsync(values, S.xv, S.nnz * sizeof(real), cudaMemcpyDeviceToHost, stream));
        if (index_bytes == 4) {
            CK(cudaMemcpyAsync(indices, S.ind, S.nnz * sizeof(int), cudaMemcpyDeviceToHost, stream));
            int* p32 = (int*)indptr;
            for (size_t i = 0; i <= S.n_rows; i++) p32[i] = (int)S.h_ptr[i];
        } else {
            uint64_t* w = nullptr;
            CK(dmalloc(&w, std::max<size_t>(S.nnz, 1) * sizeof(uint64_t)));
            deferred.push_back(w);
            widen_ids_kernel<uint64_t><<<grid, 256, 0, stream>>>(S.ind, S.nnz, w);
            LAUNCHED();
            CK(cudaMemcpyAsync(indices, w, S.nnz * sizeof(uint64_t), cudaMemcpyDeviceToHost, stream));
            uint64_t* p64 = (uint64_t*)indptr;
            for (size_t i = 0; i <= S.n_rows; i++) p64[i] = (uint64_t)S.h_ptr[i];
        }
        return sync_all();
    }

    // ---- factors_multiple (src/pred.c:66-199): rows of A for new data, B and Bsum fixed ---------
    // The handle holds the new rows' CSR on the CSR side and B; A (dimA rows) is produced here.  Bsum and Amean
    // are k host reals.  A_out == NULL leaves the rows on the device only (A of this handle).
    int factors_multiple(void* A_out, const void* Bsum_v, const void* Amean_v, const pmf_b200_params& p,
                         int reuse_mean) override
    {
        CK(cudaSetDevice(device));
        const real* Bsum = (const real*)Bsum_v;
        const real* Amean = (const real*)Amean_v;
        const real l2 = (real)p.l2_reg, w = (real)p.w_mult;
        real step = (real)p.step_size;
        {   // initialise every row to the mean of the old A (:144-147); tncg without reuse_mean starts
            // from 1e-3 inside the solver, rows are zero-filled here only to be deterministic
            const bool mean = reuse_mean || p.method != PMF_TNCG;
            real* d_mean = nullptr;
            if (mean) {
                CK(dmalloc(&d_mean, (size_t)k * sizeof(real)));
                deferred.push_back(d_mean);
                CK(cudaMemcpyAsync(d_mean, Amean, (size_t)k * sizeof(real), cudaMemcpyHostToDevice, stream));
            }
            const int grid = (int)std::min<size_t>((dimA * (size_t)ldf + 255) / 256, (size_t)num_sms * 8);
            fill_rows_kernel<real><<<std::max(grid, 1), 256, 0, stream>>>(A, dimA, k, ldf, d_mean);
            LAUNCHED();
            CK(cudaGetLastError());
            if (sync_all()) return 1;
        }
        pmf_b200_params q = p;
        q.early_stop = 0;
        std::vector<real> scaled(k);
        if (p.method == PMF_PG) {
            const real step0 = step;
            for (size_t it = 0; it < p.numiter; it++) {                               // :152-167
                for (int c = 0; c < k; c++) scaled[c] = Bsum[c] * (-step);            // w == 1: scaled once
                const real* cs = (w == (real)1) ? scaled.data() : Bsum;               // w != 1: raw sums, scaled in-kernel
                const double cdiv = (double)(real)(1. / (1. + 2. * (double)l2 * (double)step));
                if (half_sweep_ex(PMF_SIDE_CSR, q, (double)step, cdiv, nullptr, cs, -step0, -1)) return 1;
                CK(cudaStreamSynchronize(stream));   // `scaled` is re-used by the next iteration
                step = (real)((double)step * 0.5);
            }
        } else if (p.method == PMF_CG) {                                              // :171-178
            if (half_sweep_ex(PMF_SIDE_CSR, q, (double)step, 1.0, nullptr, Bsum, (real)1,
                              (long long)(p.maxupd * p.numiter))) return 1;
        } else {                                                                      // :180-188
            q.reuse_prev = reuse_mean;
            if (half_sweep_ex(PMF_SIDE_CSR, q, (double)step, 1.0, nullptr, Bsum, (real)1, -1)) return 1;
        }
        CK(cudaStreamSynchronize(stream));
        return get_factors(A_out, nullptr);
    }

    // ---- numiter alternating sweeps (src/poismf.c:506-608) -------------------------
    // hooks of the pipelined drop-in call: `before_first_A` runs on the host right after the first B
    // half-sweep has been enqueued (it uploads the CSR orientation behind it), `after_last_B` right
    // after the last one (it marks B as final), `after_last_A` once the last A half-sweep has been
    // enqueued (it downloads B while A's rows are still being solved; a pageable destination makes
    // that copy block the host, hence only after the enqueue)
    struct SweepHooks {
        std::function<int()> before_first_A, after_last_B, after_last_A;
    };
    int sweeps(const pmf_b200_params& p) override { return sweeps_ex(p, nullptr); }
    int sweeps_ex(const pmf_b200_params& p, SweepHooks* hk)
    {
        // the reference carries step_size as real_t: round it the same way
        real step = (real)p.step_size;
        const real l2 = (real)p.l2_reg;
        bool stopA = false, stopB = false;
        if (sides[1].n_rows != dimB || (!hk && sides[0].n_rows != dimA))
            return fail("sweeps: handle holds a shard; drive it with pmf_b200_half_sweep");
        for (size_t it = 0; it < p.numiter; it++) {
            if (g_interrupted) return 2;
            const double cdiv = (double)(real)(1. / (1. + 2. * (double)l2 * (double)step));   // :511
            unsigned long long unch = 0;
            if (!(p.method == PMF_TNCG && stopB)) {
                if (half_sweep(PMF_SIDE_CSC, p, (double)step, cdiv, &unch)) return 1;
                if (p.method == PMF_TNCG && p.early_stop)
                    stopB = ((double)unch / (double)dimB) >= .95;                             // :402
            }
            if (hk && it == 0 && hk->before_first_A()) return 1;
            if (hk && it + 1 == p.numiter && hk->after_last_B()) return 1;
            if (p.method == PMF_PG) step = (real)((double)step * 0.5);                        // :532
            if (g_interrupted) return 2;
            if (!(p.method == PMF_TNCG && stopA)) {
                if (half_sweep(PMF_SIDE_CSR, p, (double)step, cdiv, &unch)) return 1;
                if (p.method == PMF_TNCG && p.early_stop)
                    stopA = ((double)unch / (double)dimA) >= .95;
            }
            if (hk && it + 1 == p.numiter && hk->after_last_A()) return 1;
            if (stopA && stopB) break;                                                        // :606
        }
        return 0;
    }

    // ---- the stateless drop-in call (run_poismf), transfers pipelined against the half-sweeps ---------
    //   stream:       A, B, CSC up | plan | B half-sweep ............ | A half-sweep ..... | A down
    //   copy_stream:                      | CSR up, plan ------------^ | (last sweep) B down
    int run_dropin(void* Ah, void* Bh, const void* Xr, const void* Xr_indptr, const void* Xr_indices, size_t nnz_r,
                   const void* Xc, const void* Xc_indptr, const void* Xc_indices, size_t nnz_c, int index_bytes,
                   const pmf_b200_params& p, const std::function<void(const char*)>& lap, bool timing,
                   bool matrix_resident) override
    {
        // matrix_resident: both orientations are already on the device from an earlier call with the
        // same arrays (POISMF_B200_CACHE_X); only the factors travel
        CK(cudaSetDevice(device));
        const bool strict = (p.flags & PMF_FLAG_STRICT) != 0;
        if (copy_in(A, Ah, dimA, stream)) return 1;
        if (copy_in(B, Bh, dimB, stream)) return 1;
        if (!matrix_resident &&
            upload_matrix(PMF_SIDE_CSC, Xc, Xc_indptr, Xc_indices, nnz_c, index_bytes, 0, dimB, stream)) return 1;
        if (plan(sides[PMF_SIDE_CSC], p, stream)) return 1;
        if (timing) { if (sync_all()) return 1; lap("up A,B,CSC+plan"); }
        bool csr_up = false, b_down = false;
        SweepHooks hk;
        hk.before_first_A = [&]() -> int {
            csr_up = true;
            if (!matrix_resident &&
                upload_matrix(PMF_SIDE_CSR, Xr, Xr_indptr, Xr_indices, nnz_r, index_bytes, 0, dimA, copy_stream)) return 1;
            if (plan(sides[PMF_SIDE_CSR], p, copy_stream)) return 1;
            CK(cudaEventRecord(ev_copy, copy_stream));
            CK(cudaStreamWaitEvent(stream, ev_copy, 0));
            if (timing) { cudaStreamSynchronize(copy_stream); lap("up CSR+plan"); cudaStreamSynchronize(stream); lap("B half-sweep"); }
            return 0;
        };
        bool b_final = false;
        hk.after_last_B = [&]() -> int {
            b_final = true;
            CK(cudaEventRecord(ev_main, stream));
            return 0;
        };
        hk.after_last_A = [&]() -> int {
            b_down = true;
            if (b_final) CK(cudaStreamWaitEvent(copy_stream, ev_main, 0));
            else { CK(cudaEventRecord(ev_main, stream)); CK(cudaStreamWaitEvent(copy_stream, ev_main, 0)); }
            return copy_out(Bh, B, dimB, copy_stream);
        };
        int rc = sweeps_ex(p, &hk);
        if (rc == 1) { sync_all(); return 1; }
        if (timing) { cudaStreamSynchronize(stream); lap("rest of sweeps"); }
        // interrupted fits (rc 2) still return the factors computed so far
        if (!b_down && hk.after_last_A()) rc = 1;
        if (copy_out(Ah, A, dimA, stream)) rc = 1;
        if (sync_all()) rc = 1;
        if (timing) lap("download");
        (void)csr_up;
        return rc;
    }
};

// ---------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------
extern "C" pmf_b200_handle* pmf_b200_create(int dtype, size_t dimA, size_t dimB, size_t k, int device)
{
    if (pmf_b200_device_count() <= 0) {
        fail("no usable CUDA device: poismf_b200 has no CPU fallback");
        return nullptr;
    }
    if (k == 0 || k > 256) { fail("k must be in [1, 256]"); return nullptr; }
    if (dimA > (size_t)INT32_MAX || dimB > (size_t)INT32_MAX) { fail("dimensions must be <= 2^31-1"); return nullptr; }
    pmf_b200_handle* h = nullptr;
    if (dtype == PMF_F32) h = new HandleT<float>();
    else if (dtype == PMF_F64) h = new HandleT<double>();
    else { fail("bad dtype"); return nullptr; }
    h->dtype = dtype; h->device = device; h->dimA = dimA; h->dimB = dimB; h->k = (int)k;
    int rc = dtype == PMF_F32 ? static_cast<HandleT<float>*>(h)->init() : static_cast<HandleT<double>*>(h)->init();
    if (rc) { delete h; return nullptr; }
    return h;
}
extern "C" void pmf_b200_destroy(pmf_b200_handle* h) { delete h; }
extern "C" int pmf_b200_ldf(const pmf_b200_handle* h) { return h->ldf; }
extern "C" int pmf_b200_set_matrix(pmf_b200_handle* h, int side, const void* values, const void* indptr,
                                   const void* indices, size_t nnz, int index_bytes, size_t row_begin, size_t n_rows)
{
    return h->set_matrix(side, values, indptr, indices, nnz, index_bytes, row_begin, n_rows);
}
extern "C" int pmf_b200_set_factors(pmf_b200_handle* h, const void* A, const void* B) { return h->set_factors(A, B); }
extern "C" int pmf_b200_get_factors(pmf_b200_handle* h, void* A, void* B) { return h->get_factors(A, B); }
extern "C" int pmf_b200_bind_factors(pmf_b200_handle* h, void* A, void* B) { return h->bind_factors(A, B); }
extern "C" int pmf_b200_set_factor_rows(pmf_b200_handle* h, int which, const void* rows, size_t row_begin, size_t n_rows)
{
    return h->set_factor_rows(which, rows, row_begin, n_rows);
}
extern "C" void* pmf_b200_factor_ptr(pmf_b200_handle* h, int which) { return h->factor_ptr(which); }
extern "C" int pmf_b200_set_stream(pmf_b200_handle* h, void* s)
{
    cudaSetDevice(h->device);
    if (h->have_stream) cudaStreamSynchronize(h->stream);      // work enqueued so far stays ordered before the switch
    if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
    h->stream = (cudaStream_t)s;
    h->own_stream = false; h->have_stream = true;
    return 0;
}
extern "C" int pmf_b200_sweeps(pmf_b200_handle* h, const pmf_b200_params* p) { return h->sweeps(*p); }
extern "C" int pmf_b200_half_sweep(pmf_b200_handle* h, int side, const pmf_b200_params* p, double step_size,
                                   double cnst_div, unsigned long long* n_unchanged)
{
    return h->half_sweep(side, *p, step_size, cnst_div, n_unchanged);
}
extern "C" int pmf_b200_ipc_export(pmf_b200_handle* h, int which, void* out) { return h->ipc_export(which, out); }
extern "C" int pmf_b200_ipc_import(pmf_b200_handle* h, int which, const void* handles, int n_ranks, int self_rank)
{
    return h->ipc_import(which, handles, n_ranks, self_rank);
}
extern "C" int pmf_b200_set_profiling(pmf_b200_handle* h, int on)
{
    h->clear_profile();
    h->profiling = on != 0;
    return 0;
}
extern "C" int pmf_b200_get_profile(pmf_b200_handle* h, pmf_b200_bin_profile* out, int max_entries)
{
    return h->get_profile(out, max_entries);
}
static void drop_matrix_cache();
static void drop_resident_matrix();
extern "C" size_t pmf_b200_release_cache(void)
{
    drop_matrix_cache();
    drop_resident_matrix();
    return DevPool::get().release(-1);
}
extern "C" int pmf_b200_sync(pmf_b200_handle* h)
{
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    if (h->exchange_status()) return fail("sharded fit: a peer did not arrive at an exchange point");
    return 0;
}

// ---- matrix cache of the stateless drop-in call (opt-in, POISMF_B200_CACHE_X=1) ------------------------
// Key: device, types, shapes, the six host pointers and a fingerprint of each array (all of indptr,
// 4096 evenly spaced 8-byte words of values / indices plus their last word).  The fingerprint detects
// ordinary in-place edits, not adversarial ones: that is why the cache is opt-in.
struct XKey {
    int device = -1, dtype = -1, index_bytes = 0;
    size_t dimA = 0, dimB = 0, k = 0, nnz_r = 0, nnz_c = 0;
    const void* ptr[6] = {};
    uint64_t fp[6] = {};
    bool operator==(const XKey& o) const
    {
        if (device != o.device || dtype != o.dtype || index_bytes != o.index_bytes || dimA != o.dimA ||
            dimB != o.dimB || k != o.k || nnz_r != o.nnz_r || nnz_c != o.nnz_c) return false;
        for (int i = 0; i < 6; i++) if (ptr[i] != o.ptr[i] || fp[i] != o.fp[i]) return false;
        return true;
    }
};
static uint64_t fingerprint(const void* p, size_t bytes, bool full)
{
    uint64_t hsh = 0x243f6a8885a308d3ULL ^ bytes;
    auto mix = [&](uint64_t v) { hsh ^= v + 0x9e3779b97f4a7c15ULL + (hsh << 6) + (hsh >> 2); };
    const size_t words = bytes / 8;
    const unsigned char* b = (const unsigned char*)p;
    auto word = [&](size_t i) { uint64_t v; memcpy(&v, b + i * 8, 8); return v; };
    if (full || words <= 8192) {
        for (size_t i = 0; i < words; i++) mix(word(i));
    } else {
        const size_t stride = words / 4096;
        for (size_t i = 0; i < words; i += stride) mix(word(i));
        mix(word(words - 1));
    }
    for (size_t i = words * 8; i < bytes; i++) mix(b[i]);
    return hsh;
}
static std::mutex g_xcache_mutex;
static pmf_b200_handle* g_xcache_handle = nullptr;
static XKey g_xcache_key;
static void drop_matrix_cache()
{
    std::lock_guard<std::mutex> g(g_xcache_mutex);
    if (g_xcache_handle) pmf_b200_destroy(g_xcache_handle);
    g_xcache_handle = nullptr;
}

// ---- run_poismf drop-in ------------------------------------------------------
static std::mutex g_sig_mutex;
static bool g_sig_locked = false;
static void on_sigint(int) { g_interrupted = 1; }

static int env_flags(int flags)
{
    const char* e = getenv("POISMF_B200_FLAGS");
    if (e && *e) flags |= atoi(e);
    return flags;
}
static int env_device()
{
    const char* e = getenv("POISMF_B200_DEVICE");
    return (e && *e) ? atoi(e) : 0;
}

extern "C" int pmf_b200_run_poismf(int dtype, int index_bytes,
                                   void* A, const void* Xr, const void* Xr_indptr, const void* Xr_indices,
                                   void* B, const void* Xc, const void* Xc_indptr, const void* Xc_indices,
                                   size_t dimA, size_t dimB, size_t k,
                                   double l2_reg, double l1_reg, double w_mult, double step_size,
                                   int method, int limit_step, size_t numiter, size_t maxupd,
                                   int early_stop, int reuse_prev, int handle_interrupt, int flags)
{
    // SIGINT handling as src/poismf.c:444-455,:618-630
    void (*old_handler)(int) = nullptr;
    bool have_lock = false;
    {
        std::lock_guard<std::mutex> g(g_sig_mutex);
        if (!g_sig_locked) {
            g_sig_locked = true; have_lock = true; g_interrupted = 0;
            old_handler = signal(SIGINT, on_sigint);
        }
    }
    int rc = 0;
    const bool timing = getenv("POISMF_B200_TIMING") != nullptr;
    auto now = []() { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6; };
    double t0 = now(), t1;
    std::function<void(const char*)> lap = [&](const char* what) {
        if (!timing) return;
        t1 = now(); fprintf(stderr, "poismf_b200 timing: %-14s %8.2f ms\n", what, t1 - t0); t0 = t1;
    };
    const size_t isz = (size_t)index_bytes;
    auto span = [&](const void* ptr, size_t n) -> size_t {
        return isz == 8 ? (size_t)(((const uint64_t*)ptr)[n] - ((const uint64_t*)ptr)[0])
                        : (size_t)(((const int*)ptr)[n] - ((const int*)ptr)[0]);
    };
    const size_t nnz_r = span(Xr_indptr, dimA), nnz_c = span(Xc_indptr, dimB);
    const size_t rsz = dtype == PMF_F32 ? 4 : 8;
    // POISMF_B200_CACHE_X: keep the uploaded matrix (both orientations + row plan) for the next call
    // with the same arrays (SURVEY 8f rank 3: repeated fits on one dataset)
    XKey key;
    const bool use_cache = getenv("POISMF_B200_CACHE_X") != nullptr && atoi(getenv("POISMF_B200_CACHE_X")) != 0;
    pmf_b200_handle* h = nullptr;
    bool resident = false;
    if (use_cache) {
        key.device = env_device(); key.dtype = dtype; key.index_bytes = index_bytes;
        key.dimA = dimA; key.dimB = dimB; key.k = k; key.nnz_r = nnz_r; key.nnz_c = nnz_c;
        const void* ptrs[6] = {Xr, Xr_indptr, Xr_indices, Xc, Xc_indptr, Xc_indices};
        const size_t bytes[6] = {nnz_r * rsz, (dimA + 1) * isz, nnz_r * isz, nnz_c * rsz, (dimB + 1) * isz, nnz_c * isz};
        for (int i = 0; i < 6; i++) { key.ptr[i] = ptrs[i]; key.fp[i] = fingerprint(ptrs[i], bytes[i], i == 1 || i == 4); }
        std::lock_guard<std::mutex> g(g_xcache_mutex);
        if (g_xcache_handle && g_xcache_key == key) { h = g_xcache_handle; resident = true; }
        else if (g_xcache_handle) pmf_b200_destroy(g_xcache_handle);
        g_xcache_handle = nullptr;       // taken (or dropped); put back after the fit
    }
    if (!h) h = pmf_b200_create(dtype, dimA, dimB, k, env_device());
    lap(resident ? "reuse handle" : "create");
    if (!h) rc = 1;
    if (!rc) {
        pmf_b200_params p;
        p.l2_reg = l2_reg; p.l1_reg = l1_reg; p.w_mult = w_mult; p.step_size = step_size;
        p.method = method; p.limit_step = limit_step; p.numiter = numiter; p.maxupd = maxupd;
        p.early_stop = early_stop; p.reuse_prev = reuse_prev; p.flags = env_flags(flags);
        rc = h->run_dropin(A, B, Xr, Xr_indptr, Xr_indices, nnz_r, Xc, Xc_indptr, Xc_indices, nnz_c, index_bytes, p,
                           lap, timing, resident);
    }
    if (h && use_cache && rc != 1) {
        std::lock_guard<std::mutex> g(g_xcache_mutex);
        if (g_xcache_handle) pmf_b200_destroy(g_xcache_handle);
        g_xcache_handle = h; g_xcache_key = key;
        h = nullptr;
    }
    if (h) pmf_b200_destroy(h);
    lap("destroy");
    if (rc == 1) fprintf(stderr, "Error: out of memory.\n");
    {
        std::lock_guard<std::mutex> g(g_sig_mutex);
        const bool was_interrupted = g_interrupted != 0;
        if (was_interrupted && rc != 1) { rc = 2; fprintf(stderr, "Error: procedure was interrupted\n"); }
        if (have_lock) {
            signal(SIGINT, old_handler);
            g_sig_locked = false;
            g_interrupted = 0;
        }
        if (was_interrupted && !handle_interrupt) raise(SIGINT);
    }
    return rc;
}

// ---- factors_multiple drop-in (src/pred.c:66-199, prototype src/poismf.h:270-280) ------------
extern "C" int pmf_b200_factors_multiple(int dtype, int index_bytes, void* A, const void* B, const void* Bsum,
                                         const void* Amean, const void* Xr, const void* Xr_indptr,
                                         const void* Xr_indices, int k, size_t dimA, size_t dimB,
                                         double l2_reg, double w_mult, double step_size, size_t niter, size_t maxupd,
                                         int method, int limit_step, int reuse_mean, int flags)
{
    pmf_b200_handle* h = pmf_b200_create(dtype, dimA, dimB, (size_t)k, env_device());
    if (!h) return 1;
    const size_t nnz = index_bytes == 8 ? (size_t)((const uint64_t*)Xr_indptr)[dimA] - (size_t)((const uint64_t*)Xr_indptr)[0]
                                        : (size_t)(((const int*)Xr_indptr)[dimA] - ((const int*)Xr_indptr)[0]);
    int rc = h->set_matrix(PMF_SIDE_CSR, Xr, Xr_indptr, Xr_indices, nnz, index_bytes, 0, dimA);
    if (!rc) rc = h->set_factors(nullptr, B);
    if (!rc) {
        pmf_b200_params p;
        p.l2_reg = l2_reg; p.l1_reg = 0; p.w_mult = w_mult; p.step_size = step_size; p.method = method;
        p.limit_step = limit_step; p.numiter = niter; p.maxupd = maxupd; p.early_stop = 0; p.reuse_prev = 0;
        p.flags = env_flags(flags);
        rc = h->factors_multiple(A, Bsum, Amean, p, reuse_mean);
    }
    pmf_b200_destroy(h);
    if (rc) fprintf(stderr, "Error: out of memory.\n");
    return rc ? 1 : 0;
}

// ---- fit straight from COO triplets (front-end ingestion on the device, SURVEY 8f rank 4) ------------
// = PoisMF._process_data + _fit (poismf/__init__.py:376-440) without the host-side tocsr()/tocsc().
extern "C" int pmf_b200_fit_coo(int dtype, int index_bytes, void* A, void* B, const void* rows, const void* cols,
                                const void* vals, size_t n_entries, size_t dimA, size_t dimB, size_t k,
                                double l2_reg, double l1_reg, double w_mult, double step_size,
                                int method, int limit_step, size_t numiter, size_t maxupd,
                                int early_stop, int reuse_prev, int flags)
{
    pmf_b200_handle* h = pmf_b200_create(dtype, dimA, dimB, k, env_device());
    if (!h) return 1;
    int rc = h->ingest_coo(rows, cols, vals, n_entries, index_bytes);
    if (!rc) rc = h->set_factors(A, B);
    if (!rc) {
        pmf_b200_params p;
        p.l2_reg = l2_reg; p.l1_reg = l1_reg; p.w_mult = w_mult; p.step_size = step_size;
        p.method = method; p.limit_step = limit_step; p.numiter = numiter; p.maxupd = maxupd;
        p.early_stop = early_stop; p.reuse_prev = reuse_prev; p.flags = env_flags(flags);
        rc = h->sweeps(p);
        if (rc != 1 && h->get_factors(A, B)) rc = 1;
    }
    pmf_b200_destroy(h);
    return rc;
}
// The conversion alone: CSR and CSC of the triplets into caller arrays sized for n_entries values /
// ids and dim+1 offsets; *nnz_out = stored entries after summing duplicates.
extern "C" int pmf_b200_coo_to_csr_csc(int dtype, int index_bytes, const void* rows, const void* cols, const void* vals,
                                       size_t n_entries, size_t dimA, size_t dimB, void* Xr, void* Xr_indptr,
                                       void* Xr_indices, void* Xc, void* Xc_indptr, void* Xc_indices, size_t* nnz_out)
{
    pmf_b200_handle* h = pmf_b200_create(dtype, dimA, dimB, 1, env_device());
    if (!h) return 1;
    int rc = h->ingest_coo(rows, cols, vals, n_entries, index_bytes);
    if (!rc) rc = h->export_matrix(PMF_SIDE_CSR, Xr, Xr_indptr, Xr_indices, index_bytes);
    if (!rc) rc = h->export_matrix(PMF_SIDE_CSC, Xc, Xc_indptr, Xc_indices, index_bytes);
    if (!rc && nnz_out) *nnz_out = h->side_nnz(PMF_SIDE_CSR);
    pmf_b200_destroy(h);
    return rc;
}
// The conversion into a fit handle: both orientations replace the handle's matrix and stay on the device.
extern "C" int pmf_b200_set_coo(pmf_b200_handle* h, const void* rows, const void* cols, const void* vals,
                                size_t n_entries, int index_bytes)
{
    if (!h) return fail("set_coo: null handle");
    const char* bad = n_entries == 0 ? "set_coo: no entries"
                    : n_entries > (size_t)INT32_MAX ? "set_coo: more than 2^31-1 triplets"
                    : (index_bytes != 4 && index_bytes != 8) ? "set_coo: index_bytes must be 4 or 8"
                    : h->has_peers() ? "set_coo: the handle is part of a sharded fit (set each rank's shard instead)"
                    : nullptr;
    if (bad) { g_err = bad; return 2; }
    return h->ingest_coo(rows, cols, vals, n_entries, index_bytes);
}

// ---- factors_single drop-in (src/pred.c:201-304, prototype src/poismf.h:281-289) --------------------
// One new row by tncg == factors_multiple on a one-row matrix.  The reference passes no row count
// for B; only the nnz rows the ids name are read, so they are gathered into a compact nnz x k
// matrix on the host and the ids renumbered 0..nnz-1 (same order => same summation order).
template <class real, class IX>
static int factors_single_impl(int dtype, real* out, size_t k, const real* Amean, int reuse_mean, const real* X,
                               const IX* X_ind, size_t nnz, const real* B, const real* Bsum, int maxupd,
                               double l2_reg, double l1_new, double l1_old, double w_mult, int flags)
{
    if (nnz == 0) { memset(out, 0, k * sizeof(real)); return 0; }           // :212-215
    std::vector<real> Bc(nnz * k), bs(Bsum, Bsum + k);
    std::vector<IX> ids(nnz);
    for (size_t t = 0; t < nnz; t++) {
        memcpy(&Bc[t * k], B + (size_t)X_ind[t] * k, k * sizeof(real));
        ids[t] = (IX)t;
    }
    // Bsum holds the old l1 already; only a positive difference is added (:218, :254-257).  (With
    // w_mult != 1 the reference adds it after the per-row adjustment; here it goes in before, a
    // last-bit difference in that one combination.)
    const real l1d = (real)l1_new - (real)l1_old;
    if (l1d > (real)0) for (size_t i = 0; i < k; i++) bs[i] += l1d;
    const IX ptr[2] = {(IX)0, (IX)nnz};
    return pmf_b200_factors_multiple(dtype, (int)sizeof(IX), out, Bc.data(), bs.data(), Amean, X, ptr, ids.data(),
                                     (int)k, 1, nnz, l2_reg, w_mult, 0., 1, (size_t)std::max(maxupd, 0), PMF_TNCG, 0,
                                     reuse_mean, flags);
}
extern "C" int pmf_b200_factors_single(int dtype, int index_bytes, void* out, size_t k, const void* Amean,
                                       int reuse_mean, const void* X, const void* X_ind, size_t nnz, const void* B,
                                       const void* Bsum, int maxupd, double l2_reg, double l1_new, double l1_old,
                                       double w_mult, int flags)
{
    if (index_bytes != 4 && index_bytes != 8) return fail("factors_single: index_bytes must be 4 or 8");
    return with_types(dtype, index_bytes, "bad dtype", [&](auto r, auto i) {
        using real = decltype(r); using IX = decltype(i);
        return factors_single_impl<real, IX>(dtype, (real*)out, k, (const real*)Amean, reuse_mean, (const real*)X,
                                             (const IX*)X_ind, nnz, (const real*)B, (const real*)Bsum, maxupd, l2_reg,
                                             l1_new, l1_old, w_mult, flags);
    });
}

// ---- dense host rows -> padded device rows, for the stateless inference entry points -----------------
// One contiguous copy + a device repack (a pitched cudaMemcpy2D of 200-byte rows runs ~10x slower over
// PCIe).  With POISMF_B200_CACHE_FACTORS=1 the padded matrix stays on the device for the next call that
// passes the same host array (pointer, shape and a sampled content fingerprint): a model that is queried
// user by user (PoisMF.topN, poismf/__init__.py:914-923) then uploads its item factors once.
struct ResidentMatrix {
    const void* host = nullptr; size_t rows = 0; int k = 0, ldf = 0, dtype = -1, device = -1;
    uint64_t fp = 0; void* dev = nullptr;
};
static std::mutex g_rm_mutex;
static ResidentMatrix g_rm;
static void drop_resident_matrix()
{
    std::lock_guard<std::mutex> g(g_rm_mutex);
    if (g_rm.dev) dfree(g_rm.dev);
    g_rm = ResidentMatrix();
}
template <class real>
static int upload_rows(real** dev_out, const real* host, size_t rows, int k, int ldf, bool* resident, bool may_cache)
{
    *resident = false;
    const int dtype = std::is_same<real, float>::value ? PMF_F32 : PMF_F64;
    const bool cache = may_cache && getenv("POISMF_B200_CACHE_FACTORS") && atoi(getenv("POISMF_B200_CACHE_FACTORS")) != 0;
    uint64_t fp = 0;
    if (cache) {
        fp = fingerprint(host, rows * (size_t)k * sizeof(real), false);
        std::lock_guard<std::mutex> g(g_rm_mutex);
        if (g_rm.dev && g_rm.host == host && g_rm.rows == rows && g_rm.k == k && g_rm.ldf == ldf && g_rm.dtype == dtype &&
            g_rm.device == env_device() && g_rm.fp == fp) {
            *dev_out = (real*)g_rm.dev; *resident = true;
            return 0;
        }
    }
    real* dev = nullptr;
    CK(dmalloc(&dev, std::max<size_t>(rows, 1) * (size_t)ldf * sizeof(real)));
    // (pageable callers' arrays go through the multi-threaded page-locked staging of staged_copy.h)
    if (ldf == k) {
        CK(Stager::get().h2d(dev, host, rows * (size_t)k * sizeof(real), 0));
        CK(cudaStreamSynchronize(0));
    } else {
        real* tmp = nullptr;
        CK(dmalloc(&tmp, std::max<size_t>(rows * (size_t)k, 1) * sizeof(real)));
        cudaError_t e = Stager::get().h2d(tmp, host, rows * (size_t)k * sizeof(real), 0);
        if (e == cudaSuccess) {
            pad_rows_kernel<real><<<148 * 8, 256>>>(tmp, dev, rows, k, ldf);
            LAUNCHED();
            e = cudaDeviceSynchronize();
        }
        dfree(tmp);
        if (e != cudaSuccess) { dfree(dev); return fail("upload failed: %s", cudaGetErrorString(e)); }
    }
    if (cache) {
        std::lock_guard<std::mutex> g(g_rm_mutex);
        if (g_rm.dev) dfree(g_rm.dev);
        g_rm.host = host; g_rm.rows = rows; g_rm.k = k; g_rm.ldf = ldf; g_rm.dtype = dtype; g_rm.device = env_device();
        g_rm.fp = fp; g_rm.dev = dev;
        *resident = true;
    }
    *dev_out = dev;
    return 0;
}

// ---- predict_multiple drop-in ------------------------------------------------
template <class real, class IX>
static int predict_impl(real* out, const real* A, const real* B, const IX* ixA, const IX* ixB, size_t n, int k,
                        size_t dimA, size_t dimB)
{
    CK(cudaSetDevice(env_device()));
    if (n == 0) return 0;
    // Few pairs (the reference's per-user call pattern, poismf/__init__.py:726-835): only the rows the pairs
    // name travel — gathered on the host into two n x k blocks, 2 n k reals instead of both whole matrices.
    // (crossover measured on B200: the host gather costs ~0.3 us per pair, the two whole uploads ~10 ms at config #2's shape)
    const bool gathered = 32 * n < dimA + dimB;
    const size_t rowsA = gathered ? n : dimA, rowsB = gathered ? n : dimB;
    DeviceBlocks mem;
    real *dA = nullptr, *dB = nullptr, *dout = nullptr;
    IX *da = nullptr, *db = nullptr;
    CK(mem.alloc(&dA, rowsA * (size_t)k * sizeof(real))); CK(mem.alloc(&dB, rowsB * (size_t)k * sizeof(real)));
    CK(mem.alloc(&dout, n * sizeof(real)));
    if (gathered) {
        std::vector<real> ga(n * (size_t)k), gb(n * (size_t)k);
        for (size_t i = 0; i < n; i++) {
            memcpy(&ga[i * k], A + (size_t)ixA[i] * k, (size_t)k * sizeof(real));
            memcpy(&gb[i * k], B + (size_t)ixB[i] * k, (size_t)k * sizeof(real));
        }
        CK(cudaMemcpy(dA, ga.data(), n * (size_t)k * sizeof(real), cudaMemcpyHostToDevice));
        CK(cudaMemcpy(dB, gb.data(), n * (size_t)k * sizeof(real), cudaMemcpyHostToDevice));
    } else {
        CK(mem.alloc(&da, n * sizeof(IX))); CK(mem.alloc(&db, n * sizeof(IX)));
        CK(cudaMemcpy(dA, A, dimA * (size_t)k * sizeof(real), cudaMemcpyHostToDevice));      // rows stay k wide: the
        CK(cudaMemcpy(dB, B, dimB * (size_t)k * sizeof(real), cudaMemcpyHostToDevice));      // kernel reads scalars
        CK(cudaMemcpy(da, ixA, n * sizeof(IX), cudaMemcpyHostToDevice));
        CK(cudaMemcpy(db, ixB, n * sizeof(IX), cudaMemcpyHostToDevice));
    }
    const int grid = (int)std::min<size_t>((n + 255) / 256, 148 * 16);
    predict_pairs_kernel<real, IX><<<grid, 256>>>(dA, dB, da, db, n, k, k, dout);
    LAUNCHED();
    CK(cudaGetLastError());
    CK(cudaMemcpy(out, dout, n * sizeof(real), cudaMemcpyDeviceToHost));
    mem.settled = true;
    return 0;
}
extern "C" int pmf_b200_predict_multiple(int dtype, int index_bytes, void* out, const void* A, const void* B,
                                         const void* ixA, const void* ixB, size_t n, int k, size_t dimA, size_t dimB)
{
    if (pmf_b200_device_count() <= 0) return fail("no usable CUDA device: poismf_b200 has no CPU fallback");
    return with_types(dtype, index_bytes, "predict_multiple: bad dtype/index width", [&](auto r, auto i) {
        using real = decltype(r); using IX = decltype(i);
        return predict_impl((real*)out, (const real*)A, (const real*)B, (const IX*)ixA, (const IX*)ixB, n, k, dimA, dimB);
    });
}

// ---- predict_multiple against the factors resident in a handle ------------------------------------------------
// Pairs per upload chunk: 8-byte ids travel in 16 MB blocks (4-byte ids in 8 MB), large enough for the threaded
// staging of pageable arrays (staged_copy.h) and for the launch between chunks to be hidden behind the copies.
static constexpr size_t PREDICT_CHUNK = (size_t)1 << 21;

// the upload stream of one pipelined call and the events of its two chunk slots, released when the call returns
// (a stream or event destroyed with work pending is released once that work completes)
struct UploadRing {
    cudaStream_t up = nullptr;
    cudaEvent_t loaded[2] = {}, consumed[2] = {};
    cudaError_t init()
    {
        cudaError_t e = cudaStreamCreateWithFlags(&up, cudaStreamNonBlocking);
        for (int s = 0; s < 2 && e == cudaSuccess; s++) {
            e = cudaEventCreateWithFlags(&loaded[s], cudaEventDisableTiming);
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&consumed[s], cudaEventDisableTiming);
        }
        return e;
    }
    ~UploadRing()
    {
        for (int s = 0; s < 2; s++) {
            if (loaded[s]) cudaEventDestroy(loaded[s]);
            if (consumed[s]) cudaEventDestroy(consumed[s]);
        }
        if (up) cudaStreamDestroy(up);
    }
};

// Chunk c's ids go up on the ring's stream into slot c % 2 (once chunk c - 2's kernel has read that slot) while chunk
// c - 1 is scored on `st`.  The scores of every chunk stay on the device until the last kernel has run; they are
// copied to `out` only if no pair was out of range, so a 2 leaves `out` untouched.
template <class real, class IX>
static int predict_fitted_impl(const real* dA, const real* dB, size_t dimA, size_t dimB, int k, int ldf, int num_sms,
                               cudaStream_t st, const IX* ixA, const IX* ixB, size_t n, real* out)
{
    size_t free_b = 0, total_b = 0;
    CK(cudaMemGetInfo(&free_b, &total_b));
    if (n > free_b / 4 / sizeof(real))
        return fail("predict_fitted: %zu scores exceed a quarter of the free device memory (%zu MB); pass fewer pairs "
                    "per call", n, free_b >> 20);
    const size_t chunk = std::min(n, PREDICT_CHUNK);
    const int nslots = n > chunk ? 2 : 1;
    DeviceBlocks mem;
    real* d_out = nullptr;
    int* d_bad = nullptr;
    IX* d_ix[2][2] = {};
    CK(mem.alloc(&d_out, n * sizeof(real)));
    CK(mem.alloc(&d_bad, sizeof(int)));
    for (int s = 0; s < nslots; s++)
        for (int w = 0; w < 2; w++) CK(mem.alloc(&d_ix[s][w], chunk * sizeof(IX)));
    UploadRing ring;               // a single chunk goes up on `st` itself: no stream or events to create
    if (nslots > 1) CK(ring.init());
    cudaStream_t up = nslots > 1 ? ring.up : st;
    CK(cudaMemsetAsync(d_bad, 0, sizeof(int), st));
    for (size_t off = 0, c = 0; off < n; off += chunk, c++) {
        const size_t m = std::min(chunk, n - off);
        const int s = (int)(c & 1);
        if (c >= 2) CK(cudaStreamWaitEvent(up, ring.consumed[s], 0));
        CK(Stager::get().h2d(d_ix[s][0], ixA + off, m * sizeof(IX), up));
        CK(Stager::get().h2d(d_ix[s][1], ixB + off, m * sizeof(IX), up));
        if (nslots > 1) {
            CK(cudaEventRecord(ring.loaded[s], up));
            CK(cudaStreamWaitEvent(st, ring.loaded[s], 0));
        }
        const int grid = (int)std::min<size_t>((m + 255) / 256, (size_t)num_sms * 16);
        predict_resident_kernel<real, IX><<<grid, 256, 0, st>>>(dA, dB, d_ix[s][0], d_ix[s][1], m, dimA, dimB, k, ldf,
                                                                d_out + off, d_bad);
        LAUNCHED();
        CK(cudaGetLastError());
        if (nslots > 1) CK(cudaEventRecord(ring.consumed[s], st));
    }
    int bad = 0;
    CK(cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (bad) {
        mem.settled = true;
        g_err = "predict_fitted: an id is outside [0, dimA) / [0, dimB)";
        return 2;
    }
    CK(Stager::get().d2h(out, d_out, n * sizeof(real), st));
    CK(cudaStreamSynchronize(st));
    mem.settled = true;
    return 0;
}

extern "C" int pmf_b200_predict_fitted(pmf_b200_handle* h, int index_bytes, const void* ixA, const void* ixB, size_t n,
                                       void* out)
{
    if (!h) return fail("predict_fitted: null handle");
    if (pmf_b200_sync(h)) return 1;             // every row of the last half-sweep (own and peers') has landed
    const void* A = h->factor_ptr(0);
    const void* B = h->factor_ptr(1);
    if (!A || !B) return fail("predict_fitted: the handle holds no factors");
    if (index_bytes != 4 && index_bytes != 8) { g_err = "predict_fitted: index_bytes must be 4 or 8"; return 2; }
    if (n == 0) return 0;
    return with_types(h->dtype, index_bytes, "predict_fitted: bad dtype", [&](auto r, auto i) {
        using real = decltype(r); using IX = decltype(i);
        return predict_fitted_impl<real, IX>((const real*)A, (const real*)B, h->dimA, h->dimB, h->k, h->ldf, h->num_sms,
                                             h->stream, (const IX*)ixA, (const IX*)ixB, n, (real*)out);
    });
}

// ---- topN ----------------------------------------------------------------------
struct ResidentFactors { const void* A; const void* B; int device; int ldf; };

// A (rowsA rows) and B (n rows) on the device, rows padded to ldf: a fit handle's replicas when rf is given
// (nothing is uploaded), else uploaded, B through the resident-matrix cache.  Uploaded blocks that the cache
// does not keep are released with `mem`.
template <class real>
static int factors_on_device(const ResidentFactors* rf, const real* A, size_t rowsA, const real* B, size_t n, int k,
                             int ldf, DeviceBlocks& mem, real** dA, real** dB, const char* what)
{
    if (rf) {
        if (rf->ldf != ldf) return fail("%s: resident factors have another row pitch", what);
        *dA = (real*)rf->A; *dB = (real*)rf->B;
        return 0;
    }
    bool resident = false;
    if (upload_rows<real>(dB, B, n, k, ldf, &resident, true)) return 1;
    if (!resident) mem.adopt(*dB);
    if (upload_rows<real>(dA, A, rowsA, k, ldf, &resident, false)) return 1;
    if (!resident) mem.adopt(*dA);
    return 0;
}

// rows user_ix[u0 .. u0 + m) of dA (rows u0 .. u0 + m without a list) -> dAsel, through the device list dusers
template <class real, class IX>
static int gather_users(const real* dA, int ldf, const IX* user_ix, size_t u0, size_t m, long long* dusers, real* dAsel)
{
    std::vector<long long> hu(m);
    for (size_t u = 0; u < m; u++) hu[u] = user_ix ? (long long)user_ix[u0 + u] : (long long)(u0 + u);
    CK(cudaMemcpy(dusers, hu.data(), m * sizeof(long long), cudaMemcpyHostToDevice));
    gather_rows_kernel<real><<<(int)std::min<size_t>((m * ldf + 255) / 256, 4096), 256>>>(dA, dusers, (int)m, ldf, dAsel);
    LAUNCHED();
    return 0;
}

// -> 0 when every one of the `count` ids on the device lies in [0, n), 2 when one does not (a negative id of a
// signed type is a huge size_t), 1 on a CUDA error.  Callers run it before any result is written.
template <class IX>
static int ids_in_range(const IX* dev_ids, size_t count, size_t n)
{
    if (!count) return 0;
    DeviceBlocks mem;
    int* d_bad = nullptr;
    int bad = 0;
    CK(mem.alloc(&d_bad, sizeof(int)));
    CK(cudaMemsetAsync(d_bad, 0, sizeof(int)));
    tc::any_id_out_of_range_kernel<IX><<<592, 256>>>(dev_ids, count, n, d_bad);
    LAUNCHED();
    CK(cudaMemcpy(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost));
    mem.settled = true;
    return bad ? 2 : 0;
}

// Batched topN over every item but the user's exclusions.  Three routes give the same ids and scores: the fused
// tensor-core select (topn_tc.cuh), the TF32 score matrix + CUB's segmented radix sort + exact re-score when the
// items are too few for the fused select, else exact scores (the reference's sums) and the segmented sort.
// Ranking = descending score; ties by ascending item id (the reference's tie order is
// qsort's, i.e. unspecified).  A single vector is the matrix A of one row: dimA = 1, n_users = 1, no user list.
template <class real, class IX>
static int topn_batch_impl(const real* A, const real* B, int k, const IX* user_ix, size_t n_users, size_t dimA,
                           const IX* excl_ptr, const IX* excl_ix, IX* outp_ix, real* outp_score, size_t n_top, size_t n,
                           bool allow_tc = true, const ResidentFactors* rf = nullptr)
{
    // rf: the factors already sit on a device, padded to ldf (a fit handle's replicas): nothing is uploaded
    CK(cudaSetDevice(rf ? rf->device : env_device()));
    if (n_top == 0 || n_top > n) return 2;
    // POISMF_B200_TOPN_TRACE=1: wall-clock of the call's phases on stderr (each mark synchronises the device)
    const bool trace = getenv("POISMF_B200_TOPN_TRACE") != nullptr;
    auto t_last = std::chrono::steady_clock::now();
    auto mark = [&](const char* what) {
        if (!trace) return;
        cudaDeviceSynchronize();
        const auto now = std::chrono::steady_clock::now();
        fprintf(stderr, "[topN] %-28s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(now - t_last).count());
        t_last = now;
    };
    // argument checks in the spirit of src/topN.c:121-128, per user: ids inside the matrices, offsets monotone,
    // enough items left after the exclusions (the excluded ids are range-checked on the device once uploaded)
    if (user_ix)
        for (size_t u = 0; u < n_users; u++)
            if ((size_t)user_ix[u] >= dimA) return 2;
    const bool have_excl = excl_ptr && excl_ix;
    if (have_excl)
        for (size_t u = 0; u < n_users; u++) {
            if (excl_ptr[u + 1] < excl_ptr[u]) return 2;
            if ((size_t)(excl_ptr[u + 1] - excl_ptr[u]) > n - n_top) return 2;
        }
    const int V = RealTraits<real>::V, ldf = round_up(k, V);
    const size_t pitch = (size_t)ldf * sizeof(real);
    const int kpad = round_up(k, 8);
    const int M_cand = (int)std::min<size_t>(n, std::min<size_t>(256, std::max<size_t>(2 * n_top, n_top + 32)));
    const size_t ntiles = (n + tc::TN - 1) / tc::TN, ngroups = (n + tc::GROUP - 1) / tc::GROUP;
    // TF32 candidates: float factors, k <= 128, n_top <= 128 and (checked on the device below) non-negative
    // factors, which the TF32 error bound assumes.  The fused select needs the items to hold 2 M_cand groups.
    // With fewer, the TF32 scores are sorted and the best M_cand re-scored exactly when there are >= 256 users
    // and n k >= 2 M_cand (k + 32): the exact re-score costs about M_cand (k + 32) per user against n k for exact
    // scores.  Wherever the exact route measured faster than this one, the rule picks it; it never picks it where
    // this one measured faster (32 768 users down to 1, 256..6 384 items, k 16/64/128, top-10/100:
    // profiles/r4_topn_sort_vs_exact.json)
    const bool fits_fused = ngroups >= (size_t)2 * M_cand;
    const bool sort_tf32 = n_users >= 256 && n * (size_t)k >= (size_t)2 * M_cand * (size_t)(k + 32);
    bool use_tc = allow_tc && std::is_same<real, float>::value && k <= 128 && n_top <= 128 && n >= 256 &&
                  (fits_fused || sort_tf32) && !getenv("POISMF_B200_TOPN_EXACT");
    bool fused = false;
    std::vector<size_t> redo;          // users whose TF32 proof failed: redone exactly afterwards
    {
        DeviceBlocks mem;
        real *dA = nullptr, *dB = nullptr;
        mark("argument checks");
        if (factors_on_device(rf, A, dimA, B, n, k, ldf, mem, &dA, &dB, "topN")) return 1;
        mark("factors on device");
        IX *dexp = nullptr, *dexi = nullptr;
        if (have_excl) {
            const size_t n_excl_total = (size_t)excl_ptr[n_users];
            CK(mem.alloc(&dexp, (n_users + 1) * sizeof(IX)));
            CK(mem.alloc(&dexi, std::max<size_t>(n_excl_total, 1) * sizeof(IX)));
            CK(cudaMemcpy(dexp, excl_ptr, (n_users + 1) * sizeof(IX), cudaMemcpyHostToDevice));
            CK(Stager::get().h2d(dexi, excl_ix, n_excl_total * sizeof(IX), 0));
            if (const int bad = ids_in_range(dexi + (size_t)excl_ptr[0], n_excl_total - (size_t)excl_ptr[0], n)) return bad;
        }
        CUtensorMap mapB;                  // B for the TMA unit, the same for every chunk of users
        if (use_tc) {
            int* d_neg = nullptr;
            CK(mem.alloc(&d_neg, sizeof(int)));
            CK(cudaMemset(d_neg, 0, sizeof(int)));
            tc::any_negative_kernel<<<256, 256>>>((const float*)dB, n * (size_t)ldf, d_neg);
            tc::any_negative_kernel<<<256, 256>>>((const float*)dA, dimA * (size_t)ldf, d_neg);
            LAUNCHED(); LAUNCHED();
            int neg = 0;
            CK(cudaMemcpy(&neg, d_neg, sizeof(int), cudaMemcpyDeviceToHost));
            use_tc = !neg && tc::make_operand_map(&mapB, (const float*)dB, n, ldf) == 0;
            fused = use_tc && fits_fused;
        }
        if (fused) {
            // ---- fused select (topn_tc.cuh): no score matrix; two passes over the tensor-core tiles ----
            const size_t words = ntiles * 4;     // exclusion bitmap: 128 bits per tile and user
            // group maxima per user: whole tiles (the scorer numbers 8 groups per visited tile, the last tile's
            // groups beyond n included)
            const size_t ngroups_alloc = ntiles * (tc::TN / tc::GROUP);
            const size_t per_user = ngroups_alloc * 4 + (have_excl ? words * 4 : 0) + (size_t)tc::CAND_SLACK * tc::CAND_CAP * 8 +
                                    (size_t)tc::CAND_TOP * 8 + pitch + n_top * 12 + 64;
            // users per batch: a quarter of the free device memory, at most 32 GB, for the per-user work arrays
            size_t mem_free = 0, mem_total = 0;
            CK(cudaMemGetInfo(&mem_free, &mem_total));
            const size_t budget = std::max<size_t>((size_t)1 << 30, std::min<size_t>(mem_free / 4, (size_t)32 << 30));
            size_t fchunk = std::max<size_t>(1, std::min<size_t>(n_users, budget / per_user));
            fchunk = std::min<size_t>(fchunk, 32768);
            real* dAsel = nullptr;
            long long *dusers = nullptr, *d_out_ids = nullptr;
            float *gmax = nullptr, *tau = nullptr, *cand_sc = nullptr, *top_sc = nullptr, *d_out_sc = nullptr;
            int *cand_id = nullptr, *cand_cnt = nullptr, *top_id = nullptr, *d_ovf = nullptr, *d_flag = nullptr;
            uint32_t* bits = nullptr;
            CK(mem.alloc(&dAsel, fchunk * pitch));
            CK(mem.alloc(&dusers, fchunk * sizeof(long long)));
            CK(mem.alloc(&gmax, fchunk * ngroups_alloc * sizeof(float)));
            CK(mem.alloc(&tau, fchunk * sizeof(float)));
            CK(mem.alloc(&cand_sc, fchunk * tc::CAND_SLACK * tc::CAND_CAP * sizeof(float)));
            CK(mem.alloc(&cand_id, fchunk * tc::CAND_SLACK * tc::CAND_CAP * sizeof(int)));
            CK(mem.alloc(&cand_cnt, fchunk * 64 * sizeof(int)));      // [user][region], regions <= 64
            CK(mem.alloc(&top_sc, fchunk * tc::CAND_TOP * sizeof(float)));
            CK(mem.alloc(&top_id, fchunk * tc::CAND_TOP * sizeof(int)));
            CK(mem.alloc(&d_ovf, fchunk * sizeof(int)));
            CK(mem.alloc(&d_out_ids, fchunk * n_top * sizeof(long long)));
            CK(mem.alloc(&d_out_sc, fchunk * n_top * sizeof(float)));
            CK(mem.alloc(&d_flag, fchunk * sizeof(int)));
            if (have_excl) CK(mem.alloc(&bits, fchunk * words * sizeof(uint32_t)));
            mark("work arrays");
            // The threshold pass visits every S-th item tile only: the M-th largest group maximum of a SAMPLE of
            // the items is a lower bound of the one over all items, so every wanted item still passes tau; about
            // S M items do (instead of M), which the candidate slots must hold (S M <= 1/4 of them)
            int S = 1;
            for (int c : {4, 2})
                if (ntiles >= (size_t)c * M_cand && (size_t)c * M_cand <= (size_t)tc::CAND_CAP / 4) { S = c; break; }
            const size_t pipe_smem = tc::pipe_smem_bytes(kpad);
            const int pipe_stages = tc::pipe_stages(kpad);
            CK(cudaFuncSetAttribute(tc::score_pipe_tf32_kernel<tc::MODE_GROUPMAX>,
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pipe_smem));
            CK(cudaFuncSetAttribute(tc::score_pipe_tf32_kernel<tc::MODE_EMIT>,
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pipe_smem));
            int num_sms = 148, dev = 0;
            CK(cudaGetDevice(&dev));
            CK(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev));
            std::vector<long long> hid;
            std::vector<float> hsc;
            std::vector<int> hfl, hov;
            for (size_t u0 = 0; u0 < n_users; u0 += fchunk) {
                const size_t m = std::min(fchunk, n_users - u0);
                if (gather_users(dA, ldf, user_ix, u0, m, dusers, dAsel)) return 1;
                CUtensorMap mapA;          // the chunk's rows: those beyond m read as zeros
                if (tc::make_operand_map(&mapA, (const float*)dAsel, m, ldf))
                    return fail("topN: cannot encode the tensor map of %zu user rows", m);
                tc::TileOut o = {};
                if (have_excl) {
                    CK(cudaMemsetAsync(bits, 0, m * words * sizeof(uint32_t)));
                    tc::exclusion_bitmap_kernel<IX><<<dim3(4, (unsigned)m), 128>>>(bits, words, dexp, dexi, u0, n);
                    LAUNCHED();
                    o.excl_bits = bits; o.excl_words = words;
                }
                o.gmax = gmax; o.tau = tau;
                o.cand_sc = cand_sc; o.cand_id = cand_id; o.cand_cnt = cand_cnt;
                o.ngroups = ((ntiles + S - 1) / S) * (tc::TN / tc::GROUP);
                const unsigned ut = (unsigned)((m + tc::PIPE_UT * tc::TM - 1) / (tc::PIPE_UT * tc::TM));   // CTAs along the users
                // one CTA per SM (shared memory), every CTA the same run of item tiles: the split of the items
                // that fills whole waves best (fewest chunks among the best: the A tiles load once per CTA)
                unsigned chunks = 1;
                {
                    double best = 0;
                    const unsigned cmax = (unsigned)std::max<size_t>(1, std::min<size_t>(ntiles / 32, 64));
                    for (unsigned c = 1; c <= cmax; c++) {
                        const size_t ctas = (size_t)c * ut, waves = (ctas + num_sms - 1) / num_sms;
                        const double eff = (double)ctas / (double)(waves * num_sms);
                        if (eff > best + 0.02) { best = eff; chunks = c; }
                    }
                }
                o.cand_regions = (int)chunks;
                // (4x the even share: a user's candidates may cluster in a few tiles)
                o.cand_cap = std::min(tc::CAND_CAP, tc::CAND_SLACK * tc::CAND_CAP / (int)chunks);
                tc::score_pipe_tf32_kernel<tc::MODE_GROUPMAX><<<dim3(chunks, ut), tc::PIPE_THREADS, pipe_smem>>>(
                    mapA, mapB, (int)m, n, kpad, S, pipe_stages, o);
                LAUNCHED();
                tc::select_threshold_kernel<<<(unsigned)m, 256>>>(gmax, o.ngroups, M_cand, tau);
                LAUNCHED();
                CK(cudaMemsetAsync(cand_cnt, 0, m * o.cand_regions * sizeof(int)));
                tc::score_pipe_tf32_kernel<tc::MODE_EMIT><<<dim3(chunks, ut), tc::PIPE_THREADS, pipe_smem>>>(
                    mapA, mapB, (int)m, n, kpad, 1, pipe_stages, o);
                LAUNCHED();
                tc::sort_candidates_kernel<<<(unsigned)m, 512>>>(cand_sc, cand_id, cand_cnt, o.cand_regions, o.cand_cap,
                                                                 top_sc, top_id, d_ovf);
                LAUNCHED();
                tc::rescore_select_kernel<<<(unsigned)m, 128>>>((const float*)dAsel, (const float*)dB, k, ldf, top_id,
                                                                top_sc, (size_t)tc::CAND_TOP, M_cand, 0, (int)n_top,
                                                                4e-3f, d_out_ids, d_out_sc, d_flag);
                LAUNCHED();
                CK(cudaGetLastError());
                mark("batch kernels");
                // results straight into the caller's arrays when the element types agree (they do for the
                // reference's size_t / float build); staged through page-locked blocks when those are pageable
                hfl.resize(m); hov.resize(m);
                if (sizeof(IX) == sizeof(long long)) {
                    CK(Stager::get().d2h((void*)(outp_ix + u0 * n_top), d_out_ids, m * n_top * sizeof(long long), 0));
                } else {
                    hid.resize(m * n_top);
                    CK(cudaMemcpy(hid.data(), d_out_ids, m * n_top * sizeof(long long), cudaMemcpyDeviceToHost));
                    for (size_t i = 0; i < m * n_top; i++) outp_ix[u0 * n_top + i] = (IX)hid[i];
                }
                if (outp_score) {
                    if (std::is_same<real, float>::value) {
                        CK(Stager::get().d2h((void*)(outp_score + u0 * n_top), d_out_sc, m * n_top * sizeof(float), 0));
                    } else {
                        hsc.resize(m * n_top);
                        CK(cudaMemcpy(hsc.data(), d_out_sc, m * n_top * sizeof(float), cudaMemcpyDeviceToHost));
                        for (size_t i = 0; i < m * n_top; i++) outp_score[u0 * n_top + i] = (real)hsc[i];
                    }
                }
                CK(cudaMemcpy(hfl.data(), d_flag, m * sizeof(int), cudaMemcpyDeviceToHost));
                CK(cudaMemcpy(hov.data(), d_ovf, m * sizeof(int), cudaMemcpyDeviceToHost));
                for (size_t u = 0; u < m; u++) if (hfl[u] || hov[u]) redo.push_back(u0 + u);
                g_topn_stats[0] += m;
                mark("batch results down");
            }
        } else {
            // ---- TF32 or exact scores of every item, then a segmented sort of each user's n scores ----
            // users per chunk: bound the score matrix to ~1 GiB
            size_t chunk = std::max<size_t>(1, std::min<size_t>(n_users, ((size_t)1 << 28) / std::max<size_t>(n, 1)));
            chunk = std::min<size_t>(chunk, 65535);
            if (chunk * n > (size_t)INT32_MAX) return fail("topN: chunk too large");
            real *dAsel = nullptr, *sc_in = nullptr, *sc_out = nullptr;
            int *id_in = nullptr, *id_out = nullptr, *seg = nullptr;
            long long* dusers = nullptr;
            void* tmp = nullptr;
            CK(mem.alloc(&dAsel, chunk * pitch));
            CK(mem.alloc(&sc_in, chunk * n * sizeof(real))); CK(mem.alloc(&sc_out, chunk * n * sizeof(real)));
            CK(mem.alloc(&id_in, chunk * n * sizeof(int))); CK(mem.alloc(&id_out, chunk * n * sizeof(int)));
            CK(mem.alloc(&seg, (chunk + 1) * sizeof(int)));
            CK(mem.alloc(&dusers, chunk * sizeof(long long)));
            std::vector<int> h_seg(chunk + 1);
            for (size_t u = 0; u <= chunk; u++) h_seg[u] = (int)(u * n);
            CK(cudaMemcpy(seg, h_seg.data(), (chunk + 1) * sizeof(int), cudaMemcpyHostToDevice));
            size_t tmp_bytes = 0;
            CK(cub::DeviceSegmentedRadixSort::SortPairsDescending(nullptr, tmp_bytes, sc_in, sc_out, id_in, id_out,
                                                                  (int)(chunk * n), (int)chunk, seg, seg + 1));
            CK(mem.alloc(&tmp, std::max<size_t>(tmp_bytes, 1)));
            long long* d_out_ids = nullptr;
            float* d_out_sc = nullptr;
            int* d_flag = nullptr;
            if (use_tc) {
                CK(mem.alloc(&d_out_ids, chunk * n_top * sizeof(long long)));
                CK(mem.alloc(&d_out_sc, chunk * n_top * sizeof(float)));
                CK(mem.alloc(&d_flag, chunk * sizeof(int)));
                CK(cudaFuncSetAttribute(tc::score_tiles_tf32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kpad * 1024));
            }
            std::vector<long long> hid;
            std::vector<int> h_ids, hfl;
            std::vector<real> h_sc;
            std::vector<float> hsc;
            for (size_t u0 = 0; u0 < n_users; u0 += chunk) {
                const size_t m = std::min(chunk, n_users - u0);
                if (gather_users(dA, ldf, user_ix, u0, m, dusers, dAsel)) return 1;
                if (use_tc) {
                    const dim3 tgrid((unsigned)ntiles, (unsigned)((m + tc::TM - 1) / tc::TM));
                    tc::score_tiles_tf32_kernel<<<tgrid, 128, (size_t)kpad * 1024>>>((const float*)dAsel, (int)m,
                                                                                   (const float*)dB, n, ldf, kpad,
                                                                                   (float*)sc_in, id_in);
                } else {
                    dim3 grid((unsigned)std::min<size_t>((n + 255) / 256, 1024), (unsigned)m);
                    score_items_kernel<real><<<grid, 256, (size_t)ldf * sizeof(real)>>>(dAsel, dB, n, k, ldf, sc_in, id_in);
                }
                LAUNCHED();
                if (have_excl) {
                    mask_excluded_kernel<real, IX><<<dim3(8, (unsigned)m), 256>>>(sc_in, n, dexp, dexi, u0);
                    LAUNCHED();
                }
                CK(cudaGetLastError());
                CK(cub::DeviceSegmentedRadixSort::SortPairsDescending(tmp, tmp_bytes, sc_in, sc_out, id_in, id_out,
                                                                      (int)(m * n), (int)m, seg, seg + 1));
                LAUNCHED();
                if (use_tc) {
                    // exact FP32 re-score of the best M TF32 candidates, final order, and the proof that nothing
                    // outside the candidates can reach the top n_top
                    tc::rescore_select_kernel<<<(unsigned)m, 128>>>((const float*)dAsel, (const float*)dB, k, ldf, id_out,
                                                                    (const float*)sc_out, n, M_cand, M_cand >= (int)n ? 1 : 0,
                                                                    (int)n_top, 4e-3f, d_out_ids, d_out_sc, d_flag);
                    LAUNCHED();
                    CK(cudaGetLastError());
                    hid.resize(m * n_top); hsc.resize(m * n_top); hfl.resize(m);
                    CK(cudaMemcpy(hid.data(), d_out_ids, m * n_top * sizeof(long long), cudaMemcpyDeviceToHost));
                    CK(cudaMemcpy(hsc.data(), d_out_sc, m * n_top * sizeof(float), cudaMemcpyDeviceToHost));
                    CK(cudaMemcpy(hfl.data(), d_flag, m * sizeof(int), cudaMemcpyDeviceToHost));
                    for (size_t i = 0; i < m * n_top; i++) outp_ix[u0 * n_top + i] = (IX)hid[i];
                    if (outp_score) for (size_t i = 0; i < m * n_top; i++) outp_score[u0 * n_top + i] = (real)hsc[i];
                    for (size_t u = 0; u < m; u++) if (hfl[u]) redo.push_back(u0 + u);
                    g_topn_stats[0] += m;
                    continue;
                }
                h_ids.resize(m * n_top); h_sc.resize(m * n_top);
                CK(cudaMemcpy2D(h_ids.data(), n_top * sizeof(int), id_out, n * sizeof(int), n_top * sizeof(int), m, cudaMemcpyDeviceToHost));
                CK(cudaMemcpy2D(h_sc.data(), n_top * sizeof(real), sc_out, n * sizeof(real), n_top * sizeof(real), m, cudaMemcpyDeviceToHost));
                for (size_t i = 0; i < m * n_top; i++) outp_ix[u0 * n_top + i] = (IX)h_ids[i];
                if (outp_score) memcpy(outp_score + u0 * n_top, h_sc.data(), m * n_top * sizeof(real));
            }
        }
        mem.settled = true;
    }
    mark("release");
    // users whose candidate set could not be proven complete: exact scorer, one call for all of them
    if (redo.empty()) return 0;
    const size_t R = redo.size();
    g_topn_stats[1] += R;
    std::vector<IX> ru(R), rptr(R + 1, 0), rix;
    for (size_t i = 0; i < R; i++) {
        const size_t u = redo[i];
        ru[i] = user_ix ? user_ix[u] : (IX)u;
        if (have_excl)
            for (size_t t = (size_t)excl_ptr[u]; t < (size_t)excl_ptr[u + 1]; t++) rix.push_back(excl_ix[t]);
        rptr[i + 1] = (IX)rix.size();
    }
    std::vector<IX> rout(R * n_top);
    std::vector<real> rsc(outp_score ? R * n_top : 0);
    const int rc = topn_batch_impl<real, IX>(A, B, k, ru.data(), R, dimA, have_excl ? rptr.data() : nullptr,
                                             have_excl ? (rix.empty() ? rptr.data() : rix.data()) : nullptr,
                                             rout.data(), outp_score ? rsc.data() : nullptr, n_top, n, false, rf);
    if (rc) return rc;
    for (size_t i = 0; i < R; i++) {
        memcpy(outp_ix + redo[i] * n_top, &rout[i * n_top], n_top * sizeof(IX));
        if (outp_score) memcpy(outp_score + redo[i] * n_top, &rsc[i * n_top], n_top * sizeof(real));
    }
    return 0;
}

// Batched top-N over per-user candidate lists (topn_include.cuh).  Lists up to `cap` items are ranked in
// shared memory, one CTA per user; longer ones go through CUB's segmented radix sort.  The path follows
// from each list's length.
template <class real, class IX>
static int topn_include_impl(const real* A, const real* B, int k, const IX* user_ix, size_t n_users, size_t dimA,
                             const IX* incl_ptr, const IX* incl_ix, IX* outp_ix, real* outp_score, size_t n_top,
                             size_t n, const ResidentFactors* rf = nullptr)
{
    using K = typename incl::OrderKey<real>::T;
    CK(cudaSetDevice(rf ? rf->device : env_device()));
    // argument checks of src/topN.c:121-128 per user, and the existing include rule n_top <= list length;
    // the item ids are range-checked on the device once uploaded, before any result is written
    if (n_top == 0 || !incl_ptr || !incl_ix) return 2;
    if (std::is_signed<IX>::value && (long long)incl_ptr[0] < 0) return 2;     // 4-byte (R) offsets are signed
    if (!user_ix && n_users > dimA) return 2;
    if (user_ix)
        for (size_t u = 0; u < n_users; u++)
            if ((size_t)user_ix[u] >= dimA) return 2;
    for (size_t u = 0; u < n_users; u++) {
        if (incl_ptr[u + 1] < incl_ptr[u]) return 2;
        const size_t len = (size_t)(incl_ptr[u + 1] - incl_ptr[u]);
        if (len > n || len < n_top) return 2;
    }
    if (n_users == 0) return 0;
    if (n >= 0xffffffffull) return fail("topN_include: item ids must fit 32 bits");
    const int V = RealTraits<real>::V, ldf = round_up(k, V);
    const size_t pitch = (size_t)ldf * sizeof(real), rowb = incl::row_bytes(ldf, sizeof(real));
    const size_t entry = sizeof(K) + sizeof(uint32_t);
    if (rowb + entry > SMEM_CTA_MAX) return fail("topN_include: k = %d leaves no shared memory to rank in", k);
    // shared-memory capacity: 16 K candidates in f32, 8 K in f64 (a power of two)
    int cap = std::is_same<real, float>::value ? 16384 : 8192;
    while (cap > 1 && rowb + (size_t)cap * entry > SMEM_CTA_MAX) cap >>= 1;
    auto len_of = [&](size_t u) { return (size_t)(incl_ptr[u + 1] - incl_ptr[u]); };

    // users per chunk: at most 32 768, and the chunk's lists and work arrays within a quarter of the free
    // device memory (at most 32 GB)
    size_t mem_free = 0, mem_total = 0;
    CK(cudaMemGetInfo(&mem_free, &mem_total));
    const size_t budget = std::max<size_t>((size_t)1 << 30, std::min<size_t>(mem_free / 4, (size_t)32 << 30));
    const size_t per_user = pitch + n_top * (sizeof(IX) + sizeof(real)) + 2 * sizeof(long long) + 2 * sizeof(int);
    const size_t per_long = 2 * entry;                      // double-buffered (id, key) of the segmented sort
    struct Chunk { size_t u0, u1, n_long, long_total; };
    std::vector<Chunk> chunks;
    size_t max_m = 0, max_list = 0, max_long = 0, max_long_total = 0;
    for (size_t u0 = 0; u0 < n_users;) {
        Chunk c = {u0, u0, 0, 0};
        size_t bytes = 0;
        while (c.u1 < n_users && c.u1 - u0 < 32768) {
            const size_t len = len_of(c.u1), lng = len > (size_t)cap ? len : 0;
            const size_t add = per_user + len * sizeof(IX) + lng * per_long;
            if (c.u1 > u0 && (bytes + add > budget || c.long_total + lng > (size_t)INT32_MAX)) break;
            bytes += add; c.long_total += lng; c.n_long += lng ? 1 : 0; c.u1++;
        }
        max_m = std::max(max_m, c.u1 - u0);
        max_list = std::max(max_list, (size_t)(incl_ptr[c.u1] - incl_ptr[u0]));
        max_long = std::max(max_long, c.n_long);
        max_long_total = std::max(max_long_total, c.long_total);
        chunks.push_back(c);
        u0 = c.u1;
    }

    DeviceBlocks mem;
    real *dB = nullptr, *dA = nullptr, *dAsel = nullptr, *d_sc = nullptr;
    IX *d_ix = nullptr, *d_out = nullptr;
    long long *dusers = nullptr, *dptr = nullptr;
    int *d_su = nullptr, *d_lu = nullptr, *d_seg = nullptr;
    uint32_t *id0 = nullptr, *id1 = nullptr;
    K *key0 = nullptr, *key1 = nullptr;
    void* tmp = nullptr;
    if (factors_on_device(rf, A, dimA, B, n, k, ldf, mem, &dA, &dB, "topN_include")) return 1;
    CK(mem.alloc(&dAsel, max_m * pitch));
    CK(mem.alloc(&dusers, max_m * sizeof(long long)));
    CK(mem.alloc(&dptr, (max_m + 1) * sizeof(long long)));
    CK(mem.alloc(&d_su, max_m * sizeof(int)));
    CK(mem.alloc(&d_ix, std::max<size_t>(max_list, 1) * sizeof(IX)));
    CK(mem.alloc(&d_out, max_m * n_top * sizeof(IX)));
    if (outp_score) CK(mem.alloc(&d_sc, max_m * n_top * sizeof(real)));
    int end_bit = 1;                                        // bits of the largest item id
    while (end_bit < 32 && ((n - 1) >> end_bit)) end_bit++;
    size_t tmp_bytes = 0;
    if (max_long) {
        CK(mem.alloc(&d_lu, max_long * sizeof(int)));
        CK(mem.alloc(&d_seg, (max_long + 1) * sizeof(int)));
        CK(mem.alloc(&id0, max_long_total * sizeof(uint32_t))); CK(mem.alloc(&id1, max_long_total * sizeof(uint32_t)));
        CK(mem.alloc(&key0, max_long_total * sizeof(K))); CK(mem.alloc(&key1, max_long_total * sizeof(K)));
        size_t t1 = 0, t2 = 0;
        CK(cub::DeviceSegmentedRadixSort::SortPairs(nullptr, t1, id0, id1, key0, key1, (int)max_long_total,
                                                    (int)max_long, d_seg, d_seg + 1, 0, end_bit));
        CK(cub::DeviceSegmentedRadixSort::SortPairsDescending(nullptr, t2, key1, key0, id1, id0,
                                                              (int)max_long_total, (int)max_long, d_seg, d_seg + 1));
        tmp_bytes = std::max(t1, t2);
        CK(mem.alloc(&tmp, std::max<size_t>(tmp_bytes, 1)));
    }
    // -> 0 ok, 2 a listed id outside [0, n), 1 CUDA error
    auto upload_lists = [&](const Chunk& c, bool check) -> int {
        const size_t off = (size_t)incl_ptr[c.u0], cnt = (size_t)incl_ptr[c.u1] - off;
        CK(Stager::get().h2d(d_ix, incl_ix + off, cnt * sizeof(IX), 0));
        return check ? ids_in_range(d_ix, cnt, n) : 0;
    };
    // with several chunks every list is checked before the first result is written, and uploaded again
    if (chunks.size() > 1)
        for (const Chunk& c : chunks)
            if (const int bad = upload_lists(c, true)) return bad;
    std::vector<long long> hp;
    std::vector<int> hsu, hlu, hseg;
    std::vector<std::pair<int, int>> classes;           // (capacity, users) of the path (a) launches
    for (const Chunk& c : chunks) {
        const size_t m = c.u1 - c.u0, off = (size_t)incl_ptr[c.u0];
        if (const int bad = upload_lists(c, chunks.size() == 1)) return bad;
        hp.resize(m + 1); hsu.clear(); classes.clear(); hlu.clear(); hseg.assign(1, 0);
        for (size_t i = 0; i < m; i++) {
            const size_t u = c.u0 + i, len = len_of(u);
            hp[i] = (long long)((size_t)incl_ptr[u] - off);
            if (len > (size_t)cap) { hlu.push_back((int)i); hseg.push_back(hseg.back() + (int)len); }
        }
        // path (a) by length class, so that one long list does not size every CTA's shared memory: lists up
        // to 4 K items share one launch (its 4 CTAs per SM, the register bound, fit in shared memory), longer
        // ones go by power of two up to `cap`
        for (size_t lo = 0, P = (size_t)std::min(cap, 4096);; lo = P, P <<= 1) {
            const size_t start = hsu.size();
            for (size_t i = 0; i < m; i++) {
                const size_t len = len_of(c.u0 + i);
                if (len > lo && len <= P) hsu.push_back((int)i);
            }
            if (hsu.size() > start) classes.push_back({(int)P, (int)(hsu.size() - start)});
            if (P >= (size_t)cap) break;
        }
        hp[m] = (long long)((size_t)incl_ptr[c.u1] - off);
        CK(cudaMemcpy(dptr, hp.data(), (m + 1) * sizeof(long long), cudaMemcpyHostToDevice));
        if (gather_users(dA, ldf, user_ix, c.u0, m, dusers, dAsel)) return 1;
        if (!hsu.empty()) CK(cudaMemcpy(d_su, hsu.data(), hsu.size() * sizeof(int), cudaMemcpyHostToDevice));
        for (size_t q = 0, first = 0; q < classes.size(); first += classes[q].second, q++) {
            const size_t smem = rowb + (size_t)classes[q].first * entry;
            CK(cudaFuncSetAttribute(incl::include_select_smem_kernel<real, IX>,
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            incl::include_select_smem_kernel<real, IX><<<(unsigned)classes[q].second, incl::SMEM_THREADS, smem>>>(
                dAsel, dB, k, ldf, dptr, d_ix, d_su + first, classes[q].first, (int)n_top, d_out, d_sc);
            LAUNCHED();
        }
        if (!hlu.empty()) {
            const int nl = (int)hlu.size(), total = hseg.back();
            CK(cudaMemcpy(d_lu, hlu.data(), nl * sizeof(int), cudaMemcpyHostToDevice));
            CK(cudaMemcpy(d_seg, hseg.data(), (nl + 1) * sizeof(int), cudaMemcpyHostToDevice));
            CK(cudaFuncSetAttribute(incl::include_score_long_kernel<real, IX>,
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rowb));
            incl::include_score_long_kernel<real, IX><<<dim3(64, (unsigned)nl), 256, rowb>>>(
                dAsel, dB, k, ldf, dptr, d_ix, d_lu, d_seg, id0, key0);
            LAUNCHED();
            // by item id, then stably by score: ties come out by ascending id
            CK(cub::DeviceSegmentedRadixSort::SortPairs(tmp, tmp_bytes, id0, id1, key0, key1, total, nl,
                                                        d_seg, d_seg + 1, 0, end_bit));
            CK(cub::DeviceSegmentedRadixSort::SortPairsDescending(tmp, tmp_bytes, key1, key0, id1, id0, total, nl,
                                                                  d_seg, d_seg + 1));
            LAUNCHED(); LAUNCHED();
            incl::include_emit_long_kernel<real, IX><<<(unsigned)nl, 128>>>(d_lu, d_seg, id0, key0, (int)n_top,
                                                                             d_out, d_sc);
            LAUNCHED();
        }
        CK(cudaGetLastError());
        CK(Stager::get().d2h(outp_ix + c.u0 * n_top, d_out, m * n_top * sizeof(IX), 0));
        if (outp_score) CK(Stager::get().d2h(outp_score + c.u0 * n_top, d_sc, m * n_top * sizeof(real), 0));
        CK(cudaStreamSynchronize(0));
    }
    mem.settled = true;
    return 0;
}

template <class real, class IX>
static int topn_single_impl(const real* a_vec, const real* B, int k, const IX* include_ix, size_t n_include,
                            IX* exclude_ix, size_t n_exclude, IX* outp_ix, real* outp_score, size_t n_top, size_t n)
{
    // argument checks of src/topN.c:121-128
    if (n_include == 0) include_ix = nullptr;
    if (n_exclude == 0) exclude_ix = nullptr;
    if (include_ix && exclude_ix) return 2;
    if (n_top == 0) return 2;
    if (n_exclude > n - n_top) return 2;
    if (n_include > n) return 2;
    if (include_ix) {
        // score only the listed items: gather them into a dense candidate matrix
        if (n_top > n_include) return 2;
        std::vector<real> cand(n_include * (size_t)k);
        for (size_t t = 0; t < n_include; t++)
            memcpy(&cand[t * k], B + (size_t)include_ix[t] * k, (size_t)k * sizeof(real));
        std::vector<IX> pos(n_top);
        int rc = topn_batch_impl<real, IX>(a_vec, cand.data(), k, nullptr, 1, 1, nullptr, nullptr, pos.data(),
                                           outp_score, n_top, n_include);
        if (rc) return rc;
        for (size_t t = 0; t < n_top; t++) outp_ix[t] = include_ix[(size_t)pos[t]];
        return 0;
    }
    if (exclude_ix) {
        // the reference sorts the caller's exclusion list in place (src/topN.c:159-160)
        std::sort(exclude_ix, exclude_ix + n_exclude);
        IX ptr[2] = {0, (IX)n_exclude};
        return topn_batch_impl<real, IX>(a_vec, B, k, nullptr, 1, 1, ptr, exclude_ix, outp_ix, outp_score, n_top, n);
    }
    return topn_batch_impl<real, IX>(a_vec, B, k, nullptr, 1, 1, nullptr, nullptr, outp_ix, outp_score, n_top, n);
}

extern "C" int pmf_b200_topN(int dtype, int index_bytes, const void* a_vec, const void* B, int k,
                             const void* include_ix, size_t n_include, const void* exclude_ix, size_t n_exclude,
                             void* outp_ix, void* outp_score, size_t n_top, size_t n)
{
    if (pmf_b200_device_count() <= 0) return fail("no usable CUDA device: poismf_b200 has no CPU fallback");
    return with_types(dtype, index_bytes, "topN: bad dtype/index width", [&](auto r, auto i) {
        using real = decltype(r); using IX = decltype(i);
        return topn_single_impl((const real*)a_vec, (const real*)B, k, (const IX*)include_ix, n_include, (IX*)exclude_ix,
                                n_exclude, (IX*)outp_ix, (real*)outp_score, n_top, n);
    });
}

extern "C" void pmf_b200_topN_stats(unsigned long long* tensor_core_users, unsigned long long* redone_exact, int reset)
{
    if (tensor_core_users) *tensor_core_users = g_topn_stats[0];
    if (redone_exact) *redone_exact = g_topn_stats[1];
    if (reset) g_topn_stats[0] = g_topn_stats[1] = 0;
}

// batched topN against the factors RESIDENT in a handle (after a fit, or set_factors / set_factor_rows): nothing
// but the user ids and the exclusion lists travels to the device.  In a sharded fit every rank holds full
// replicas of A and B, so each rank can rank its own share of the users right after the last sweep.
extern "C" int pmf_b200_topN_fitted(pmf_b200_handle* h, int index_bytes, const void* user_ix, size_t n_users,
                                    const void* excl_ptr, const void* excl_ix, void* outp_ix, void* outp_score,
                                    size_t n_top)
{
    if (!h) return fail("topN_fitted: null handle");
    if (pmf_b200_sync(h)) return 1;             // every row of the last half-sweep (own and peers') has landed
    ResidentFactors rf = {h->factor_ptr(0), h->factor_ptr(1), h->device, h->ldf};
    if (!rf.A || !rf.B) return fail("topN_fitted: the handle holds no factors");
    const size_t dimA = h->dimA, n = h->dimB;
    const int k = h->k;
    return with_types(h->dtype, index_bytes, "topN_fitted: bad dtype/index width", [&](auto r, auto i) {
        using real = decltype(r); using IX = decltype(i);
        return topn_batch_impl<real, IX>(nullptr, nullptr, k, (const IX*)user_ix, n_users, dimA, (const IX*)excl_ptr,
                                         (const IX*)excl_ix, (IX*)outp_ix, (real*)outp_score, n_top, n, true, &rf);
    });
}

extern "C" int pmf_b200_topN_batch(int dtype, int index_bytes, const void* A, const void* B, int k,
                                   const void* user_ix, size_t n_users, size_t dimA,
                                   const void* excl_ptr, const void* excl_ix,
                                   void* outp_ix, void* outp_score, size_t n_top, size_t n)
{
    if (pmf_b200_device_count() <= 0) return fail("no usable CUDA device: poismf_b200 has no CPU fallback");
    return with_types(dtype, index_bytes, "topN_batch: bad dtype/index width", [&](auto r, auto i) {
        using real = decltype(r); using IX = decltype(i);
        return topn_batch_impl((const real*)A, (const real*)B, k, (const IX*)user_ix, n_users, dimA, (const IX*)excl_ptr,
                               (const IX*)excl_ix, (IX*)outp_ix, (real*)outp_score, n_top, n);
    });
}

extern "C" int pmf_b200_topN_batch_include(int dtype, int index_bytes, const void* A, const void* B, int k,
                                           const void* user_ix, size_t n_users, size_t dimA,
                                           const void* incl_ptr, const void* incl_ix,
                                           void* outp_ix, void* outp_score, size_t n_top, size_t n)
{
    if (pmf_b200_device_count() <= 0) return fail("no usable CUDA device: poismf_b200 has no CPU fallback");
    return with_types(dtype, index_bytes, "topN_batch_include: bad dtype/index width", [&](auto r, auto i) {
        using real = decltype(r); using IX = decltype(i);
        return topn_include_impl((const real*)A, (const real*)B, k, (const IX*)user_ix, n_users, dimA, (const IX*)incl_ptr,
                                 (const IX*)incl_ix, (IX*)outp_ix, (real*)outp_score, n_top, n);
    });
}

extern "C" int pmf_b200_topN_fitted_include(pmf_b200_handle* h, int index_bytes, const void* user_ix, size_t n_users,
                                            const void* incl_ptr, const void* incl_ix, void* outp_ix, void* outp_score,
                                            size_t n_top)
{
    if (!h) return fail("topN_fitted_include: null handle");
    if (pmf_b200_sync(h)) return 1;
    ResidentFactors rf = {h->factor_ptr(0), h->factor_ptr(1), h->device, h->ldf};
    if (!rf.A || !rf.B) return fail("topN_fitted_include: the handle holds no factors");
    const size_t dimA = h->dimA, n = h->dimB;
    const int k = h->k;
    return with_types(h->dtype, index_bytes, "topN_fitted_include: bad dtype/index width", [&](auto r, auto i) {
        using real = decltype(r); using IX = decltype(i);
        return topn_include_impl<real, IX>(nullptr, nullptr, k, (const IX*)user_ix, n_users, dimA, (const IX*)incl_ptr,
                                           (const IX*)incl_ix, (IX*)outp_ix, (real*)outp_score, n_top, n, &rf);
    });
}

// ---- batched top-N for new users: fold them in against fixed item factors, then rank them ------------------------
// = PoisMF.topN_new / predict_factors (poismf/__init__.py:502-576, :977-1075) for many users in one call: the rows
// are solved by factors_multiple (src/pred.c:66-199) on a second handle that binds the item factors in place, and
// ranked by topn_batch_impl / topn_include_impl straight from the device.

// Bsum = column sums of B + l1 (when > 0), Amean = column means of A, k host reals each (the attributes PoisMF keeps
// after a fit, poismf/__init__.py:438-439).  Fixed-order sums (launch_column_sums): the same bits on every call and on
// every replica of a sharded fit.
template <class real>
static int fit_stats_impl(const real* dA, size_t dimA, const real* dB, size_t dimB, int k, int ldf, int device,
                          double l1, real* Bsum, real* Amean)
{
    CK(cudaSetDevice(device));
    int num_sms = 148;
    CK(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, device));
    const int n_partial = num_sms * 4;
    DeviceBlocks mem;
    real *partial = nullptr, *d_out = nullptr;
    CK(mem.alloc(&partial, (size_t)n_partial * ldf * sizeof(real)));
    CK(mem.alloc(&d_out, 2 * (size_t)k * sizeof(real)));
    ColsumFinal<real> fin = {};
    fin.l1 = (real)l1;
    if (launch_column_sums(dB, dimB, k, ldf, fin, false, partial, n_partial, d_out, (cudaStream_t)0)) return 1;
    fin.l1 = (real)0;
    if (launch_column_sums(dA, dimA, k, ldf, fin, false, partial, n_partial, d_out + k, (cudaStream_t)0)) return 1;
    std::vector<real> h(2 * (size_t)k);
    CK(cudaMemcpy(h.data(), d_out, 2 * (size_t)k * sizeof(real), cudaMemcpyDeviceToHost));
    mem.settled = true;
    for (int c = 0; c < k; c++) {
        if (Bsum) Bsum[c] = h[c];
        if (Amean) Amean[c] = h[k + c] / (real)dimA;
    }
    return 0;
}

// -> 2 when the arguments of a new-user call are invalid (checked on the host before anything reaches the device),
// else 0.  The fold-in ids are range-checked here: they are narrowed to int32 on upload and gather rows of B.
template <class IX>
static int check_new_users(const void* Xr, const IX* Xr_indptr, const IX* Xr_indices, size_t n_new, size_t n,
                           const pmf_b200_params* p, const void* excl_ptr, const void* excl_ix, const void* incl_ptr,
                           const void* incl_ix, const void* outp_ix, size_t n_top, const void* A_out)
{
    if (!p || p->early_stop) return 2;
    if (p->method != PMF_PG && p->method != PMF_CG && p->method != PMF_TNCG) return 2;
    if (!outp_ix && !A_out) return 2;
    if ((excl_ptr || excl_ix) && (incl_ptr || incl_ix)) return 2;
    if (outp_ix && (n_top == 0 || n_top > n)) return 2;
    if (n_new > (size_t)INT32_MAX || n > (size_t)INT32_MAX) return 2;
    if (n_new == 0) return 0;
    if (!Xr_indptr) return 2;
    if (std::is_signed<IX>::value && (long long)Xr_indptr[0] < 0) return 2;
    for (size_t u = 0; u < n_new; u++)
        if (Xr_indptr[u + 1] < Xr_indptr[u]) return 2;
    const size_t nnz = (size_t)(Xr_indptr[n_new] - Xr_indptr[0]);
    if (nnz && (!Xr || !Xr_indices)) return 2;
    size_t top = 0;                       // a negative id of a signed type is a huge size_t
    for (size_t t = 0; t < nnz; t++) top = std::max(top, (size_t)Xr_indices[t]);
    if (nnz && top >= n) return 2;
    return 0;
}

// The fold-in and the ranking, B = dB [n x ldf] on `device`.  Bsum_used = Bsum + l1 (in real, when l1 > 0).
template <class real, class IX>
static int topn_new_impl(real* dB, size_t n, int k, int device, const real* Bsum, const real* Amean, double l1,
                         const real* Xr, const IX* Xr_indptr, const IX* Xr_indices, size_t n_new, const pmf_b200_params& p,
                         const IX* excl_ptr, const IX* excl_ix, const IX* incl_ptr, const IX* incl_ix, IX* outp_ix,
                         real* outp_score, size_t n_top, real* A_out)
{
    if (n_new == 0) return 0;
    std::vector<real> bs(Bsum, Bsum + k);
    const real l1r = (real)l1;
    if (l1r > (real)0) for (int c = 0; c < k; c++) bs[c] += l1r;
    HandleT<real> fold;                   // the new users' rows against the bound B: only A and the CSR are allocated
    fold.dtype = std::is_same<real, float>::value ? PMF_F32 : PMF_F64;
    fold.device = device; fold.dimA = n_new; fold.dimB = n; fold.k = k;
    if (fold.init(dB)) return 1;
    const size_t nnz = (size_t)(Xr_indptr[n_new] - Xr_indptr[0]);
    if (fold.set_matrix(PMF_SIDE_CSR, Xr, Xr_indptr, Xr_indices, nnz, (int)sizeof(IX), 0, n_new)) return 1;
    pmf_b200_params q = p;                // as pmf_b200_factors_multiple passes them; reuse_prev is reuse_mean
    q.l1_reg = 0; q.early_stop = 0; q.reuse_prev = 0;
    if (fold.factors_multiple(nullptr, bs.data(), Amean, q, p.reuse_prev)) return 1;
    if (outp_ix) {
        const ResidentFactors rf = {fold.A, dB, device, fold.ldf};
        const int rc = (incl_ptr || incl_ix)
            ? topn_include_impl<real, IX>(nullptr, nullptr, k, nullptr, n_new, n_new, incl_ptr, incl_ix, outp_ix,
                                          outp_score, n_top, n, &rf)
            : topn_batch_impl<real, IX>(nullptr, nullptr, k, nullptr, n_new, n_new, excl_ptr, excl_ix, outp_ix,
                                        outp_score, n_top, n, true, &rf);
        if (rc) return rc;
    }
    return A_out ? fold.get_factors(A_out, nullptr) : 0;
}

extern "C" int pmf_b200_topN_new_batch(int dtype, int index_bytes, const void* B, const void* Bsum, const void* Amean,
                                       int k, size_t n, const void* Xr, const void* Xr_indptr, const void* Xr_indices,
                                       size_t n_new, const pmf_b200_params* p,
                                       const void* excl_ptr, const void* excl_ix, const void* incl_ptr,
                                       const void* incl_ix, void* outp_ix, void* outp_score, size_t n_top, void* A_out)
{
    if (pmf_b200_device_count() <= 0) return fail("no usable CUDA device: poismf_b200 has no CPU fallback");
    return with_types(dtype, index_bytes, "topN_new_batch: bad dtype/index width", [&](auto r, auto i) {
        using real = decltype(r); using IX = decltype(i);
        if (!B || !Bsum || !Amean || k < 1 || k > 256) return 2;
        if (const int bad = check_new_users<IX>(Xr, (const IX*)Xr_indptr, (const IX*)Xr_indices, n_new, n, p, excl_ptr,
                                                excl_ix, incl_ptr, incl_ix, outp_ix, n_top, A_out)) return bad;
        if (n_new == 0) return 0;
        const int device = env_device();
        CK(cudaSetDevice(device));
        DeviceBlocks mem;
        real* dB = nullptr;
        bool resident = false;
        if (upload_rows<real>(&dB, (const real*)B, n, k, round_up(k, RealTraits<real>::V), &resident, true)) return 1;
        if (!resident) mem.adopt(dB);
        const int rc = topn_new_impl<real, IX>(dB, n, k, device, (const real*)Bsum, (const real*)Amean, p->l1_reg,
                                               (const real*)Xr, (const IX*)Xr_indptr, (const IX*)Xr_indices, n_new, *p,
                                               (const IX*)excl_ptr, (const IX*)excl_ix, (const IX*)incl_ptr,
                                               (const IX*)incl_ix, (IX*)outp_ix, (real*)outp_score, n_top, (real*)A_out);
        mem.settled = rc != 1;
        return rc;
    });
}

extern "C" int pmf_b200_topN_new_fitted(pmf_b200_handle* h, int index_bytes, const void* Bsum, const void* Amean,
                                        const void* Xr, const void* Xr_indptr, const void* Xr_indices, size_t n_new,
                                        const pmf_b200_params* p,
                                        const void* excl_ptr, const void* excl_ix, const void* incl_ptr,
                                        const void* incl_ix, void* outp_ix, void* outp_score, size_t n_top, void* A_out)
{
    if (!h) return fail("topN_new_fitted: null handle");
    if (pmf_b200_sync(h)) return 1;             // every row of the last half-sweep (own and peers') has landed
    return with_types(h->dtype, index_bytes, "topN_new_fitted: bad dtype/index width", [&](auto r, auto i) {
        using real = decltype(r); using IX = decltype(i);
        const size_t n = h->dimB;
        const int k = h->k;
        if (const int bad = check_new_users<IX>(Xr, (const IX*)Xr_indptr, (const IX*)Xr_indices, n_new, n, p, excl_ptr,
                                                excl_ix, incl_ptr, incl_ix, outp_ix, n_top, A_out)) return bad;
        real* dB = (real*)h->factor_ptr(1);
        if (!dB) return fail("topN_new_fitted: the handle holds no factors");
        std::vector<real> stats;
        if (!Bsum || !Amean) {
            stats.resize(2 * (size_t)k);
            if (fit_stats_impl<real>((const real*)h->factor_ptr(0), h->dimA, dB, n, k, h->ldf, h->device, 0.0,
                                     stats.data(), stats.data() + k)) return 1;
        }
        return topn_new_impl<real, IX>(dB, n, k, h->device, Bsum ? (const real*)Bsum : stats.data(),
                                       Amean ? (const real*)Amean : stats.data() + k, p->l1_reg, (const real*)Xr,
                                       (const IX*)Xr_indptr, (const IX*)Xr_indices, n_new, *p, (const IX*)excl_ptr,
                                       (const IX*)excl_ix, (const IX*)incl_ptr, (const IX*)incl_ix, (IX*)outp_ix,
                                       (real*)outp_score, n_top, (real*)A_out);
    });
}

extern "C" int pmf_b200_fit_stats(pmf_b200_handle* h, double l1_reg, void* Bsum_out, void* Amean_out)
{
    if (!h) return fail("fit_stats: null handle");
    if (!Bsum_out && !Amean_out) return 2;
    if (pmf_b200_sync(h)) return 1;
    return with_types(h->dtype, 8, "fit_stats: bad dtype", [&](auto r, auto) {
        using real = decltype(r);
        return fit_stats_impl<real>((const real*)h->factor_ptr(0), h->dimA, (const real*)h->factor_ptr(1), h->dimB,
                                    h->k, h->ldf, h->device, l1_reg, (real*)Bsum_out, (real*)Amean_out);
    });
}
