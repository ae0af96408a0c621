/* poismf_b200 — C ABI of the B200-native poismf hot path (libpoismf_b200.so).
 *
 * Plain C symbols, plain pointers and sizes: this is the boundary a maintainer of
 * david-cortes/poismf binds instead of compiling src/poismf.c, src/pred.c and
 * src/topN.c into the wrapper (see INTEGRATION.md).  Every entry point names the
 * reference interface it replaces.
 *
 * Value types:  PMF_F32 <-> real_t=float  (-DUSE_FLOAT, src/poismf.h:100-108)
 *               PMF_F64 <-> real_t=double (src/poismf.h:91-99)
 * Index types:  index_bytes = 8 <-> sparse_ix=size_t (Python, src/poismf.h:76)
 *               index_bytes = 4 <-> sparse_ix=int    (R,      src/poismf.h:86)
 *
 * Return codes follow the reference: 0 ok, 1 out of memory / CUDA failure,
 * 2 interrupted (run) or invalid arguments (topN).  There is no CPU fallback: if
 * no CUDA device is usable every compute entry point fails with 1 and a message
 * on stderr.
 */
#ifndef POISMF_B200_H
#define POISMF_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum { PMF_F32 = 0, PMF_F64 = 1 };
enum { PMF_TNCG = 1, PMF_CG = 2, PMF_PG = 3 };          /* == Method, src/poismf.h:225 */
enum { PMF_SIDE_CSR = 0, PMF_SIDE_CSC = 1 };            /* CSR drives the A update, CSC the B update */

/* Numerics-mode flags (argument `flags`, or env POISMF_B200_FLAGS for the drop-in calls) */
enum {
    PMF_FLAG_STRICT    = 1,  /* sequential sums, no FMA: mimics the reference built with naive BLAS */
    PMF_FLAG_NO_CACHED = 2,  /* cg: recompute every line-search objective from the factors        */
    PMF_FLAG_NO_LOCKSTEP = 4 /* keep the heaviest rows on per-row teams: results then do not depend on how rows are
                                sharded over GPUs (the lock-step path sums a heavy row's non-zeros in an order that
                                depends on which other heavy rows the device holds; it is reproducible run to run) */
};

/* Hyper-parameters of a fit; same meaning as the arguments of run_poismf
 * (src/poismf.h:226-233, documented at src/poismf.c:407-434). */
typedef struct pmf_b200_params {
    double l2_reg, l1_reg, w_mult, step_size;
    int method;            /* PMF_TNCG / PMF_CG / PMF_PG */
    int limit_step;
    size_t numiter, maxupd;
    int early_stop, reuse_prev;
    int flags;             /* PMF_FLAG_* */
} pmf_b200_params;

typedef struct pmf_b200_handle pmf_b200_handle;

/* ---- library ------------------------------------------------------------ */
int         pmf_b200_device_count(void);          /* 0 when no usable CUDA device */
const char* pmf_b200_last_error(void);            /* message of the last failure on this thread */
uint64_t    pmf_b200_kernel_launches(void);       /* kernels launched by this library so far */

/* ---- device-resident fit (what run_poismf does between its H2D and D2H) --- */
/* A handle owns the device copy of one problem: factors A [dimA x k], B [dimB x k]
 * (stored with a row stride of ldf = k rounded up to 16 bytes, pads zero) and the
 * count matrix in CSR and CSC.  For sharded fits a handle holds only the rows
 * [row_begin,row_end) of each compressed matrix but full replicas of A and B. */
pmf_b200_handle* pmf_b200_create(int dtype, size_t dimA, size_t dimB, size_t k, int device);
void pmf_b200_destroy(pmf_b200_handle* h);
int  pmf_b200_ldf(const pmf_b200_handle* h);       /* device row stride of A and B, in elements */

/* Upload one orientation of X from HOST arrays laid out as the reference expects
 * (values real_t[nnz]; indptr sparse_ix[n_rows+1] relative to the first local row;
 * indices sparse_ix[nnz]).  row_begin/n_rows select the shard (0, dim for a full fit). */
int pmf_b200_set_matrix(pmf_b200_handle* h, int side, const void* values, const void* indptr,
                        const void* indices, size_t nnz, int index_bytes,
                        size_t row_begin, size_t n_rows);
int pmf_b200_set_factors(pmf_b200_handle* h, const void* A_host, const void* B_host);  /* H2D, dense [dim x k] */
int pmf_b200_get_factors(pmf_b200_handle* h, void* A_host, void* B_host);              /* D2H, dense [dim x k] */
/* Use caller-owned DEVICE buffers ([dim x ldf], pads zero) for A and B, e.g. torch tensors. */
int pmf_b200_bind_factors(pmf_b200_handle* h, void* A_dev, void* B_dev);
void* pmf_b200_factor_ptr(pmf_b200_handle* h, int which /*0=A,1=B*/);
int pmf_b200_set_stream(pmf_b200_handle* h, void* cuda_stream);   /* e.g. torch's current stream */

/* numiter full alternating sweeps (src/poismf.c:506-608) on the device copy.
 * Asynchronous on the handle's stream except for tncg early stopping. */
int pmf_b200_sweeps(pmf_b200_handle* h, const pmf_b200_params* p);
/* One half-sweep, for the sharding layer (poismf_b200/sharding.py): updates the
 * local rows of B (side=CSC) or A (side=CSR).  `step_size` is the CURRENT pg step
 * (the caller applies the halving of src/poismf.c:532) and `cnst_div` the sweep's
 * 1/(1+2*l2*step) of src/poismf.c:511; the side selects pg's column-sum scaling
 * (once on the B side, :523-524; twice on the A side, :573-577).
 * *n_unchanged (may be NULL) receives the numerator of tncg's early-stop test: the
 * number of local rows that moved less than 1e-4 (src/poismf.c:393-396). */
int pmf_b200_half_sweep(pmf_b200_handle* h, int side, const pmf_b200_params* p, double step_size,
                        double cnst_div, unsigned long long* n_unchanged);
int pmf_b200_sync(pmf_b200_handle* h);

/* ---- fused "update rows -> refresh every replica" over NVLink peer memory ----
 * Sharded fits keep a replica of A and B on every GPU.  Instead of an NCCL collective after
 * each half-sweep, the row kernels store every freshly solved row straight into the peers'
 * replicas (plain stores to peer-mapped pointers; one process per GPU, so the mapping goes
 * through CUDA IPC).  Usage: every rank exports its two factor buffers (64-byte handles), the
 * handles are all-gathered by the caller (e.g. torch.distributed), every rank imports them.
 * Completion is signalled ON THE DEVICE when the ranks also exchange `which = 2`, their epoch
 * slots: after its half-sweep a rank writes the half-sweep's number into its slot on every
 * rank, and the next half-sweep's kernels are preceded by a one-warp kernel that waits until
 * all slots have reached it.  The host then enqueues whole fits without waiting between
 * half-sweeps (without the slots the caller needs a stream sync + a process barrier there).
 * pmf_b200_sync returns 1 if a peer failed to arrive within ~30 s. */
#define PMF_B200_IPC_HANDLE_BYTES 64
int pmf_b200_ipc_export(pmf_b200_handle* h, int which /*0=A,1=B,2=epoch slots*/, void* handle_out);
/* handles: n_ranks x 64 bytes in rank order (own entry ignored).  n_ranks <= 8. */
int pmf_b200_ipc_import(pmf_b200_handle* h, int which, const void* handles, int n_ranks, int self_rank);
/* Rows [row_begin, row_begin + n_rows) of A (which = 0) or B (1), k reals per row in host memory, into the
 * own replica and — over NVLink, through the mappings imported above — into every peer's: the ranks of a
 * sharded fit each upload 1/N of the initial factors (poismf/__init__.py:419-425 draws them on the host). */
int pmf_b200_set_factor_rows(pmf_b200_handle* h, int which, const void* rows, size_t row_begin, size_t n_rows);

/* Per-launch device timing of the row kernels (CUDA events on the handle's stream),
 * for bench.py's roofline line: one entry per (side, row bin). */
typedef struct pmf_b200_bin_profile {
    int side;                  /* PMF_SIDE_CSR / PMF_SIDE_CSC */
    int block_team;            /* < 0: -lanes per row (sub-warp / warp teams); 1: CTA per row; 2..16: CTAs per row (cluster);
                                  100 + w: register-tile kernel with w warps per row; 200: the heaviest rows, lock-step path */
    int cap;                   /* staged tile capacity (0: tile read from global memory) */
    int nrows;                 /* rows in the bin */
    unsigned long long nnz;    /* non-zeros in the bin */
    unsigned long long launches;
    double ms;                 /* summed device time of those launches */
} pmf_b200_bin_profile;
int pmf_b200_set_profiling(pmf_b200_handle* h, int on);                       /* also clears the counters */
int pmf_b200_get_profile(pmf_b200_handle* h, pmf_b200_bin_profile* out, int max_entries);  /* returns #entries */

/* ---- drop-in entry points (host pointers in, host pointers out) ---------- */
/* Replaces run_poismf, src/poismf.c:435-632 (prototype src/poismf.h:226-233).  Stateless like the
 * reference: everything is uploaded, swept and downloaded inside the call.  The transfers are
 * pipelined against the half-sweeps (CSR goes up behind the first B half-sweep, B comes down behind
 * the last A half-sweep), pageable buffers are staged by host threads, and the device blocks go
 * back to a per-process cache (pmf_b200_release_cache).  With env POISMF_B200_CACHE_X=1 the
 * uploaded matrix is kept for the next call on the same arrays. */
int pmf_b200_run_poismf(int dtype, int index_bytes,
                        void* A, const void* Xr, const void* Xr_indptr, const void* Xr_indices,
                        void* B, const void* Xc, const void* Xc_indptr, const void* Xc_indices,
                        size_t dimA, size_t dimB, size_t k,
                        double l2_reg, double l1_reg, double w_mult, double step_size,
                        int method, int limit_step, size_t numiter, size_t maxupd,
                        int early_stop, int reuse_prev, int handle_interrupt, int flags);

/* Replaces factors_multiple, src/pred.c:66-199 (prototype src/poismf.h:270-280): factors for dimA
 * NEW rows given in CSR, with B [dimB x k] and Bsum (column sums of B, l1 already added) fixed.
 * A [dimA x k] is output only.  dimB is needed for the device copy of B (the reference takes none). */
int pmf_b200_factors_multiple(int dtype, int index_bytes, void* A, const void* B, const void* Bsum,
                              const void* Amean, const void* Xr, const void* Xr_indptr, const void* Xr_indices,
                              int k, size_t dimA, size_t dimB,
                              double l2_reg, double w_mult, double step_size, size_t niter, size_t maxupd,
                              int method, int limit_step, int reuse_mean, int flags);

/* Front-end ingestion on the device (the reference does it on the host with SciPy,
 * poismf/__init__.py:376-416: coo.tocsr() and coo.tocsc()).  `rows`, `cols` [n_entries] ids at
 * index_bytes width, `vals` [n_entries] counts, any order, duplicates allowed (they are summed).
 * pmf_b200_fit_coo = that conversion + run_poismf's sweeps with the matrix never leaving the device;
 * A [dimA x k] and B [dimB x k] are in/out host arrays.  Returns run_poismf's codes, or 2 when an id
 * is outside [0, dim).  pmf_b200_coo_to_csr_csc is the conversion alone, into caller arrays sized
 * n_entries (values, ids) and dim+1 (offsets); *nnz_out = entries stored after summing duplicates. */
int pmf_b200_fit_coo(int dtype, int index_bytes, void* A, void* B, const void* rows, const void* cols,
                     const void* vals, size_t n_entries, size_t dimA, size_t dimB, size_t k,
                     double l2_reg, double l1_reg, double w_mult, double step_size,
                     int method, int limit_step, size_t numiter, size_t maxupd,
                     int early_stop, int reuse_prev, int flags);
int pmf_b200_coo_to_csr_csc(int dtype, int index_bytes, const void* rows, const void* cols, const void* vals,
                            size_t n_entries, size_t dimA, size_t dimB, void* Xr, void* Xr_indptr,
                            void* Xr_indices, void* Xc, void* Xc_indptr, void* Xc_indices, size_t* nnz_out);

/* Replaces factors_single, src/pred.c:201-304 (prototype src/poismf.h:281-289): factors of ONE new row
 * (nnz counts X at item ids X_ind) by tncg, with B and Bsum (old l1 already added) fixed; l1_new - l1_old
 * is added to Bsum when positive.  `out` [k] is output only; nnz == 0 gives zeros.  Same math as
 * pmf_b200_factors_multiple on a one-row matrix (only the nnz rows of B the ids name are uploaded). */
int pmf_b200_factors_single(int dtype, int index_bytes, void* out, size_t k, const void* Amean, int reuse_mean,
                            const void* X, const void* X_ind, size_t nnz, const void* B, const void* Bsum,
                            int maxupd, double l2_reg, double l1_new, double l1_old, double w_mult, int flags);

/* Replaces predict_multiple, src/pred.c:42-64 (prototype src/poismf.h:250-257). */
int pmf_b200_predict_multiple(int dtype, int index_bytes, void* out, const void* A, const void* B,
                              const void* ixA, const void* ixB, size_t n, int k,
                              size_t dimA, size_t dimB);

/* Replaces topN, src/topN.c:112-284 (prototype src/poismf.h:240-247) for ONE user. */
int pmf_b200_topN(int dtype, int index_bytes, const void* a_vec, const void* B, int k,
                  const void* include_ix, size_t n_include, const void* exclude_ix, size_t n_exclude,
                  void* outp_ix, void* outp_score, size_t n_top, size_t n);

/* Batched top-N: scores `n_users` rows of A (selected by user_ix, or rows 0..n_users-1
 * when NULL) against all n items of B, excluding per user the item ids
 * excl_ix[excl_ptr[u] .. excl_ptr[u+1]) (both may be NULL).  Output is
 * [n_users x n_top] item ids (sparse_ix) and optionally scores.  No reference
 * equivalent: the reference loops topN per user (poismf/__init__.py:914-923). */
int pmf_b200_topN_batch(int dtype, int index_bytes, const void* A, const void* B, int k,
                        const void* user_ix, size_t n_users, size_t dimA,
                        const void* excl_ptr, const void* excl_ix,
                        void* outp_ix, void* outp_score, size_t n_top, size_t n);

/* The same ranking against the factors RESIDENT in a handle (after pmf_b200_sweeps / half_sweep, set_factors or
 * set_factor_rows): A = the handle's dimA x k user factors, B = its dimB x k item factors; only the user ids and
 * the exclusion lists are uploaded.  The call first waits for the handle's stream and, in a sharded fit, for
 * the peers' rows of the last half-sweep (like pmf_b200_sync), so every rank of a sharded fit can rank its own
 * share of the users against its replicas right after the last sweep (PoisMF.fit -> topN without a round trip
 * of the factors through the host, poismf/__init__.py:440,914-923).  Same return codes as pmf_b200_topN_batch. */
int pmf_b200_topN_fitted(pmf_b200_handle* h, int index_bytes, const void* user_ix, size_t n_users,
                         const void* excl_ptr, const void* excl_ix,
                         void* outp_ix, void* outp_score, size_t n_top);

/* Batched top-N where user u ranks ONLY the items incl_ix[incl_ptr[u] .. incl_ptr[u+1]) (any order; duplicates are
 * ranked as given, like src/topN.c).  Users are selected by user_ix, or rows 0..n_users-1 when NULL.  Scores are
 * the exact sequential, unfused dots <a_u, B_j> (the bits of the reference's strict build); the ranking is
 * descending score, ties by ascending item id.  Output [n_users x n_top] item ids and optionally scores.
 * Returns 2, before any result is written, when n_top == 0, a user id is >= dimA, incl_ptr is not monotone,
 * a list is longer than n or shorter than n_top, or a listed id is >= n; 1 on a CUDA failure.  No reference
 * equivalent: the reference loops topN(include) per user. */
int pmf_b200_topN_batch_include(int dtype, int index_bytes, const void* A, const void* B, int k,
                                const void* user_ix, size_t n_users, size_t dimA,
                                const void* incl_ptr, const void* incl_ix,
                                void* outp_ix, void* outp_score, size_t n_top, size_t n);

/* The same against the factors resident in a fit handle (waits like pmf_b200_topN_fitted). */
int pmf_b200_topN_fitted_include(pmf_b200_handle* h, int index_bytes, const void* user_ix, size_t n_users,
                                 const void* incl_ptr, const void* incl_ix,
                                 void* outp_ix, void* outp_score, size_t n_top);

/* Batched top-N for NEW users (PoisMF.topN_new / predict_factors for many users at once, poismf/__init__.py:502-576,
 * :977-1075): the n_new users given as CSR rows (values real_t[nnz], indptr sparse_ix[n_new+1], indices
 * sparse_ix[nnz]) are folded in against the fixed item factors B [n x k], then ranked against B.
 * Fold-in = factors_multiple (src/pred.c:66-199) with the parameters of *p: method, numiter (niter), maxupd,
 * step_size, limit_step, l2_reg, w_mult, flags as there; reuse_prev = reuse_mean; early_stop must be 0; the column
 * sums used are Bsum + l1_reg (in real_t, added when l1_reg > 0).  A caller holding the model's Bsum (old l1 already
 * in it) passes the positive part of l1_new - l1_old as l1_reg.  PoisMF.topN_new is method PMF_TNCG, numiter 1,
 * step_size 0, limit_step 0.  Rows without non-zeros get zero factors.  The new users' factors stay on the device.
 * Ranking = pmf_b200_topN_batch of those rows (same routes, ids and scores), or with include lists
 * pmf_b200_topN_batch_include.  Exclusion lists (excl_ptr/excl_ix) or include lists (incl_ptr/incl_ix) per new user
 * are optional, not both; nothing is excluded implicitly (pass the fold-in CSR's indptr/indices as the exclusion lists
 * to leave out the users' own items).  Bsum, Amean: k reals each, required.  outp_ix [n_new x n_top] required,
 * outp_score optional, A_out [n_new x k] optional.  B goes through the POISMF_B200_CACHE_FACTORS cache.
 * Returns 2, before any output is written, when Xr_indptr is not monotone, a fold-in item id is >= n, early_stop is
 * set or the method is unknown, both kinds of lists are given, n_top is 0 or > n, a list fails the checks of the
 * two ranking entries, Bsum or Amean is NULL, or no output is requested; 1 on a CUDA failure. */
int pmf_b200_topN_new_batch(int dtype, int index_bytes, const void* B, const void* Bsum, const void* Amean,
                            int k, size_t n, const void* Xr, const void* Xr_indptr, const void* Xr_indices,
                            size_t n_new, const pmf_b200_params* p,
                            const void* excl_ptr, const void* excl_ix, const void* incl_ptr, const void* incl_ix,
                            void* outp_ix, void* outp_score, size_t n_top, void* A_out);
/* The same against the factors resident in a fit handle: B = the handle's item factors, read in place (nothing but
 * the new users' rows, k reals of statistics and the lists travels to the device).  Bsum / Amean may be NULL: they
 * are then computed on the device from the handle's B and A as pmf_b200_fit_stats(h, 0, ...) does.  outp_ix may be
 * NULL: fold-in only (PoisMF.transform against a resident fit) into A_out; at least one of outp_ix / A_out.  Waits
 * like pmf_b200_topN_fitted first; the handle's factors, matrices and plans are left untouched. */
int pmf_b200_topN_new_fitted(pmf_b200_handle* h, int index_bytes, const void* Bsum, const void* Amean,
                             const void* Xr, const void* Xr_indptr, const void* Xr_indices, size_t n_new,
                             const pmf_b200_params* p,
                             const void* excl_ptr, const void* excl_ix, const void* incl_ptr, const void* incl_ix,
                             void* outp_ix, void* outp_score, size_t n_top, void* A_out);
/* Column sums of the handle's B plus l1_reg (when > 0) into Bsum_out, column means of its A into Amean_out (k reals
 * each, either may be NULL): the Bsum / Amean attributes PoisMF keeps after a fit (poismf/__init__.py:438-439).
 * Summed in a fixed order on the device, so every call and every replica of a sharded fit gives the same bits. */
int pmf_b200_fit_stats(pmf_b200_handle* h, double l1_reg, void* Bsum_out, void* Amean_out);

/* Counters of the calling thread's topN calls: users scored by the tensor-core candidate scorer,
 * and how many of those had to be redone by the exact scorer because the TF32 error bound could
 * not prove their candidate set complete. */
void pmf_b200_topN_stats(unsigned long long* tensor_core_users, unsigned long long* redone_exact, int reset);

/* Device blocks released by the calls above are cached per process for the next call (the reference's
 * API is stateless, so every call would otherwise pay a dozen cudaMalloc/cudaFree round trips; env
 * POISMF_B200_POOL_MB caps the idle bytes, 0 disables, default half of the device's memory).
 * This returns all idle blocks to the driver; result: bytes released. */
size_t pmf_b200_release_cache(void);

#ifdef __cplusplus
}
#endif
#endif /* POISMF_B200_H */
