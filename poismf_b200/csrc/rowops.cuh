// poismf_b200 — per-row evaluation primitives.
//
// A row's sub-problem touches the gathered rows {F[j] : j in the row's non-zeros}
// ("tile") many times (once per objective/gradient evaluation).  The tile is
// staged ONCE per half-sweep into shared memory with 16-byte cp.async copies
// (row stride `kp` chosen so that 16-byte accesses by consecutive lanes to
// consecutive tile rows are bank-conflict free), and every evaluation then runs
// out of shared memory:
//   dots  : one lane per non-zero, sequential over the k components
//           (== the reference's cblas_tdot per non-zero, src/poismf.c:204,219,259)
//   gaxpy : one lane per 16-byte component chunk, sequential over the non-zeros
//           (== the reference's chain of cblas_taxpy into grad, :218-221,:260-261)
// Rows whose tile does not fit the team's shared-memory slice run the same code
// reading the factor rows straight from global memory / L2 (tile == nullptr).
#pragma once
#include <type_traits>
#include "common.cuh"

namespace pmf {

template <class real> struct Vec16;
template <> struct Vec16<float> { using type = float4; };
template <> struct Vec16<double> { using type = double2; };

PMF_DEVINL float vdot4(const float4& a, const float4& b, float s)
{
    s = fmaf(a.x, b.x, s); s = fmaf(a.y, b.y, s); s = fmaf(a.z, b.z, s); s = fmaf(a.w, b.w, s);
    return s;
}
PMF_DEVINL double vdot4(const double2& a, const double2& b, double s)
{
    s = fma(a.x, b.x, s); s = fma(a.y, b.y, s);
    return s;
}
PMF_DEVINL void vfma(float4& acc, float c, const float4& b)
{
    acc.x = fmaf(c, b.x, acc.x); acc.y = fmaf(c, b.y, acc.y);
    acc.z = fmaf(c, b.z, acc.z); acc.w = fmaf(c, b.w, acc.w);
}
PMF_DEVINL void vfma(double2& acc, double c, const double2& b)
{
    acc.x = fma(c, b.x, acc.x); acc.y = fma(c, b.y, acc.y);
}
template <class F> PMF_DEVINL float4 vbase(F f, int i0, float) { return make_float4(f(i0), f(i0 + 1), f(i0 + 2), f(i0 + 3)); }
template <class F> PMF_DEVINL double2 vbase(F f, int i0, double) { return make_double2(f(i0), f(i0 + 1)); }
PMF_DEVINL void vzero(float4& v) { v = make_float4(0.f, 0.f, 0.f, 0.f); }
PMF_DEVINL void vzero(double2& v) { v = make_double2(0., 0.); }
PMF_DEVINL void vaddto(float4& a, const float4& b) { a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w; }
PMF_DEVINL void vaddto(double2& a, const double2& b) { a.x += b.x; a.y += b.y; }

PMF_DEVINL void cp_async16(void* smem_dst, const void* gmem_src)
{
    unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem_src) : "memory");
}
PMF_DEVINL void cp_async_wait_all()
{
    asm volatile("cp.async.commit_group;\n cp.async.wait_group 0;\n" ::: "memory");
}

// Everything a team needs to know about the row it is working on.
template <class real> struct RowView {
    const real* tile;  // staged tile in shared memory (row stride kp) or nullptr
    const real* F;     // fixed factor matrix in global memory (row stride ldf, pads are 0)
    const int* ind;    // the row's non-zero indices (global)
    const real* xv;    // the row's non-zero values (shared copy when staged, else global)
    real* pa;          // per-non-zero scratch: <x, F_j> at the current point
    real* pb;          // per-non-zero scratch: coefficients / terms
    real* pc;          // per-non-zero scratch: <x_trial, F_j>
    real* gscr;        // team-size * 16 bytes of reduction scratch (fast gaxpy)
    int n;             // non-zeros in this row
    int k, kp, ldf;    // components; tile stride; global stride (multiple of 16 bytes)
    PMF_DEVINL const real* rowp(int t) const
    {
        return tile ? tile + (size_t)t * kp : F + (size_t)ind[t] * ldf;
    }
};

// Gather the row's tile (and its values) into shared memory.  The indices are first copied
// to shared memory (coalesced; `idx_s` may alias one of the per-non-zero scratch arrays), so
// that the 16-byte cp.async gathers are not chained behind global index loads.
template <class real, class Team>
PMF_DEVINL void stage_tile(const Team& tm, const real* __restrict__ F, const int* __restrict__ ind,
                           const real* __restrict__ xv_g, int n, int ldf, int kp,
                           real* tile, real* xv_s, int* idx_s)
{
    constexpr int V = RealTraits<real>::V;
    const int L = ldf / V;  // 16-byte chunks per factor row
    for (int t = tm.rank(); t < n; t += tm.size()) { idx_s[t] = ind[t]; xv_s[t] = xv_g[t]; }
    tm.sync();
    // thread -> (row t, chunk c), advanced without divisions
    const int sz = tm.size();
    const int dq = sz / L, dr = sz - dq * L;
    int t = tm.rank() / L, c = tm.rank() - t * L;
    while (t < n) {
        cp_async16(tile + (size_t)t * kp + c * V, F + (size_t)idx_s[t] * ldf + c * V);
        t += dq; c += dr;
        if (c >= L) { c -= L; t++; }
    }
    cp_async_wait_all();
    tm.sync();
}

// Fast-mode dot products: lane `rank` handles non-zeros rank, rank+sz, ... NR at a time.
template <int NR, class real>
PMF_DEVINL void dots_fast(const RowView<real>& rv, const real* a, real* out, int rank, int sz)
{
    using VT = typename Vec16<real>::type;
    constexpr int V = RealTraits<real>::V;
    const int n = rv.n, nv = rv.ldf / V;
    const VT* av = reinterpret_cast<const VT*>(a);
    for (int t = rank; t < n; t += NR * sz) {
        const VT* r[NR];
        if (rv.tile) {       // staged tile: shared-memory addressing only (row t at tile + t*kp)
            const VT* tv = reinterpret_cast<const VT*>(rv.tile);
            const int kpv = rv.kp / V;
#pragma unroll
            for (int j = 0; j < NR; j++) r[j] = tv + ((t + j * sz < n) ? (t + j * sz) : t) * kpv;
            real s[NR];
#pragma unroll
            for (int j = 0; j < NR; j++) s[j] = 0;
#pragma unroll 2
            for (int c = 0; c < nv; c++) {
                const VT x = av[c];
#pragma unroll
                for (int j = 0; j < NR; j++) s[j] = vdot4(x, r[j][c], s[j]);
            }
#pragma unroll
            for (int j = 0; j < NR; j++) if (t + j * sz < n) out[t + j * sz] = s[j];
        } else {             // tile in global memory / L2
            const VT* Fv = reinterpret_cast<const VT*>(rv.F);
            const size_t ldv = (size_t)rv.ldf / V;
#pragma unroll
            for (int j = 0; j < NR; j++) r[j] = Fv + (size_t)rv.ind[(t + j * sz < n) ? (t + j * sz) : t] * ldv;
            real s[NR];
#pragma unroll
            for (int j = 0; j < NR; j++) s[j] = 0;
#pragma unroll 2
            for (int c = 0; c < nv; c++) {
                const VT x = av[c];
#pragma unroll
                for (int j = 0; j < NR; j++) s[j] = vdot4(x, __ldg(r[j] + c), s[j]);
            }
#pragma unroll
            for (int j = 0; j < NR; j++) if (t + j * sz < n) out[t + j * sz] = s[j];
        }
    }
}

// Fast-mode dot products for a tile that is NOT staged (rows streamed from global memory / L2):
// a group of G lanes reads one factor row with coalesced 16-byte loads (lane c takes chunks c, c+32, ...),
// keeps its chunks of `a` in registers, and the G partial sums are folded with shuffles.
template <class real, class Team>
PMF_DEVINL void dots_stream(const Team& tm, const RowView<real>& rv, const real* a, real* out)
{
    using VT = typename Vec16<real>::type;
    constexpr int V = RealTraits<real>::V;
    // chunks per lane: enough for ldf = 256 (the largest k a handle takes), i.e. 64 chunks of 16 bytes in
    // float and 128 in double
    constexpr int NCH = (256 / V + 31) / 32;
    const int n = rv.n, L = rv.ldf / V;
    int G = 1;
    while (G < L && G < 32) G <<= 1;
    const int lane = threadIdx.x & 31, c = lane & (G - 1);
    const int gid = tm.rank() / G, ngroups = tm.size() / G;
    const VT* av = reinterpret_cast<const VT*>(a);
    const VT* Fv = reinterpret_cast<const VT*>(rv.F);
    const size_t ldv = (size_t)rv.ldf / V;
    VT zero; vzero(zero);
    bool has[NCH]; VT ac[NCH];                                  // chunk c + 32 j only when L > 32 j (G == 32)
#pragma unroll
    for (int j = 0; j < NCH; j++) { has[j] = c + 32 * j < L; ac[j] = has[j] ? av[c + 32 * j] : zero; }
    // warp-uniform trip count (the shuffles below need every lane of the warp): iterate on the
    // warp's first group and predicate the memory accesses
    const int gpw = 32 / G;                                     // groups per warp
    const int sub = lane / G;
    constexpr int U = 4;                                        // rows in flight per lane group
    for (int base = (tm.rank() >> 5) * gpw; base < n; base += U * ngroups) {
        int tt[U]; bool ok[U]; const VT* r[U]; real sacc[U];
#pragma unroll
        for (int u = 0; u < U; u++) { tt[u] = base + sub + u * ngroups; ok[u] = tt[u] < n; }
        int id[U];
#pragma unroll
        for (int u = 0; u < U; u++) id[u] = rv.ind[ok[u] ? tt[u] : 0];          // all index loads first
#pragma unroll
        for (int u = 0; u < U; u++) r[u] = Fv + (size_t)id[u] * ldv;
        VT b[U][NCH];
#pragma unroll
        for (int u = 0; u < U; u++)                                             // then all row loads
#pragma unroll
            for (int j = 0; j < NCH; j++) b[u][j] = has[j] ? __ldg(r[u] + c + 32 * j) : zero;
#pragma unroll
        for (int u = 0; u < U; u++) {
            sacc[u] = vdot4(ac[0], b[u][0], (real)0);
#pragma unroll
            for (int j = 1; j < NCH; j++) if (has[j]) sacc[u] = vdot4(ac[j], b[u][j], sacc[u]);
        }
        for (int o = G >> 1; o > 0; o >>= 1) {
#pragma unroll
            for (int u = 0; u < U; u++) sacc[u] += __shfl_xor_sync(0xffffffffu, sacc[u], o);
        }
        if (c == 0) {
#pragma unroll
            for (int u = 0; u < U; u++) if (ok[u]) out[tt[u]] = sacc[u];
        }
    }
    (void)gid;
}

// out[t] = <a, F_t>  for every non-zero t of the row.  `a` is a shared-memory
// vector of kp reals whose pads [k, kp) are zero.
template <bool STRICT, class real, class Team>
PMF_DEVINL void dots(const Team& tm, const RowView<real>& rv, const real* a, real* out)
{
    const int n = rv.n;
    if (STRICT) {
        const int k = rv.k;
        for (int t = tm.rank(); t < n; t += tm.size()) {
            const real* r = rv.rowp(t);
            real s = 0;
            for (int i = 0; i < k; i++) s = add_rn(s, mul_rn(a[i], r[i]));
            out[t] = s;
        }
    } else {
        const int sz = tm.size();
        if (!rv.tile && sz >= 32) { dots_stream(tm, rv, a, out); tm.sync(); return; }
        // rows per lane and pass: as many as the row has, up to 4 (they share each load of `a`)
        if (n <= sz) dots_fast<1>(rv, a, out, tm.rank(), sz);
        else if (n <= 2 * sz) dots_fast<2>(rv, a, out, tm.rank(), sz);
        else dots_fast<4>(rv, a, out, tm.rank(), sz);
    }
    tm.sync();
}

// g[i] (+)= sum_t coef[t] * F_t[i].
//   STRICT: g[i] is accumulated in place, t ascending, two roundings per term
//           (exactly the reference's chain of axpy calls on `grad`).
//   fast  : partial sums per thread group, then g[i] = g[i] + total.
// `g` is a shared vector of kp reals.  Ends with a team sync.
struct NoBase {};
template <bool STRICT, class real, class Team, class BaseFn = NoBase>
PMF_DEVINL void gaxpy(const Team& tm, const RowView<real>& rv, const real* coef, real* g, BaseFn basefn = BaseFn())
{
    // basefn(i) (fast mode only) gives the value g[i] starts from; without it g is accumulated onto
    constexpr bool HAS_BASE = !std::is_same<BaseFn, NoBase>::value;
    const int n = rv.n;
    if (STRICT) {
        const int k = rv.k;
        for (int i = tm.rank(); i < k; i += tm.size()) {
            real acc = g[i];
            for (int t = 0; t < n; t++) acc = add_rn(acc, mul_rn(coef[t], rv.rowp(t)[i]));
            g[i] = acc;
        }
        tm.sync();
        return;
    }
    using VT = typename Vec16<real>::type;
    constexpr int V = RealTraits<real>::V;
    const int L = rv.ldf / V;
    const int sz = tm.size(), rk = tm.rank();
    VT* scr = reinterpret_cast<VT*>(rv.gscr);
    VT* gv = reinterpret_cast<VT*>(g);
    // partial sums of this team's (slice of the) non-zeros go to `tot` = scr[0..L)
    if (L <= sz) {
        const int groups = sz / L;
        const int grp = rk / L, c = rk - grp * L;
        VT acc0, acc1;
        vzero(acc0); vzero(acc1);
        if (grp < groups) {
            int t = grp;
            if (rv.tile) {          // resident tile: pointer arithmetic only
                const VT* p = reinterpret_cast<const VT*>(rv.tile) + grp * (rv.kp / V) + c;
                const int stride = groups * (rv.kp / V);
                for (; t + groups < n; t += 2 * groups) {
                    const VT b0 = p[0], b1 = p[stride];
                    vfma(acc0, coef[t], b0);
                    vfma(acc1, coef[t + groups], b1);
                    p += 2 * stride;
                }
                if (t < n) vfma(acc0, coef[t], p[0]);
            } else {                // tile in global memory / L2: four independent loads in flight
                const VT* Fv = reinterpret_cast<const VT*>(rv.F) + c;
                const size_t ldv = (size_t)rv.ldf / V;
                VT acc2, acc3;
                vzero(acc2); vzero(acc3);
                for (; t + 3 * groups < n; t += 4 * groups) {
                    const int i0 = rv.ind[t], i1 = rv.ind[t + groups], i2 = rv.ind[t + 2 * groups], i3 = rv.ind[t + 3 * groups];
                    const VT b0 = __ldg(Fv + (size_t)i0 * ldv), b1 = __ldg(Fv + (size_t)i1 * ldv);
                    const VT b2 = __ldg(Fv + (size_t)i2 * ldv), b3 = __ldg(Fv + (size_t)i3 * ldv);
                    vfma(acc0, coef[t], b0);
                    vfma(acc1, coef[t + groups], b1);
                    vfma(acc2, coef[t + 2 * groups], b2);
                    vfma(acc3, coef[t + 3 * groups], b3);
                }
                for (; t < n; t += groups) vfma(acc0, coef[t], __ldg(Fv + (size_t)rv.ind[t] * ldv));
                vaddto(acc0, acc2); vaddto(acc1, acc3);
            }
            vaddto(acc0, acc1);
        }
        scr[rk] = acc0;
        tm.sync();
        if (rk < L) {  // group 0 folds the other groups in a fixed order
            VT tot = scr[rk];
            for (int gq = 1; gq < groups; gq++) vaddto(tot, scr[gq * L + rk]);
            if (Team::is_gang) {
                scr[rk] = tot;   // groups >= 1 here is read by nobody else: safe to overwrite slot rk
            } else {
                VT base;
                if constexpr (HAS_BASE) base = vbase(basefn, rk * V, real()); else base = gv[rk];
                vaddto(base, tot);
                gv[rk] = base;
            }
        }
    } else {
        // fewer lanes than 16-byte chunks: each lane owns chunks rk, rk+sz, ... and walks all t
        for (int c0 = rk; c0 < L; c0 += 2 * sz) {
            const int c1 = c0 + sz;
            const bool two = c1 < L;
            VT acc0, acc1;
            vzero(acc0); vzero(acc1);
            if (rv.tile) {
                const VT* p = reinterpret_cast<const VT*>(rv.tile) + c0;
                const int kpv = rv.kp / V, off1 = two ? sz : 0;
                for (int t = 0; t < n; t++, p += kpv) {
                    const real ct = coef[t];
                    vfma(acc0, ct, p[0]);
                    vfma(acc1, ct, p[off1]);
                }
            } else {
                const VT* Fv = reinterpret_cast<const VT*>(rv.F);
                const size_t ldv = (size_t)rv.ldf / V;
                for (int t = 0; t < n; t++) {
                    const VT* p = Fv + (size_t)rv.ind[t] * ldv;
                    const real ct = coef[t];
                    vfma(acc0, ct, __ldg(p + c0));
                    if (two) vfma(acc1, ct, __ldg(p + c1));
                }
            }
            if (Team::is_gang) {
                scr[c0] = acc0;
                if (two) scr[c1] = acc1;
            } else {
                VT base;
                if constexpr (HAS_BASE) base = vbase(basefn, c0 * V, real()); else base = gv[c0];
                vaddto(base, acc0);
                gv[c0] = base;
                if (two) {
                    VT b1;
                    if constexpr (HAS_BASE) b1 = vbase(basefn, c1 * V, real()); else b1 = gv[c1];
                    vaddto(b1, acc1); gv[c1] = b1;
                }
            }
        }
    }
    if (Team::is_gang) {
        // fold the per-CTA partial vectors of the cluster, then add onto g
        tm.sync();
        tm.nnz_vec_sum(rv.gscr, rv.ldf);
        for (int c = rk; c < L; c += sz) {
            VT base;
            if constexpr (HAS_BASE) base = vbase(basefn, c * V, real()); else base = gv[c];
            vaddto(base, scr[c]);
            gv[c] = base;
        }
    }
    tm.sync();
    // keep pads at zero (F pads are zero, so this is already the case; be explicit)
}

// Sequential sum over the non-zeros of  x_t * log(p_t)  (the `lsum` of
// src/poismf.c:200-206,255-263).  Every member gets the same value.
template <bool STRICT, class real, class Team>
PMF_DEVINL real sum_xlogp(const Team& tm, const RowView<real>& rv, const real* p)
{
    const int n = rv.n;
    if (STRICT) {
        real s = 0;
        if (tm.rank() == 0)
            for (int t = 0; t < n; t++) s = xlogp_acc<true>(s, rv.xv[t], p[t]);
        return tm.bcast0(s);
    }
    real s = 0;
    for (int t = tm.rank(); t < n; t += tm.size()) s += xlogp(rv.xv[t], p[t]);
    return tm.nnz_sum(s);
}

// Constants of one half-sweep's row sub-problems.
template <class real> struct HalfSweepConsts {
    real l2;        // l2_reg
    real two_l2;    // (real)(2. * l2_reg): the axpy alpha of src/poismf.c:215,239,269
    real w;         // w_mult
    real wm1;       // (real)(w_mult - 1.)  src/poismf.c:113
    real step_w;    // pg: step_size * w_mult      (:151)
    real neg_step;  // pg: -step_size              (:460,:533)
    real pre_scale; // pg, w != 1: extra factor on the weighted sums (1 in run_poismf; -step0 in
                    // factors_multiple, which scales them twice: src/pred.c:126 and :160)
    real cdiv;      // pg: 1/(1+2*l2*step)         (:511)
    real clip_thr;  // smallest `real` v with (double)v >= 1e-15: the cg clip of nonnegcg.c:303 in `real` arithmetic
    int maxupd;
    int limit_step, reuse_prev, early_stop;
    int method;
};

// csum_row = (w-1) * sum_t F_t + csum  [* neg_step for pg]   (adjustment_Bsum, :85-123;
// pg scaling :526,:576).  Only when w != 1.
template <bool STRICT, class real, class Team>
PMF_DEVINL void weighted_colsum(const Team& tm, const RowView<real>& rv, const real* csum,
                                const HalfSweepConsts<real>& hc, real* ones, real* out)
{
    const int k = rv.k;
    for (int t = tm.rank(); t < rv.n; t += tm.size()) ones[t] = (real)1;
    vfill(tm, out, (real)0, rv.kp);
    tm.sync();
    gaxpy<STRICT>(tm, rv, ones, out);
    for (int i = tm.rank(); i < k; i += tm.size()) {
        real v = mul<STRICT>(out[i], hc.wm1);
        v = add<STRICT>(v, csum[i]);
        if (hc.method == M_PG) { v = mul<STRICT>(v, hc.pre_scale); v = mul<STRICT>(v, hc.neg_step); }
        out[i] = v;
    }
    tm.sync();
}

// f = <csum,x> + l2<x,x> - w * sum x_t log<x,F_t>      (calc_fun_single, :194-208)
// Leaves <x,F_t> in `pout`.
template <bool STRICT, class real, class Team>
PMF_DEVINL real eval_f_cg(const Team& tm, const RowView<real>& rv, const real* csum,
                          const HalfSweepConsts<real>& hc, const real* x, real* pout)
{
    dots<STRICT>(tm, rv, x, pout);
    real reg = vdot<STRICT>(tm, csum, x, rv.k);
    reg = mad<STRICT>(hc.l2, vdot<STRICT>(tm, x, x, rv.k), reg);
    const real ls = sum_xlogp<STRICT>(tm, rv, pout);
    return sub<STRICT>(reg, mul<STRICT>(ls, hc.w));
}

// grad = csum + 2 l2 x - w * sum (x_t/<x,F_t>) F_t     (calc_grad_single[_w], :210-240)
// `p` must hold <x,F_t>.  Uses rv.pb for the coefficients.
template <bool STRICT, class real, class Team>
PMF_DEVINL void eval_g_cg(const Team& tm, const RowView<real>& rv, const real* csum,
                          const HalfSweepConsts<real>& hc, const real* x, const real* p, real* g)
{
    const int k = rv.k;
    for (int t = tm.rank(); t < rv.n; t += tm.size()) rv.pb[t] = -rv.xv[t] / p[t];
    if (hc.w == (real)1) {
        for (int i = tm.rank(); i < k; i += tm.size()) g[i] = mad<STRICT>(hc.two_l2, x[i], csum[i]);
        tm.sync();
        gaxpy<STRICT>(tm, rv, rv.pb, g);
    } else {
        vfill(tm, g, (real)0, k);
        tm.sync();
        gaxpy<STRICT>(tm, rv, rv.pb, g);
        for (int i = tm.rank(); i < k; i += tm.size()) {
            real v = mul<STRICT>(g[i], hc.w);
            v = add<STRICT>(v, csum[i]);
            g[i] = mad<STRICT>(hc.two_l2, x[i], v);
        }
        tm.sync();
    }
}

// f (WITHOUT the l2 term, Q3) and grad in one go      (calc_fun_and_grad, :242-273)
template <bool STRICT, class real, class Team>
PMF_DEVINL real eval_fg_tn(const Team& tm, const RowView<real>& rv, const real* csum,
                           const HalfSweepConsts<real>& hc, const real* x, real* g)
{
    const int k = rv.k;
    dots<STRICT>(tm, rv, x, rv.pa);
    for (int t = tm.rank(); t < rv.n; t += tm.size()) rv.pb[t] = -rv.xv[t] / rv.pa[t];
    vfill(tm, g, (real)0, k);
    tm.sync();
    gaxpy<STRICT>(tm, rv, rv.pb, g);
    const real ls = sum_xlogp<STRICT>(tm, rv, rv.pa);
    const real reg = vdot<STRICT>(tm, csum, x, k);
    for (int i = tm.rank(); i < k; i += tm.size()) {
        real v = g[i];
        if (hc.w != (real)1) v = mul<STRICT>(v, hc.w);
        v = add<STRICT>(v, csum[i]);
        g[i] = mad<STRICT>(hc.two_l2, x[i], v);
    }
    tm.sync();
    return sub<STRICT>(reg, mul<STRICT>(ls, hc.w));
}

}  // namespace pmf
