// poismf_b200 — truncated-Newton CG row solver with bounds (device).
//
// Follows /root/reference/src/tnc.c (TNC 1.3 trimmed to "lower bound 0, no upper
// bound") as it is driven by src/poismf.c:324-404:
//   tnc            :251-463     tnc_minimize      :554-993
//   tnc_direction  :1162-1341   hessianTimesVector:1388-1435 (finite difference)
//   msolve/ssbfgs  :1444-1575   initPreconditioner:1580-1658
//   linearSearch   :1664-1813   getptcInit/Iter   :1822-2154 (Gill-Murray)
// with the fixed arguments of the call site (eta .25, stepmx 10, accuracy 0,
// fmin 0, ftol 1e-4, xtol -1, pgtol -1, rescale 1.3, maxCGit = clamp(k/2,1,50)).
//
// The reference is C without tgmath: in the float build many sub-expressions are
// evaluated in double (literals like 1.0, fabs(), sqrt()).  Those promotions are
// written out explicitly below (D(...)) because they change float rounding; for
// real == double they are no-ops.  The strict translation unit is compiled with
// --fmad=false so that none of the scalar expressions is contracted.
//
// Layout: every k-vector lives in the team's shared memory (kp reals, pads zero);
// scalar state is replicated in the registers of every team member and all
// members take every branch together.
#pragma once
#include "rowops.cuh"
#include "sweep_consts.h"

namespace pmf {

enum { TV_X = 0, TV_CSUM, TV_XSCALE, TV_XOFFSET, TV_OLDG, TV_G, TV_TMP, TV_DIAGB, TV_PK, TV_SK,
       TV_YK, TV_SR, TV_YR, TV_R, TV_V, TV_ZK, TV_EMAT, TV_GV, TV_W0, TV_W1, TV_W2, TV_GFULL,
       TV_PREV, TV_PIVOT };

#define PMF_EW(i) for (int i = tm.rank(); i < n; i += tm.size())
typedef double D;

template <class real> struct GmState {   // getptc's 24 scalars (tnc.c:1822-1830)
    real reltol, abstol, tnytol, xbnd, u, fu, gu, xmin, fmin, gmin, xw, fw, gw, a, b, oldf, b1,
        scxbnd, e, step, factor, gtest1, gtest2, tol;
    bool braktd;
};
enum { GM_OK = 0, GM_EVAL = 1, GM_EINVAL = 2, GM_FAIL = 3 };

template <class real> PMF_DEVINL void gm_clip_step(GmState<real>& q)   // tnc.c:1875-1886 == :2141-2152
{
    if (q.step >= q.scxbnd) {
        q.step = q.scxbnd;
        q.scxbnd = (real)(D(q.scxbnd) - (D(q.reltol) * fabs(D(q.xbnd)) + D(q.abstol)) / (1.0 + D(q.reltol)));
    }
    q.u = q.step;
    if (fabs(D(q.step)) < D(q.tol) && q.step < (real)0) q.u = -q.tol;
    if (fabs(D(q.step)) < D(q.tol) && q.step >= (real)0) q.u = q.tol;
}

template <class real> PMF_DEVINL int gm_init(GmState<real>& q, real eta, real rmu)   // :1822-1888
{
    if (q.u <= (real)0 || q.xbnd <= q.tnytol || q.gu > (real)0) return GM_EINVAL;
    if (q.xbnd < q.abstol) q.abstol = q.xbnd;
    q.tol = q.abstol;
    q.a = 0; q.xw = 0; q.xmin = 0;
    q.oldf = q.fu; q.fmin = q.fu; q.fw = q.fu;
    q.gw = q.gu; q.gmin = q.gu;
    q.step = q.u; q.factor = (real)5.0; q.braktd = false;
    q.scxbnd = q.xbnd;
    q.b = (real)(D(q.scxbnd) + D(q.reltol) * fabs(D(q.scxbnd)) + D(q.abstol));
    q.e = q.b + q.b;
    q.b1 = q.b;
    q.gtest1 = -rmu * q.gu;
    q.gtest2 = -eta * q.gu;
    gm_clip_step(q);
    return GM_EVAL;
}

template <class real> PMF_DEVINL int gm_iter(GmState<real>& q, real big, real rtsmll, real fpresn)   // :1890-2154
{
    real abgw, absr, p, qq, r, s, scale, denom, a1, d1, d2, sumsq, abgmin, chordm, chordu, xmidpt, twotol;
    bool to_check = false;

    if (q.fu <= q.fmin) {
        chordu = q.oldf - (q.xmin + q.u) * q.gtest1;
        if (q.fu > chordu) {
            chordm = q.oldf - q.xmin * q.gtest1;
            q.gu = -q.gmin;
            denom = chordm - q.fmin;
            if (fabs(D(denom)) < 1e-15) {
                denom = (real)1e-15;
                if (chordm - q.fmin < (real)0) denom = -denom;
            }
            if (q.xmin != (real)0) q.gu = q.gmin * (chordu - q.fu) / denom;
            q.fu = (real)(0.5 * D(q.u) * D(q.gmin + q.gu) + D(q.fmin));
            if (q.fu < q.fmin) q.fu = q.fmin;
        } else {
            q.fw = q.fmin; q.fmin = q.fu;
            q.gw = q.gmin; q.gmin = q.gu;
            q.xmin += q.u; q.a -= q.u; q.b -= q.u;
            q.xw = -q.u; q.scxbnd -= q.u;
            if (q.gu <= (real)0) q.a = 0;
            else { q.b = 0; q.braktd = true; }
            q.tol = (real)(fabs(D(q.xmin)) * D(q.reltol) + D(q.abstol));
            to_check = true;
        }
    }
    if (!to_check) {
        if (q.u < (real)0) q.a = q.u;
        else { q.b = q.u; q.braktd = true; }
        q.xw = q.u; q.fw = q.fu; q.gw = q.gu;
    }

    twotol = q.tol + q.tol;
    xmidpt = (real)(0.5 * D(q.a + q.b));
    const bool convrg = (fabs(D(xmidpt)) <= D(twotol) - 0.5 * D(q.b - q.a)) ||
                        (fabs(D(q.gmin)) <= D(q.gtest2) && q.fmin < q.oldf &&
                         ((fabs(D(q.xmin - q.xbnd)) > D(q.tol)) || (!q.braktd)));
    if (convrg) {
        if (q.xmin != (real)0) return GM_OK;
        if (fabs(D(q.oldf - q.fw)) <= D(fpresn)) return GM_FAIL;
        q.tol = (real)(0.1 * D(q.tol));
        if (q.tol < q.tnytol) return GM_FAIL;
        q.reltol = (real)(0.1 * D(q.reltol));
        q.abstol = (real)(0.1 * D(q.abstol));
        twotol = (real)(0.1 * D(twotol));
    }

    r = 0; qq = 0; s = 0;
    if (fabs(D(q.e)) > D(q.tol)) {
        bool minimum_found = false;
        r = (real)(3.0 * D(q.fmin - q.fw) / D(q.xw) + D(q.gmin) + D(q.gw));
        absr = (real)fabs(D(r));
        qq = absr;
        if (q.gw != (real)0 && q.gmin != (real)0) {
            abgw = (real)fabs(D(q.gw));
            abgmin = (real)fabs(D(q.gmin));
            s = (real)(sqrt(D(abgmin)) * sqrt(D(abgw)));
            if (q.gw / abgw * q.gmin > (real)0) {
                if (r >= s || r <= -s) {
                    qq = (real)(sqrt(fabs(D(r + s))) * sqrt(fabs(D(r - s))));
                } else {
                    r = 0; qq = 0;
                    minimum_found = true;
                }
            } else {
                sumsq = 1; p = 0;
                if (absr >= s) {
                    if (absr > rtsmll) p = absr * rtsmll;
                    if (s >= p) { const real value = s / absr; sumsq = (real)(1.0 + D(value * value)); }
                    scale = absr;
                } else {
                    if (s > rtsmll) p = s * rtsmll;
                    if (absr >= p) { const real value = absr / s; sumsq = (real)(1.0 + D(value * value)); }
                    scale = s;
                }
                sumsq = (real)sqrt(D(sumsq));
                qq = big;
                if (scale < big / sumsq) qq = scale * sumsq;
            }
        }
        if (!minimum_found) {
            if (q.xw < (real)0) qq = -qq;
            s = q.xw * (q.gmin - r - qq);
            qq = q.gw - q.gmin + qq + qq;
            if (qq > (real)0) s = -s;
            if (qq <= (real)0) qq = -qq;
            r = q.e;
            if (q.b1 != q.step || q.braktd) q.e = q.step;
        }
    }

    a1 = q.a;
    q.b1 = q.b;
    q.step = xmidpt;
    if ((!q.braktd) || ((q.a == (real)0 && q.xw < (real)0) || (q.b == (real)0 && q.xw > (real)0))) {
        if (q.braktd) {
            d1 = q.xw;
            d2 = q.a;
            if (q.a == (real)0) d2 = q.b;
            q.u = -d1 / d2;
            q.step = (real)(5.0 * D(d2) * (0.1 + 1.0 / D(q.u)) / 11.0);
            if (q.u < (real)1) q.step = (real)(0.5 * D(d2) * sqrt(D(q.u)));
        } else {
            q.step = -q.factor * q.xw;
            if (q.step > q.scxbnd) q.step = q.scxbnd;
            if (q.step != q.scxbnd) q.factor = (real)(5.0 * D(q.factor));
        }
        if (q.step <= (real)0) a1 = q.step;
        if (q.step > (real)0) q.b1 = q.step;
    }

    if (fabs(D(s)) <= fabs(0.5 * D(qq) * D(r)) || s <= qq * a1 || s >= qq * q.b1) {
        q.e = q.b - q.a;
    } else {
        q.step = s / qq;
        if (q.step - q.a < twotol || q.b - q.step < twotol) {
            if (xmidpt <= (real)0) q.step = -q.tol;
            else q.step = q.tol;
        }
    }
    gm_clip_step(q);
    return GM_EVAL;
}

// Solver context: vectors + the row's evaluation closure.
template <bool STRICT, class real, class Team> struct TnCtx {
    const Team& tm;
    const RowView<real>& rv;
    const HalfSweepConsts<real>& hc;
    real* V;
    int n, kp;
    int nfeval, maxnfeval;
    PMF_DEVINL real* vec(int id) const { return V + (size_t)id * kp; }
    PMF_DEVINL int* pivot() const { return reinterpret_cast<int*>(V + (size_t)TV_PIVOT * kp); }
    PMF_DEVINL real fg(const real* x, real* g) const
    {
        return eval_fg_tn<STRICT>(tm, rv, vec(TV_CSUM), hc, x, g);
    }
    PMF_DEVINL real dot(const real* a, const real* b) const { return vdot<STRICT>(tm, a, b, n); }
    PMF_DEVINL real nrm2(const real* a) const { return vnrm2<STRICT>(tm, a, n); }
    PMF_DEVINL void project(real* x) const
    {
        const int* pv = pivot();
        PMF_EW(i) if (pv[i] != 0) x[i] = 0;
        tm.sync();
    }
};

// ssbfgs / ssbfgs2 (tnc.c:1533-1575); out may alias hjv
template <bool STRICT, class real, class Team>
PMF_DEVINL void tn_ssbfgs(const TnCtx<STRICT, real, Team>& c, real gamma, const real* sj, const real* hjv,
                          const real* hjyj, real yjsj, real yjhyj, real vsj, real vhyj, real* out)
{
    const Team& tm = c.tm; const int n = c.n;
    real beta, delta;
    if (yjsj == (real)0) { delta = 0; beta = 0; }
    else {
        delta = (real)((D(gamma * yjhyj / yjsj) + 1.0) * D(vsj) / D(yjsj) - D(gamma * vhyj / yjsj));
        beta = -gamma * vsj / yjsj;
    }
    PMF_EW(i) out[i] = gamma * hjv[i] + delta * sj[i] + beta * hjyj[i];
    tm.sync();
}

// msolve (tnc.c:1444-1528)
template <bool STRICT, class real, class Team>
PMF_DEVINL void tn_msolve(const TnCtx<STRICT, real, Team>& c, const real* g, real* y, bool upd1,
                          real yksk, real yrsr, bool lreset)
{
    const Team& tm = c.tm; const int n = c.n;
    const real* diagb = c.vec(TV_DIAGB);
    const real *sk = c.vec(TV_SK), *yk = c.vec(TV_YK), *sr = c.vec(TV_SR), *yr = c.vec(TV_YR);
    if (upd1) {
        PMF_EW(i) y[i] = g[i] / diagb[i];
        tm.sync();
        return;
    }
    const real gsk = c.dot(g, sk);
    real *hg = c.vec(TV_W0), *hyr = c.vec(TV_W1), *hyk = c.vec(TV_W2);
    if (lreset) {
        PMF_EW(i) {
            const real rd = (real)(1.0 / D(diagb[i]));
            hg[i] = g[i] * rd; hyk[i] = yk[i] * rd;
        }
        tm.sync();
        const real ykhyk = c.dot(yk, hyk);
        const real ghyk = c.dot(g, hyk);
        tn_ssbfgs(c, (real)1, sk, hg, hyk, yksk, ykhyk, gsk, ghyk, y);
    } else {
        PMF_EW(i) {
            const real rd = (real)(1.0 / D(diagb[i]));
            hg[i] = g[i] * rd; hyk[i] = yk[i] * rd; hyr[i] = yr[i] * rd;
        }
        tm.sync();
        const real gsr = c.dot(g, sr);
        const real ghyr = c.dot(g, hyr);
        const real yrhyr = c.dot(yr, hyr);
        tn_ssbfgs(c, (real)1, sr, hg, hyr, yrsr, yrhyr, gsr, ghyr, hg);
        const real yksr = c.dot(yk, sr);
        const real ykhyr = c.dot(yk, hyr);
        tn_ssbfgs(c, (real)1, sr, hyk, hyr, yrsr, yrhyr, yksr, ykhyr, hyk);
        const real ykhyk = c.dot(hyk, yk);
        const real ghyk = c.dot(hyk, g);
        tn_ssbfgs(c, (real)1, sk, hg, hyk, yksk, ykhyk, gsk, ghyk, y);
    }
}

// initPreconditioner (tnc.c:1580-1658)
template <bool STRICT, class real, class Team>
PMF_DEVINL void tn_init_precond(const TnCtx<STRICT, real, Team>& c, bool lreset, real yksk, real yrsr, bool upd1)
{
    const Team& tm = c.tm; const int n = c.n;
    real *diagb = c.vec(TV_DIAGB), *emat = c.vec(TV_EMAT), *bsk = c.vec(TV_W0);
    const real *sk = c.vec(TV_SK), *yk = c.vec(TV_YK), *sr = c.vec(TV_SR), *yr = c.vec(TV_YR);
    if (upd1) {
        PMF_EW(i) emat[i] = diagb[i];
        tm.sync();
        return;
    }
    if (lreset) {
        PMF_EW(i) bsk[i] = diagb[i] * sk[i];
        tm.sync();
        real sds = c.dot(sk, bsk);
        if (yksk == (real)0) yksk = 1;
        if (sds == (real)0) sds = 1;
        PMF_EW(i) {
            const real td = diagb[i];
            emat[i] = td - td * td * sk[i] * sk[i] / sds + yk[i] * yk[i] / yksk;
        }
        tm.sync();
    } else {
        PMF_EW(i) bsk[i] = diagb[i] * sr[i];
        tm.sync();
        real sds = c.dot(sr, bsk);
        const real srds = c.dot(sk, bsk);
        const real yrsk = c.dot(yr, sk);
        if (yrsr == (real)0) yrsr = 1;
        if (sds == (real)0) sds = 1;
        PMF_EW(i) {
            const real td = diagb[i];
            bsk[i] = td * sk[i] - bsk[i] * srds / sds + yr[i] * yrsk / yrsr;
            emat[i] = td - td * td * sr[i] * sr[i] / sds + yr[i] * yr[i] / yrsr;
        }
        tm.sync();
        sds = c.dot(sk, bsk);
        if (yksk == (real)0) yksk = 1;
        if (sds == (real)0) sds = 1;
        PMF_EW(i) emat[i] -= bsk[i] * bsk[i] / sds + yk[i] * yk[i] / yksk;
        tm.sync();
    }
}

// hessianTimesVector by finite differences (tnc.c:1388-1435): gv <- (grad(x+delta v) - g)/delta
template <bool STRICT, class real, class Team>
PMF_DEVINL void tn_hvp(TnCtx<STRICT, real, Team>& c, const real* x, real fscale, real accuracy, real xnorm)
{
    const Team& tm = c.tm; const int n = c.n;
    real *xv = c.vec(TV_W0), *gv = c.vec(TV_GV);
    const real *v = c.vec(TV_V), *g = c.vec(TV_G), *xs = c.vec(TV_XSCALE), *xo = c.vec(TV_XOFFSET);
    const real delta = (real)(D(accuracy) * (D(xnorm) + 1.0));
    PMF_EW(i) {
        real t = x[i] + delta * v[i];
        t = add_rn(mul_rn(t, xs[i]), xo[i]);   // unscalex :482 (never contracted, see solve_tn)
        xv[i] = (t < (real)0) ? (real)0 : t;   // coercex  :466
    }
    tm.sync();
    (void)c.fg(xv, gv);
    const real dinv = (real)(1.0 / D(delta));
    PMF_EW(i) {
        real t = gv[i] * (xs[i] * fscale);     // scaleg :504
        t = (t - g[i]) * dinv;
        gv[i] = (xs[i] == (real)0) ? (real)0 : t;   // projectConstants :1028
    }
    tm.sync();
}

// tnc_direction (tnc.c:1162-1341)
template <bool STRICT, class real, class Team>
PMF_DEVINL void tn_direction(TnCtx<STRICT, real, Team>& c, real* zsol, const real* x, int maxCGit, bool upd1,
                             real yksk, real yrsr, bool lreset, real fscale, real accuracy, real gnorm,
                             real xnorm)
{
    const Team& tm = c.tm; const int n = c.n;
    real *g = c.vec(TV_G), *r = c.vec(TV_R), *v = c.vec(TV_V), *zk = c.vec(TV_ZK), *gv = c.vec(TV_GV),
         *emat = c.vec(TV_EMAT), *diagb = c.vec(TV_DIAGB);
    real alpha, beta, qold, qnew, rhsnrm, tol, vgv, rz, rzold, qtest, pr, gtp;

    if (maxCGit == 0) {
        PMF_EW(i) zsol[i] = -g[i];
        tm.sync();
        c.project(zsol);
        return;
    }
    rhsnrm = gnorm; tol = (real)1e-12; qold = 0; rzold = 0;
    tn_init_precond(c, lreset, yksk, yrsr, upd1);
    PMF_EW(i) { r[i] = -g[i]; v[i] = 0; zsol[i] = 0; }
    tm.sync();

    for (int k = 0; k < maxCGit; k++) {
        c.project(r);
        tn_msolve(c, r, zk, upd1, yksk, yrsr, lreset);
        c.project(zk);
        rz = c.dot(r, zk);
        if ((rz / rhsnrm < tol) || (c.nfeval >= (c.maxnfeval - 1))) {
            if (k == 0) {
                PMF_EW(i) zsol[i] = -g[i];
                tm.sync();
                c.project(zsol);
            }
            break;
        }
        beta = (k == 0) ? (real)0 : rz / rzold;
        PMF_EW(i) v[i] = zk[i] + beta * v[i];
        tm.sync();
        c.project(v);
        tn_hvp(c, x, fscale, accuracy, xnorm);
        ++c.nfeval;
        c.project(gv);
        vgv = c.dot(v, gv);
        if (vgv / rhsnrm < tol) {
            if (k == 0) {
                tn_msolve(c, g, zsol, upd1, yksk, yrsr, lreset);
                PMF_EW(i) zsol[i] = -zsol[i];
                tm.sync();
                c.project(zsol);
            }
            break;
        }
        {   // diagonalScaling (tnc.c:1347-1362)
            const real vr = (real)(1.0 / D(c.dot(v, r)));
            const real vgv2 = (real)(1.0 / D(c.dot(v, gv)));
            PMF_EW(i) {
                real e = emat[i] + (-r[i] * r[i] * vr + gv[i] * gv[i] * vgv2);
                emat[i] = (D(e) <= 1e-6) ? (real)1 : e;
            }
            tm.sync();
        }
        alpha = rz / vgv;
        PMF_EW(i) { zsol[i] = zsol[i] + alpha * v[i]; r[i] = r[i] + (-alpha) * gv[i]; }
        tm.sync();
        gtp = c.dot(zsol, g);
        pr = c.dot(r, zsol);
        qnew = (real)(D(gtp + pr) * 0.5);
        qtest = (real)(D(k + 1) * (1.0 - D(qold / qnew)));
        if (D(qtest) <= 0.5) break;
        if (gtp > (real)0) {
            PMF_EW(i) zsol[i] = zsol[i] + (-alpha) * v[i];
            tm.sync();
            break;
        }
        qold = qnew;
        rzold = rz;
    }
    PMF_EW(i) diagb[i] = emat[i];              // :1329
    tm.sync();
}

enum { LSR_OK = 0, LSR_MAXFUN = 1, LSR_FAIL = 2 };

// linearSearch (tnc.c:1664-1813)
template <bool STRICT, class real, class Team>
PMF_DEVINL int tn_linesearch(TnCtx<STRICT, real, Team>& c, real fscale, real eta, real ftol, real xbnd,
                             const real* p, real* x, real& f, real& alpha, real* gfull)
{
    const Team& tm = c.tm; const int n = c.n;
    const real EPS = RealTraits<real>::eps();
    real *temp = c.vec(TV_W0), *tempg = c.vec(TV_W1), *newg = c.vec(TV_W2);
    const real *xs = c.vec(TV_XSCALE), *xo = c.vec(TV_XOFFSET);
    const int* pv = c.pivot();
    const int maxlsit = 64;
    int itcnt = 0, itest;
    GmState<real> q;

    PMF_EW(i) temp[i] = gfull[i] * (xs[i] * fscale);
    tm.sync();
    q.gu = c.dot(temp, p);
    PMF_EW(i) temp[i] = (pv[i] != 0) ? (real)0 : x[i];
    tm.sync();
    const real xnorm = c.nrm2(temp);

    const real rteps = (real)sqrt(D(EPS));
    const real pe = c.nrm2(p) + EPS;
    q.reltol = (real)(D(rteps) * (D(xnorm) + 1.0) / D(pe));
    q.abstol = (real)(D(-EPS) * (1.0 + fabs(D(f))) / D(q.gu - EPS));
    q.tnytol = (real)(D(EPS) * (D(xnorm) + 1.0) / D(pe));
    const real rtsmll = EPS;
    const real big = (real)(1.0 / D(EPS * EPS));
    const real fpresn = ftol;
    q.u = alpha; q.fu = f; q.fmin = f; q.xbnd = xbnd;
    q.xmin = alpha;   // the reference aliases *alpha with getptc's xmin
    q.gmin = 0; q.xw = 0; q.fw = 0; q.gw = 0; q.a = 0; q.b = 0; q.oldf = 0; q.b1 = 0; q.scxbnd = 0;
    q.e = 0; q.step = 0; q.factor = 0; q.gtest1 = 0; q.gtest2 = 0; q.tol = 0; q.braktd = false;

    itest = gm_init(q, eta, (real)1e-4);
    if (itest == GM_EVAL) alpha = q.xmin;

    while (itest == GM_EVAL) {
        if ((++itcnt > maxlsit) || (c.nfeval >= c.maxnfeval)) break;
        const real ualpha = alpha + q.u;
        PMF_EW(i) {
            real t = x[i] + ualpha * p[i];
            t = add_rn(mul_rn(t, xs[i]), xo[i]);
            temp[i] = (t < (real)0) ? (real)0 : t;
        }
        tm.sync();
        q.fu = c.fg(temp, tempg);
        ++c.nfeval;
        q.fu *= fscale;
        PMF_EW(i) temp[i] = tempg[i] * (xs[i] * fscale);
        tm.sync();
        q.gu = c.dot(temp, p);
        itest = gm_iter(q, big, rtsmll, fpresn);
        alpha = q.xmin;
        if (alpha == ualpha) {
            PMF_EW(i) newg[i] = tempg[i];
            tm.sync();
        }
    }
    if (itest == GM_OK) {
        f = q.fmin;
        PMF_EW(i) { x[i] = x[i] + alpha * p[i]; gfull[i] = newg[i]; }
        tm.sync();
        return LSR_OK;
    } else if (itcnt > maxlsit) return LSR_FAIL;
    else if (itest != GM_EVAL) return LSR_FAIL;
    return LSR_MAXFUN;
}

// tncg_iteration's per-row body (src/poismf.c:363-396) + tnc (:251-463) + tnc_minimize (:554-993).
// V: the team's vectors; V[TV_X] holds the row's current values on entry and the
// solution on exit.
template <bool STRICT, class real, class Team>
PMF_DEVINL void solve_tn(const Team& tm, const RowView<real>& rv, const HalfSweepConsts<real>& hc,
                         real* V, const real* /*Mrow*/, unsigned long long* n_unchanged)
{
    const int n = rv.k;
    const real EPS = RealTraits<real>::eps();
    TnCtx<STRICT, real, Team> c{tm, rv, hc, V, n, rv.kp, 0, hc.maxupd};
    real *x = c.vec(TV_X), *g = c.vec(TV_G), *temp = c.vec(TV_TMP), *pk = c.vec(TV_PK),
         *gfull = c.vec(TV_GFULL), *xs = c.vec(TV_XSCALE), *xo = c.vec(TV_XOFFSET),
         *diagb = c.vec(TV_DIAGB), *oldg = c.vec(TV_OLDG), *sk = c.vec(TV_SK), *yk = c.vec(TV_YK),
         *sr = c.vec(TV_SR), *yr = c.vec(TV_YR), *prev = c.vec(TV_PREV);
    int* pivot = c.pivot();

    int maxCGit = (int)fmax(1., fmin(50., D((real)n) / 2.));            // poismf.c:342
    if (hc.early_stop) { PMF_EW(i) prev[i] = x[i]; }                     // :374-377
    if (!hc.reuse_prev) { PMF_EW(i) x[i] = (real)1e-3; }                 // :379-381
    tm.sync();

    // ---- tnc() prologue (:323-436)
    PMF_EW(i) x[i] = (x[i] < (real)0) ? (real)0 : x[i];
    tm.sync();
    bool solved = false;
    real f = 0, fscale = 1;
    if (c.maxnfeval >= 1) {
        solved = true;
        f = c.fg(x, gfull);
        c.nfeval++;
        PMF_EW(i) { xs[i] = (real)(1.0 + fabs(D(x[i]))); xo[i] = x[i]; }
        tm.sync();
        const real rteps = (real)sqrt(D(EPS));
        real stepmx = (real)10.;
        const real eta = (real)0.25, rescale = (real)1.3, fmin_ = 0, ftol = (real)1e-4;
        if (maxCGit > n) maxCGit = n;
        const real accuracy = rteps;
        const real pgtol = (real)(1e-2 * sqrt(D(accuracy)));
        const real xtol = rteps;

        // ---- tnc_minimize (:647-963)
        real fLastReset, difnew = 0, epsred = (real)0.05, oldgtp, difold, oldf, xnorm, newscale, gnorm,
             ustpmax, fLastConstraint, spe, yrsr = 0, yksk = 0, alpha = 0;
        int icycle = n - 1, oldnfeval;
        bool lreset = false, newcon = true, upd1 = true, remcon;

        PMF_EW(i) { if (xs[i] > (real)0) x[i] = (x[i] - xo[i]) / xs[i]; }           // scalex :492
        tm.sync();
        f *= fscale;
        PMF_EW(i) {                                                                 // setConstraints :513
            int pvt;
            if (xs[i] == (real)0) pvt = 2;
            else if (D(x[i] * xs[i] + xo[i] - (real)0) <= D(EPS) * 10.0 * (fabs(0.0) + 1.0)) pvt = -1;
            else pvt = 0;
            real gi = gfull[i] * (xs[i] * fscale);                                   // :666-667
            if ((real)(-pvt) * gi < (real)0) pvt = 0;                                // :670-674
            pivot[i] = pvt;
            g[i] = (pvt != 0) ? (real)0 : gi;                                        // project :676
            diagb[i] = 1;                                                            // :693-695
        }
        tm.sync();
        gnorm = c.nrm2(g);
        fLastConstraint = f; fLastReset = f;

        for (;;) {
            if (c.nrm2(g) <= pgtol * fscale) {                                       // :700-712
                break;
            }
            if (c.nfeval >= c.maxnfeval) break;                                      // :715
            newscale = c.nrm2(g);                                                    // :721-746
            if ((newscale > EPS) && (fabs(log10(D(newscale))) > D(rescale))) {
                newscale = (real)(1.0 / D(newscale));
                f *= newscale; fscale *= newscale; gnorm *= newscale;
                fLastConstraint *= newscale; fLastReset *= newscale; difnew *= newscale;
                PMF_EW(i) { g[i] *= newscale; diagb[i] = 1; }
                tm.sync();
                upd1 = true; icycle = n - 1; newcon = true;
            }
            PMF_EW(i) temp[i] = (pivot[i] != 0) ? (real)0 : x[i];                    // :748-751
            tm.sync();
            xnorm = c.nrm2(temp);
            oldnfeval = c.nfeval;

            tn_direction(c, pk, x, maxCGit, upd1, yksk, yrsr, lreset, fscale, accuracy, gnorm, xnorm);

            if (!newcon) {                                                           // :770-785
                if (!lreset) {
                    PMF_EW(i) { sr[i] = sr[i] + sk[i]; yr[i] = yr[i] + yk[i]; }
                    icycle++;
                } else {
                    PMF_EW(i) { sr[i] = sk[i]; yr[i] = yk[i]; }
                    fLastReset = f;
                    icycle = 1;
                }
            }
            PMF_EW(i) oldg[i] = g[i];                                                // :787
            tm.sync();
            oldf = f;
            oldgtp = c.dot(pk, g);
            ustpmax = stepmx / (c.nrm2(pk) + EPS);                                   // :792

            {   // stepMax (:1041-1067) with low = 0, up = +inf: a min over components
                // (the sequential recurrence `if (t > step*d) step = t/d` is order-free
                //  for d<0, t<=0: it keeps the smallest t/d seen)
                real m = ustpmax;
                if (STRICT) {   // keep the reference's sequential recurrence bit for bit
                    if (tm.rank() == 0)
                        for (int i = 0; i < n; i++)
                            if (pivot[i] == 0 && pk[i] < (real)0) {
                                const real t = ((real)0 - xo[i]) / xs[i] - x[i];
                                if (t > m * pk[i]) m = t / pk[i];
                            }
                    spe = tm.bcast0(m);
                } else {
                    PMF_EW(i) {
                        if (pivot[i] == 0 && pk[i] < (real)0) {
                            const real t = ((real)0 - xo[i]) / xs[i] - x[i];
                            if (t > m * pk[i]) m = t / pk[i];
                        }
                    }
                    spe = tm.min(m);
                }
            }

            if (spe > (real)0) {
                {   // initialStep (:1368-1383)
                    const real fm = fmin_ / fscale;
                    const real d = (real)fabs(D(f - fm));
                    alpha = 1;
                    if (D(d) * 2.0 <= D(-oldgtp) && d >= EPS) alpha = (real)(D(d) * -2.0 / D(oldgtp));
                    if (alpha >= spe) alpha = spe;
                }
                const int lsrc = tn_linesearch(c, fscale, eta, ftol, spe, pk, x, f, alpha, gfull);
                if (lsrc == LSR_FAIL) break;                                         // :818
                if (D(alpha) >= 0.9 * D(ustpmax)) stepmx = (real)(D(stepmx) * 1e2);  // :824
                if (D(alpha - spe) >= D(-EPS) * 10.0) newcon = true;                 // :833
                else {
                    if (lsrc != LSR_OK) break;
                    newcon = false;
                }
            } else newcon = true;

            if (newcon) {                                                            // :855-863, addConstraint :1072
                int added = 0;
                const real tolc = (real)(D(EPS) * 10.0 * (fabs(0.0) + 1.0));
                PMF_EW(i) {
                    if (pivot[i] == 0 && pk[i] != (real)0 && pk[i] < (real)0) {
                        if (x[i] * xs[i] + xo[i] - (real)0 <= tolc) {
                            pivot[i] = -1;
                            x[i] = ((real)0 - xo[i]) / xs[i];
                            added = 1;
                        }
                    }
                }
                added = tm.max(added);
                tm.sync();
                if (!added && c.nfeval == oldnfeval) break;                          // TNC_NOPROGRESS
                fLastConstraint = f;
            }

            difold = difnew;                                                         // :875-887
            difnew = oldf - f;
            if (icycle == 1) {
                if (D(difnew) > D(difold) * 2.0) epsred += epsred;
                if (D(difnew) < D(difold) * 0.5) epsred = (real)(D(epsred) * 0.5);
            }
            PMF_EW(i) {                                                              // :889-894
                const real gi = gfull[i] * (xs[i] * fscale);
                g[i] = gi;
                temp[i] = (pivot[i] != 0) ? (real)0 : gi;
            }
            tm.sync();
            gnorm = c.nrm2(temp);

            {   // removeConstraint (:1113-1146): argmin of -pivot*g, FIRST index on ties
                remcon = false;
                if (!((D(fLastConstraint - f) <= D(oldgtp) * -0.5) && (gnorm > pgtol * fscale))) {
                    real cmax = 0; int imax = 0x7fffffff;
                    PMF_EW(i) {
                        if (pivot[i] == 2) continue;
                        const real t = (real)(-pivot[i]) * g[i];
                        if (t < cmax) { cmax = t; imax = i; }   // strided scan keeps the first minimum per lane
                    }
                    const real best = tm.min(cmax);
                    if (best < (real)0) {
                        int cand = (cmax == best) ? imax : 0x7fffffff;
                        cand = tm.min(cand);
                        tm.sync();
                        if (tm.rank() == 0) pivot[cand] = 0;
                        remcon = true;
                    }
                    tm.sync();
                }
            }
            if (remcon) {                                                            // :901-907
                PMF_EW(i) temp[i] = (pivot[i] != 0) ? (real)0 : g[i];
                tm.sync();
                gnorm = c.nrm2(temp);
                fLastConstraint = f;
            }
            if (!remcon && !newcon) {                                                // :909-929
                if (fabs(D(difnew)) <= D(ftol * fscale)) break;
                if (alpha * c.nrm2(pk) <= xtol) break;
            }
            c.project(g);                                                            // :931

            if (!newcon) {                                                           // :940-962
                PMF_EW(i) { yk[i] = g[i] - oldg[i]; sk[i] = alpha * pk[i]; }
                tm.sync();
                yksk = c.dot(yk, sk);
                if (icycle == (n - 1) || difnew < epsred * (fLastReset - f)) lreset = true;
                else {
                    yrsr = c.dot(yr, sr);
                    lreset = (yrsr <= (real)0);
                }
                upd1 = false;
            }
        }
        // unscalex is never contracted into an FMA, not even in fast mode: a variable pinned at
        // the bound has x = (0 - xo)/xs, and only the separately rounded product gives back an
        // exact 0 (SURVEY.md §4.1 item 3: with FMA the reference's float build loses its sparsity)
        PMF_EW(i) {                                                                  // :971-972
            const real t = add_rn(mul_rn(x[i], xs[i]), xo[i]);
            x[i] = (t < (real)0) ? (real)0 : t;
        }
        tm.sync();
    }
    (void)solved;

    if (hc.early_stop) {                                                             // poismf.c:393-396
        PMF_EW(i) prev[i] = prev[i] + (real)(-1.) * x[i];
        tm.sync();
        const real dd = c.dot(prev, prev);
        if (tm.rank() == 0 && tm.owns_row() && D(dd) <= 1e-4) atomicAdd(n_unchanged, 1ULL);
    }
}

#undef PMF_EW
}  // namespace pmf
