// theta_transform.cuh -- per-theta prologue of the log-density kernels (K2 in DESIGN.md).
//
// theta -> AR roots, MA coefficients, sigma^2, prior bounds, log-prior, and the constants of
// the Kalman filter in the rotated state space, reduced to its independent real half.
//
// Reference behaviour restated here (paths relative to /root/reference/src):
//   CARp::ARRoots                 carpack.cpp:137-172
//   CARp::CheckPriorBounds        carpack.cpp:314-374   (CAR1: 116-130, base: carpack.hpp:178-191)
//   CARp::Variance                carpack.cpp:377-409
//   CARMA::ExtractMA / polycoefs  carpack.cpp:522-580, 742-756
//   ZCARMA::ExtractMA / LogPrior  carpack.cpp:687-698, carpack.hpp:444-456
//   CARMA_Base::LogPrior          carpack.hpp:118-126
//   KalmanFilterp::Reset          kfilter.cpp:138-186  (J, rotated MA coefficients b, stationary V)
//
// Rotated state space, real half.  The AR roots produced by ARRoots are, per quadratic factor,
// either a complex-conjugate pair or two real roots (plus one real root when p is odd), and the MA
// coefficients are real.  Hence the rotated state x (kfilter.cpp:194-201) satisfies
// x_{2s+1} = conj(x_{2s}) on a conjugate pair and is real on real roots, and the covariance P has
// only p(p+1)/2 independent real numbers.  We carry z = (Re x_{2s}, Im x_{2s}) for a conjugate pair,
// (x_{2s}, x_{2s+1}) for a real pair, and x_{p-1} for the odd root; the observation row b becomes
// the real row c, and Cov(z, y) under the stationary law becomes the real vector h = V b^H.
// (The components are additionally rescaled by their MA coefficient so that c is a 0/1 row: see the
// "real half" block at the end of transform_theta.)
#pragma once
#include <math.h>

#include "../../include/carma_b200.h"
#include "device_math.cuh"
#include "fast_math.cuh"

namespace carma {

constexpr int MAX_P = CARMA_MAX_P;
constexpr int MAX_D = 3 + MAX_P + MAX_P;  // >= 3+p+q and 4+p

__host__ __device__ inline int model_dim(int kind, int p, int q) {
    if (kind == CARMA_KIND_CAR1) return 4;
    if (kind == CARMA_KIND_CARMA) return 3 + p + q;
    if (kind == CARMA_KIND_ZCARMA) return 4 + p;
    return 3 + p;
}

template <int P>
struct RealParams {
    // Rates pre-multiplied by the table step of fast_math.cuh (64/ln2 for decays, 64/pi for phases):
    //   slot s < P/2, conjugate pair w, conj(w): le[s] = Re w * 64/ln2,      ls[s] = Im w * 64/pi  (first root: Im <= 0)
    //                 real pair w_b < w_a < 0  : le[s] = w_a * 64/ln2,       ls[s] = (w_b - w_a) * 64/ln2  (<= 0)
    //   odd P: le[P/2] = w_{P-1} * 64/ln2
    // Components: conjugate pair -> (Re, Im) of the MA-normalised rotated state; real pair -> (x_a + x_b, x_a - x_b);
    // the observation is the sum of the FIRST component of every slot (+ the odd root's), for every kind of slot.
    double le[(P + 1) / 2];
    double ls[P / 2 > 0 ? P / 2 : 1];
    double h[P];  // stationary Cov(z, y)
    double v0;    // stationary Var(y) = Re(b V b^H)
    double scale, mu, logprior;
    unsigned cmask;  // bit s set: slot s is a conjugate pair
};

// observation row of the real basis: 1 on the first component of every 2x2 slot and on the odd root
template <int P>
__host__ __device__ constexpr double obs_c(int k) { return ((k & 1) == 0) ? 1.0 : 0.0; }

// Largest |rate * dt| in table steps the range reductions accept: rates are clamped to it in transform_theta
// (dt_max = the longest gap of the series).  Unreachable inside the prior (|w| <= 2 pi / dt_min) unless
// dt_max / dt_min > 2e6; beyond it e^{w dt} differs from 0 by less than e^{-2^30 ln2/64 dt_min/dt_max}.
constexpr double RATE_CAP_STEPS = 1073741824.0;         // 2^30: exp, k fits an int
constexpr double PHASE_CAP_STEPS = 1125899906842624.0;  // 2^50: sin/cos, t = x + MAGIC exact

enum { TT_OK = 0, TT_NEG_INF = 1 };

// ---- divisions of the prologue.  An IEEE FP64 division costs ~14 issued instructions on sm_100a (reciprocal seed,
// Newton steps, range check, a branch around the slow-path call) and splits the basic block; the round-1 prologue
// executed ~170 of them per theta and was 17-19 % of K1 at ny = 270.  Here: one branch-free reciprocal-multiply with
// a residual correction (error < 1 ulp; operands are normal numbers for every theta the prior admits -- a
// denominator outside the normal range yields a non-finite result, which transform_theta catches at its end and
// redoes with IEEE divisions), complex divisions as ONE complex reciprocal times a complex product (what LAPACK's
// zgetf2 does with the pivots: it scales the column by 1/pivot), and no division at all in the prior-bound tests
// unless a value falls within 1e-12 relative of its bound.
template <bool FAST>
__host__ __device__ __forceinline__ double div_(double a, double b) {
    if (!FAST) return a / b;
    const double r = rcp_fast(b);
    const double q = a * r;
    return fma(fma(-b, q, a), r, q);
}
// 1 / b, Smith's scaling (robust against overflow of |b|^2)
template <bool FAST>
__host__ __device__ __forceinline__ cxd crcp(cxd b) {
    if (fabs(b.re) >= fabs(b.im)) {
        const double r = div_<FAST>(b.im, b.re), den = fma(b.im, r, b.re);
        const double id = div_<FAST>(1.0, den);
        return cxd{id, -r * id};
    } else {
        const double r = div_<FAST>(b.re, b.im), den = fma(b.re, r, b.im);
        const double id = div_<FAST>(1.0, den);
        return cxd{r * id, -id};
    }
}
template <bool FAST>
__host__ __device__ __forceinline__ cxd cdiv_(cxd a, cxd b) {
    if (!FAST) return cdiv(a, b);
    return a * crcp<true>(b);
}
template <bool FAST>
__host__ __device__ __forceinline__ cxd cdiv_simple(cxd a, cxd b) {
    double inv = div_<FAST>(1.0, b.re * b.re + b.im * b.im);
    return cxd{(a.re * b.re + a.im * b.im) * inv, (a.im * b.re - a.re * b.im) * inv};
}

// roots of prod_s (q1_s + q2_s x + x^2) [ * (x + q_last) ]  from log quadratic terms
template <int N>
__host__ __device__ __forceinline__ unsigned quad_roots_dev(const double* logq, int n, cxd* w) {
    unsigned cmask = 0;
#pragma unroll
    for (int s = 0; s < N / 2; s++) {
        if (2 * s + 1 < n) {
            double q1 = exp(logq[2 * s]);
            double q2 = exp(logq[2 * s + 1]);
            // no FMA contraction here: the sign of the discriminant selects the branch
#ifdef __CUDA_ARCH__
            double disc = __dsub_rn(__dmul_rn(q2, q2), __dmul_rn(4.0, q1));
#else
            volatile double q2q2 = q2 * q2;
            double disc = q2q2 - 4.0 * q1;
#endif
            if (disc > 0) {
                double sq = sqrt(disc);
                w[2 * s] = cx(-0.5 * (q2 + sq), 0.0);
                w[2 * s + 1] = cx(-0.5 * (q2 - sq), 0.0);
            } else {
                double re = -0.5 * q2;
                double im = -0.5 * sqrt(-disc);
                w[2 * s] = cx(re, im);
                w[2 * s + 1] = cx(re, -im);
                cmask |= 1u << s;
            }
        }
    }
    if (n & 1) w[n - 1] = cx(-exp(logq[n - 1]), 0.0);
    return cmask;
}

// Solve E J = e_{P-1} with E(i,k) = w_k^i (kfilter.cpp:144-158) by LU with partial pivoting
// (pivot = max |re|+|im|, as LAPACK izamax).  Fully unrolled, row swaps predicated, so everything
// stays in registers.  Returns false on an exactly singular system.
template <int P, bool FAST>
__host__ __device__ __forceinline__ bool vandermonde_solve_last(const cxd* w, cxd* J) {
    cxd A[P][P];
    cxd rhs[P], pinv[P];
#pragma unroll
    for (int k = 0; k < P; k++) {
        cxd pw = cx(1, 0);
        A[0][k] = pw;
#pragma unroll
        for (int i = 1; i < P; i++) {
            pw = pw * w[k];
            A[i][k] = pw;
        }
        rhs[k] = cx(k == P - 1 ? 1.0 : 0.0, 0.0);
    }
    bool ok = true;
#pragma unroll
    for (int k = 0; k < P; k++) {
        int piv = k;
        double best = fabs(A[k][k].re) + fabs(A[k][k].im);
#pragma unroll
        for (int i = k + 1; i < P; i++) {
            double v = fabs(A[i][k].re) + fabs(A[i][k].im);
            if (v > best) { best = v; piv = i; }
        }
        if (!(best > 0.0) || !isfinite(best)) ok = false;
#pragma unroll
        for (int i = k + 1; i < P; i++) {
            if (i == piv) {
#pragma unroll
                for (int j = k; j < P; j++) { cxd tmp = A[k][j]; A[k][j] = A[i][j]; A[i][j] = tmp; }
                cxd tr = rhs[k]; rhs[k] = rhs[i]; rhs[i] = tr;
            }
        }
        pinv[k] = crcp<FAST>(A[k][k]);  // one reciprocal per pivot: column scaled by it, reused in the back-substitution
#pragma unroll
        for (int i = k + 1; i < P; i++) {
            cxd l = FAST ? A[i][k] * pinv[k] : cdiv(A[i][k], A[k][k]);
#pragma unroll
            for (int j = k + 1; j < P; j++) A[i][j] = A[i][j] - l * A[k][j];
            rhs[i] = rhs[i] - l * rhs[k];
        }
    }
#pragma unroll
    for (int i = P - 1; i >= 0; i--) {
        cxd s = rhs[i];
#pragma unroll
        for (int j = i + 1; j < P; j++) s = s - A[i][j] * J[j];
        J[i] = FAST ? s * pinv[i] : cdiv(s, A[i][i]);
    }
    return ok;
}

// Same elimination, same operation order (bit-identical J), with the P x P complex matrix held in shared
// memory instead of registers: element (i,j) of the calling thread is scr[((i*P + j)*2 + {0,1}) * stride].
// K1 uses it: 100 registers' worth of matrix no longer compete with the 128-register cap of the kernel, so the
// prologue stops spilling ~1 kB per thread to local memory (which reached DRAM as dead write-backs).
template <int P, bool FAST>
__host__ __device__ __forceinline__ bool vandermonde_solve_last_smem(const cxd* w, cxd* J, double* scr, int stride) {
    auto ld = [&](int i, int j) { const double* q = scr + (size_t)((i * P + j) * 2) * stride; return cxd{q[0], q[stride]}; };
    auto st = [&](int i, int j, cxd v) { double* q = scr + (size_t)((i * P + j) * 2) * stride; q[0] = v.re; q[stride] = v.im; };
    cxd rhs[P], pinv[P];
#pragma unroll
    for (int k = 0; k < P; k++) {
        cxd pw = cx(1, 0);
        st(0, k, pw);
#pragma unroll
        for (int i = 1; i < P; i++) {
            pw = pw * w[k];
            st(i, k, pw);
        }
        rhs[k] = cx(k == P - 1 ? 1.0 : 0.0, 0.0);
    }
    bool ok = true;
#pragma unroll
    for (int k = 0; k < P; k++) {
        int piv = k;
        cxd akk = ld(k, k);
        double best = fabs(akk.re) + fabs(akk.im);
#pragma unroll
        for (int i = k + 1; i < P; i++) {
            cxd a = ld(i, k);
            double v = fabs(a.re) + fabs(a.im);
            if (v > best) { best = v; piv = i; }
        }
        if (!(best > 0.0) || !isfinite(best)) ok = false;
        if (piv != k) {  // rows addressed at run time: free in shared memory
#pragma unroll
            for (int j = k; j < P; j++) { cxd a = ld(k, j), b = ld(piv, j); st(k, j, b); st(piv, j, a); }
        }
#pragma unroll
        for (int i = k + 1; i < P; i++) {  // the right-hand side stays in registers: predicated exchange
            if (i == piv) { cxd tr = rhs[k]; rhs[k] = rhs[i]; rhs[i] = tr; }
        }
        akk = ld(k, k);
        pinv[k] = crcp<FAST>(akk);
        cxd rowk[P];  // row k of the active block stays in registers for the whole column
#pragma unroll
        for (int j = k + 1; j < P; j++) rowk[j] = ld(k, j);
#pragma unroll
        for (int i = k + 1; i < P; i++) {
            cxd l = FAST ? ld(i, k) * pinv[k] : cdiv(ld(i, k), akk);
#pragma unroll
            for (int j = k + 1; j < P; j++) st(i, j, ld(i, j) - l * rowk[j]);
            rhs[i] = rhs[i] - l * rhs[k];
        }
    }
#pragma unroll
    for (int i = P - 1; i >= 0; i--) {
        cxd s = rhs[i];
#pragma unroll
        for (int j = i + 1; j < P; j++) s = s - ld(i, j) * J[j];
        J[i] = FAST ? s * pinv[i] : cdiv(s, ld(i, i));
    }
    return ok;
}

// Returns TT_NEG_INF when the log-density is -inf (bounds violated / singular), else TT_OK.
// __noinline__: the prologue (LU on a PxP complex matrix) gets its own register allocation, so it
// cannot push spills into the time loop of the calling kernel.
// Vr (optional): packed upper triangle (row-major, P(P+1)/2) of the stationary covariance in the real
// basis, V_r = T V T^H restricted to its real part, where z = T x.  Only the scan kernels need it.
// lu_scratch (optional, SMEM_LU): this thread's slot of a shared-memory scratch of 2 P^2 doubles per thread,
// laid out [element][thread] with `lu_stride` threads (see vandermonde_solve_last_smem).
// dt_max: longest sampling gap of the series the parameters will be used on (rate clamp, see RATE_CAP_STEPS).
// A model given by its state-space parameters instead of theta (the KalmanFilterp class API: sigsqr, omega, ma --
// kfilter.hpp:303-334).  The roots must be closed under conjugation and arranged in slots by the host (series.h:
// arrange_roots): slot s holds a conjugate pair (first root Im <= 0, bit s of cmask set) or two real roots, an odd
// order ends with one real root.
struct ExplicitModel {
    double sigsqr, scale, mu;
    double w_re[MAX_P], w_im[MAX_P];
    double ma[MAX_P];
    unsigned cmask;
};

// FAST: the reciprocal-multiply divisions above (hot path); !FAST: IEEE divisions (reached only when the fast
// evaluation produced a non-finite constant, i.e. some denominator left the normal range).
// EXPLICIT: roots, MA coefficients, sigma^2, scale and mu come from `ex` (no bounds, no prior); th is not read.
template <int P, bool WITH_V, bool SMEM_LU, bool FAST, bool EXPLICIT = false>
__host__ __device__ __noinline__ int transform_theta_impl(int kind, int q, unsigned flags, const carma_prior_t& pr,
                                                          const double* th, double dt_max, RealParams<P>& out, double* Vr,
                                                          double* lu_scratch, int lu_stride, const ExplicitModel* ex = nullptr) {
    constexpr double PI = 3.14159265358979323846;
    const double ysigma = EXPLICIT ? 0.0 : th[0], scale = EXPLICIT ? ex->scale : th[1];
    out.scale = scale;
    out.mu = EXPLICIT ? ex->mu : th[2];

    cxd w[P];
    unsigned cmask = 0;
    if (EXPLICIT) {
#pragma unroll
        for (int i = 0; i < P; i++) w[i] = cx(ex->w_re[i], ex->w_im[i]);
        cmask = ex->cmask;
    } else if (kind == CARMA_KIND_CAR1) {
        // carpack.hpp:265: omega = exp(theta3); the state-space root is -omega
        w[0] = cx(-exp(th[3]), 0.0);
    } else {
        cmask = quad_roots_dev<P>(th + 3, P, w);
    }
    out.cmask = cmask;

    // ---- prior bounds
    if (EXPLICIT) {
        // none: an explicit model is taken as given
    } else if (kind == CARMA_KIND_CAR1) {
        double omega = -w[0].re;
        if ((omega > pr.max_freq) || (omega < pr.min_freq) || (ysigma > pr.max_stdev) || (ysigma < 0) ||
            (scale < 0.5) || (scale > 2.0))
            return TT_NEG_INF;
    } else if (!(flags & CARMA_IGNORE_BOUNDS)) {
        bool ok = true;
        if ((ysigma > pr.max_stdev) || (ysigma < 0) || (scale < 0.5) || (scale > 2.0)) ok = false;
        // centroid / width bounds and ordering (carpack.cpp:318-352): x / 2 / pi against a bound.  The product
        // x * (1/2pi) is within 2 ulp of that quotient; only a comparison closer than 1e-12 relative to its
        // threshold is redone with the reference's divisions.
        // unique_roots(ar_roots, 1e-4) (carpack.cpp:709-732): |(w_i - w_j) / (w_i + w_j)| > 1e-4 for every pair, decided
        // on the squared moduli unless the ratio is within 1e-9 of the threshold.
        bool unsure = false;
        if (FAST) {
            constexpr double INV2PI = 0.15915494309189533576888;
            constexpr double G = 1e-12;
            double prev_cent = 0.0;
#pragma unroll
            for (int i = 0; i < P; i++) {
                const double cent = fabs(w[i].im) * INV2PI, width = -w[i].re * INV2PI;
                ok = ok && (cent < pr.max_freq) && (width < pr.max_freq) && (width > pr.min_freq);
                unsure = unsure || (fabs(cent - pr.max_freq) <= G * pr.max_freq) || (fabs(width - pr.max_freq) <= G * pr.max_freq) ||
                         (fabs(width - pr.min_freq) <= G * pr.min_freq);
                if (i > 0) {
                    const double gap = cent - prev_cent;
                    if (gap > 1e-8) ok = false;
                    unsure = unsure || (fabs(gap - 1e-8) <= G * fmax(cent, prev_cent));
                }
                prev_cent = cent;
            }
#pragma unroll
            for (int i = 0; i < P - 1; i++)
#pragma unroll
                for (int j = i + 1; j < P; j++) {
                    const cxd dmn = w[i] - w[j], sm = w[i] + w[j];
                    const double n2 = dmn.re * dmn.re + dmn.im * dmn.im, d2 = sm.re * sm.re + sm.im * sm.im;
                    if (!(n2 > 1.000000001e-8 * d2)) {
                        if (n2 < 0.999999999e-8 * d2) ok = false;
                        else unsure = true;  // also NaN / overflowed squares
                    }
                }
        }
        if (!FAST || unsure) {
            ok = !((ysigma > pr.max_stdev) || (ysigma < 0) || (scale < 0.5) || (scale > 2.0));
            double prev_cent = 0.0;
#pragma unroll
            for (int i = 0; i < P; i++) {
                double cent = fabs(w[i].im) / 2.0 / PI;
                double width = -w[i].re / 2.0 / PI;
                ok = ok && (cent < pr.max_freq) && (width < pr.max_freq) && (width > pr.min_freq);
                if (i > 0 && (cent - prev_cent > 1e-8)) ok = false;
                prev_cent = cent;
            }
            double min_frac = 100.0 * 1e-4;
#pragma unroll
            for (int i = 0; i < P - 1; i++)
#pragma unroll
                for (int j = i + 1; j < P; j++) {
                    double frac = cabs_(cdiv(w[i] - w[j], w[i] + w[j]));
                    if (frac < min_frac) min_frac = frac;
                }
            if (!(min_frac > 1e-4)) ok = false;
        }
        if (!ok) return TT_NEG_INF;
    }

    // ---- MA coefficients
    double ma[P];
#pragma unroll
    for (int i = 0; i < P; i++) ma[i] = (i == 0) ? 1.0 : 0.0;
    if (EXPLICIT) {
#pragma unroll
        for (int i = 0; i < P; i++) ma[i] = ex->ma[i];
    } else if (kind == CARMA_KIND_CARMA && q > 0) {
        cxd r[P];
#pragma unroll
        for (int i = 0; i < P; i++) r[i] = cx(0, 0);
        quad_roots_dev<P>(th + 3 + P, q, r);
        if (SMEM_LU) {
            // polynomial from its roots (carpack.cpp:742-756) with the run-time-indexed coefficient array in the
            // shared scratch (free before the LU needs it) instead of local memory
            auto ld = [&](int j) { const double* p_ = lu_scratch + (size_t)(2 * j) * lu_stride; return cxd{p_[0], p_[lu_stride]}; };
            auto st = [&](int j, cxd v) { double* p_ = lu_scratch + (size_t)(2 * j) * lu_stride; p_[0] = v.re; p_[lu_stride] = v.im; };
            st(0, cx(1.0, 0.0));
            for (int j = 1; j <= q; j++) st(j, cx(0, 0));
#pragma unroll
            for (int i = 0; i < P; i++)
                if (i < q)
                    for (int j = i + 1; j >= 1; j--) st(j, ld(j) - r[i] * ld(j - 1));
            const double norm = ld(q).re;
#pragma unroll
            for (int i = 0; i < P; i++)
                if (i <= q) ma[i] = div_<FAST>(ld(q - i).re, norm);
        } else {
            cxd cf[P];
#pragma unroll
            for (int i = 0; i < P; i++) cf[i] = cx(0, 0);
            cf[0] = cx(1.0, 0.0);
            for (int i = 0; i < q; i++)
                for (int j = i + 1; j >= 1; j--) cf[j] = cf[j] - r[i] * cf[j - 1];
            double norm = cf[q].re;
            for (int i = 0; i <= q; i++) ma[i] = div_<FAST>(cf[q - i].re, norm);
        }
    } else if (kind == CARMA_KIND_ZCARMA) {
        double x = th[3 + P];
        double kn = exp(x) / (1.0 + exp(x));
        double kappa = (pr.kappa_high - pr.kappa_low) * kn + pr.kappa_low;
        double binom = 1.0;
#pragma unroll
        for (int i = 1; i < P; i++) {
            binom = binom * (double)(P - i) / (double)i;  // C(P-1, i)
            ma[i] = rint(binom) / pow(kappa, (double)i);
        }
    }

    // ---- rotated MA row b_k = beta(w_k), beta(-w_k), and Variance(w, beta, sigma=1)
    cxd b[P];
    cxd var_acc = cx(0, 0);
#pragma unroll
    for (int k = 0; k < P; k++) {
        cxd s1 = cx(ma[P - 1], 0), s2 = cx(ma[P - 1], 0);
        cxd mw = -w[k];
#pragma unroll
        for (int l = P - 2; l >= 0; l--) {
            s1 = s1 * w[k] + cx(ma[l], 0);
            s2 = s2 * mw + cx(ma[l], 0);
        }
        b[k] = s1;
        cxd dp = cx(1, 0);
#pragma unroll
        for (int l = 0; l < P; l++)
            if (l != k) dp = dp * ((w[l] - w[k]) * (conj(w[l]) + w[k]));
        cxd denom = (-2.0 * w[k].re) * dp;
        var_acc = var_acc + cdiv_<FAST>(s1 * s2, denom);
    }
    double sigsqr;
    if (EXPLICIT)
        sigsqr = ex->sigsqr;
    else if (kind == CARMA_KIND_CAR1)
        sigsqr = 2.0 * ysigma * ysigma * (-w[0].re);  // carpack.hpp:272-274
    else
        sigsqr = div_<FAST>(ysigma * ysigma, var_acc.re);  // carpack.hpp:316-319, 391-395

    // ---- J = E^{-1} e_p for the Vandermonde E (kfilter.cpp:144-158): LU with partial pivoting, as
    // arma::solve -> zgesv does.  (The closed form J_k = 1/prod_{l!=k}(w_k - w_l) has a smaller forward
    // error per element but is NOT what the reference computes: the LU solution is backward stable,
    // i.e. exact for slightly perturbed roots, and the massive cancellation in b V b^H for clustered
    // roots is benign under such consistent perturbations while it amplifies independent ones.)
    cxd J[P];
    bool solved;
    if (SMEM_LU) solved = vandermonde_solve_last_smem<P, FAST>(w, J, lu_scratch, lu_stride);
    else solved = vandermonde_solve_last<P, FAST>(w, J);
    if (!solved) return TT_NEG_INF;  // arma::solve throws -> -inf (carpack.hpp:154-164)

    // ---- stationary covariance V (kfilter.cpp:165-172), h = V b^H, v0 = Re(b V b^H)
    cxd h[P];
#pragma unroll
    for (int i = 0; i < P; i++) h[i] = cx(0, 0);
    cxd Vfull[WITH_V ? P : 1][WITH_V ? P : 1];  // only materialised for the scan kernels
#pragma unroll
    for (int i = 0; i < P; i++) {
#pragma unroll
        for (int j = i; j < P; j++) {
            cxd num = (-sigsqr) * (J[i] * conj(J[j]));
            cxd vij = cdiv_simple<FAST>(num, w[i] + conj(w[j]));
            h[i] = h[i] + vij * conj(b[j]);
            if (j > i) h[j] = h[j] + conj(vij) * conj(b[i]);
            if (WITH_V) { Vfull[i][j] = vij; Vfull[j][i] = conj(vij); }
        }
    }
    if (WITH_V) {
        // z_m = sum_k T[m][k] x_k with at most two non-zeros per row (x^_k = s_k x_k, s = 2b on a conjugate pair,
        // b on a real root):
        //   conjugate pair (a, a+1): u = (x^_a + conj-partner)/2, v = (x^_a - partner)/(2i)
        //   real pair (a = 2s+1, b = 2s): u = x^_a + x^_b, v = x^_a - x^_b;   odd root: z = x^
        int k0[P], k1[P];
        cxd t0[P], t1[P];
#pragma unroll
        for (int m = 0; m < P; m++) {
            int s = m >> 1;
            const bool in_slot = m < 2 * (P / 2);
            bool is_c = in_slot && ((cmask >> s) & 1u);
            if (is_c) {
                k0[m] = 2 * s; k1[m] = 2 * s + 1;
                cxd sc = 2.0 * b[2 * s];
                if ((m & 1) == 0) { t0[m] = 0.5 * sc; t1[m] = 0.5 * conj(sc); }
                else { t0[m] = cx(0.0, -0.5) * sc; t1[m] = cx(0.0, 0.5) * conj(sc); }
            } else if (in_slot) {
                k0[m] = 2 * s + 1; k1[m] = 2 * s;
                t0[m] = cx(b[2 * s + 1].re, 0.0);
                t1[m] = cx(((m & 1) == 0) ? b[2 * s].re : -b[2 * s].re, 0.0);
            } else {
                k0[m] = m; k1[m] = m; t0[m] = cx(b[m].re, 0.0); t1[m] = cx(0.0, 0.0);
            }
        }
        int o = 0;
        for (int m = 0; m < P; m++)
            for (int n = m; n < P; n++) {
                cxd acc = t0[m] * Vfull[k0[m]][k0[n]] * conj(t0[n]) + t0[m] * Vfull[k0[m]][k1[n]] * conj(t1[n]) +
                          t1[m] * Vfull[k1[m]][k0[n]] * conj(t0[n]) + t1[m] * Vfull[k1[m]][k1[n]] * conj(t1[n]);
                Vr[o++] = acc.re;
            }
    }
    double v0 = 0.0;
#pragma unroll
    for (int i = 0; i < P; i++) v0 += b[i].re * h[i].re - b[i].im * h[i].im;
    out.v0 = v0;

    // ---- real half, in the observation-normalised basis.  Each rotated component is rescaled by its own
    // MA coefficient, x^_k = s_k x_k with s = 2 b (conjugate pair) or b (real root); the scaling commutes
    // with the diagonal transition, and the observation becomes y = sum of the FIRST component of every
    // slot: a real pair is carried as (x^_a + x^_b, x^_a - x^_b), a = the root closer to zero, so its
    // transition e^{w_a dt} [[ch, sh], [sh, ch]] has the shape of a rotation (fast_math.cuh) and the time
    // loop needs neither multiplications by b nor a per-lane observation row.
    const double rate_cap = RATE_CAP_STEPS / dt_max, phase_cap = PHASE_CAP_STEPS / dt_max;
#pragma unroll
    for (int s = 0; s < P / 2; s++) {
        if ((cmask >> s) & 1u) {
            out.le[s] = fmax(w[2 * s].re * K_EXP_SCALE, -rate_cap);
            out.ls[s] = fmax(w[2 * s].im * K_ROT_SCALE, -phase_cap);
            // h restricted to the conjugate-symmetric subspace: (h_{2s} + conj(h_{2s+1})) / 2.  The LU
            // solution J is not exactly conjugate-symmetric (its error is cond(E) eps, consistent across
            // components); averaging keeps c.h == Re(b V b^H) to rounding, which is what the reference's
            // full complex recursion sees to first order in that asymmetry.
            cxd hs = cx(0.5 * (h[2 * s].re + h[2 * s + 1].re), 0.5 * (h[2 * s].im - h[2 * s + 1].im));
            cxd sc = 2.0 * b[2 * s];
            cxd hh = sc * hs;
            out.h[2 * s] = hh.re;
            out.h[2 * s + 1] = hh.im;
        } else {
            // ARRoots order: w[2s] = -(q2 + sqrt(disc))/2 < w[2s+1] = -(q2 - sqrt(disc))/2 < 0
            out.le[s] = fmax(w[2 * s + 1].re * K_EXP_SCALE, -rate_cap);
            out.ls[s] = fmax((w[2 * s].re - w[2 * s + 1].re) * K_EXP_SCALE, -rate_cap);
            const double ha = b[2 * s + 1].re * h[2 * s + 1].re, hb = b[2 * s].re * h[2 * s].re;
            out.h[2 * s] = ha + hb;
            out.h[2 * s + 1] = ha - hb;
        }
    }
    if (P & 1) {
        out.le[P / 2] = fmax(w[P - 1].re * K_EXP_SCALE, -rate_cap);
        out.h[P - 1] = b[P - 1].re * h[P - 1].re;
    }
    if (P < 2) out.ls[0] = 0.0;

    // ---- log prior (carpack.hpp:118-126, 444-456)
    double lp = 0.0;
    if (!EXPLICIT && !(flags & CARMA_LOGLIK_ONLY)) {
        lp = -0.5 * pr.measerr_dof / scale - (1.0 + pr.measerr_dof / 2.0) * log(scale);
        if (kind == CARMA_KIND_ZCARMA) {
            double x = th[3 + P];
            lp += -x - 2.0 * log(1.0 + exp(-x));
        }
    }
    out.logprior = lp;
    return TT_OK;
}

template <int P, bool WITH_V = false, bool SMEM_LU = false>
__host__ __device__ __forceinline__ int transform_theta(int kind, int q, unsigned flags, const carma_prior_t& pr,
                                                        const double* th, double dt_max, RealParams<P>& out,
                                                        double* Vr = nullptr, double* lu_scratch = nullptr, int lu_stride = 0) {
    int st = transform_theta_impl<P, WITH_V, SMEM_LU, true>(kind, q, flags, pr, th, dt_max, out, Vr, lu_scratch, lu_stride);
    if (st == TT_OK) {
        // every constant of the recursion must be finite; otherwise a denominator left the range of the fast
        // reciprocal (or theta itself is absurd): let the IEEE-division version decide
        double chk = out.v0;
#pragma unroll
        for (int i = 0; i < P; i++) chk += out.h[i];
        if (!isfinite(chk)) st = transform_theta_impl<P, WITH_V, SMEM_LU, false>(kind, q, flags, pr, th, dt_max, out, Vr, lu_scratch, lu_stride);
    }
    return st;
}

// The constants of the recursion for an explicit model (fast divisions first, IEEE divisions if anything is not finite).
template <int P, bool WITH_V = false>
__host__ __device__ __forceinline__ int explicit_constants(const ExplicitModel& ex, double dt_max, RealParams<P>& out,
                                                           double* Vr = nullptr) {
    const carma_prior_t pr{};
    int st = transform_theta_impl<P, WITH_V, false, true, true>(CARMA_KIND_CARMA, 0, 0u, pr, nullptr, dt_max, out, Vr, nullptr, 0, &ex);
    if (st == TT_OK) {
        double chk = out.v0;
#pragma unroll
        for (int i = 0; i < P; i++) chk += out.h[i];
        if (!isfinite(chk))
            st = transform_theta_impl<P, WITH_V, false, false, true>(CARMA_KIND_CARMA, 0, 0u, pr, nullptr, dt_max, out, Vr, nullptr, 0, &ex);
    }
    return st;
}

// One theta row -> AR roots w, MA coefficients ma (beta_0 = 1, zero beyond q; ZCARMA: binomial / kappa^i) and sigma^2 of
// the driving noise, with the formulas of CarmaSample._ar_roots / _ma_coefs / _sigma_noise (Car1Sample for CAR(1):
// sigma^2 = 2 omega var) and IEEE division throughout.  pr: only the kappa bounds are read (ZCARMA).  AR_POLY: also the
// AR polynomial prod (x - w_k), highest power first (numpy.poly), into ac[P + 1].  Shared by derived_params_kernel
// (loglik.cu) and the PSD kernels (posterior.cu).
template <int P, bool AR_POLY = false>
__device__ __forceinline__ double derive_row(int kind, int q, const carma_prior_t& pr, const double* th, cxd* w, double* ma,
                                             cxd* ac = nullptr) {
    if (kind == CARMA_KIND_CAR1) w[0] = cx(-exp(th[3]), 0.0);
    else quad_roots_dev<P>(th + 3, P, w);
    if (AR_POLY) {
        ac[0] = cx(1.0, 0.0);
#pragma unroll
        for (int i = 1; i <= P; i++) ac[i] = cx(0.0, 0.0);
#pragma unroll
        for (int i = 0; i < P; i++)
#pragma unroll
            for (int j = P; j >= 1; j--)
                if (j <= i + 1) ac[j] = ac[j] - w[i] * ac[j - 1];
    }
    // MA coefficients (carpack.cpp:522-580, 687-698)
#pragma unroll
    for (int i = 0; i < P; i++) ma[i] = (i == 0) ? 1.0 : 0.0;
    if (kind == CARMA_KIND_CARMA && q > 0) {
        cxd rt[P], cf[P];
#pragma unroll
        for (int i = 0; i < P; i++) { rt[i] = cx(0, 0); cf[i] = cx(0, 0); }
        quad_roots_dev<P>(th + 3 + P, q, rt);
        cf[0] = cx(1.0, 0.0);
        for (int i = 0; i < q; i++)
            for (int j = i + 1; j >= 1; j--) cf[j] = cf[j] - rt[i] * cf[j - 1];
        const double norm = cf[q].re;
        for (int i = 0; i <= q; i++) ma[i] = cf[q - i].re / norm;
    } else if (kind == CARMA_KIND_ZCARMA) {
        const double x = th[3 + P];
        const double kn = exp(x) / (1.0 + exp(x));
        const double kappa = (pr.kappa_high - pr.kappa_low) * kn + pr.kappa_low;
        double binom = 1.0;
#pragma unroll
        for (int i = 1; i < P; i++) {
            binom = binom * (double)(P - i) / (double)i;
            ma[i] = rint(binom) / pow(kappa, (double)i);
        }
    }
    // Variance(w, beta, sigma = 1) (carpack.cpp:377-409) -> sigma^2 = var / Variance
    cxd var_acc = cx(0, 0);
#pragma unroll
    for (int k = 0; k < P; k++) {
        cxd s1 = cx(ma[P - 1], 0), s2 = cx(ma[P - 1], 0);
        const cxd mw = -w[k];
#pragma unroll
        for (int l = P - 2; l >= 0; l--) {
            s1 = s1 * w[k] + cx(ma[l], 0);
            s2 = s2 * mw + cx(ma[l], 0);
        }
        cxd dp = cx(1, 0);
#pragma unroll
        for (int l = 0; l < P; l++)
            if (l != k) dp = dp * ((w[l] - w[k]) * (conj(w[l]) + w[k]));
        var_acc = var_acc + cdiv(s1 * s2, (-2.0 * w[k].re) * dp);
    }
    const double ysigma = th[0];
    return (kind == CARMA_KIND_CAR1) ? 2.0 * ysigma * ysigma * (-w[0].re) : ysigma * ysigma / var_acc.re;
}

}  // namespace carma
