// kalman_real.cuh -- the CARMA(p,q) Kalman filter recursion, one filter per thread, whole state
// in registers (K1 in DESIGN.md).
//
// Reference recursion restated (paths relative to /root/reference/src):
//   KalmanFilterp::Reset   kfilter.cpp:138-186     P = V, x = 0, var_0 = Re(b V b^H) + yerr_0^2
//   KalmanFilterp::Update  kfilter.cpp:189-215     K = P b^H / var;  x += K innov;  P -= var K K^H;
//                                                  rho = exp(omega dt); x = rho o x;
//                                                  P = (rho rho^H) o (P - V) + V;
//                                                  mean = Re(b x); var = Re(b P b^H) + yerr^2
//   CARMA_Base::LogDensity carpack.hpp:167-171     ll = sum -1/2 log var_i - 1/2 (y_i - mean_i - mu)^2 / var_i
//
// What is different from a transliteration (all exact algebraic identities):
//   * the state is the independent real half z of the rotated complex state (theta_transform.cuh);
//     the Hadamard product (rho rho^H) o . becomes the block-diagonal congruence Phi . Phi^T with 2x2
//     blocks  e^{a dt} [[cos, -sin],[sin, cos]]  (conjugate pair) or  e^{a dt} [[ch, sh],[sh, ch]]  (two real
//     roots, in the sum/difference basis): every block is [[A, sB],[B, A]] with s = -1 / +1;
//   * D = P - V is stored instead of P, so V never enters the time loop: g = P b^H = D c + h,
//     var = c.g + yerr^2, and the predict step is D <- Phi D Phi^T (no subtract/add of V);
//   * g is computed once per step and reused for the gain, the state update and the variance;
//   * the observation row c is (1,0,1,0,...[,1]) for every kind of slot, so g, var and mean are plain sums.
// The time loop is dispatch bound on sm_100a (fast_math.cuh): it is written to minimise the number of
// instructions of ANY kind -- one basic block per step, loop constants from the constant bank, shared-memory
// operands addressed off one register, the sum of log(var) kept as a mantissa product plus an integer exponent
// sum without any per-step range branch (a sticky flag sends the rare out-of-range case to an exact slow path).
#pragma once
#include "fast_math.cuh"
#include "theta_transform.cuh"

namespace carma {

template <int P>
struct KalmanReal {
    static constexpr int NS = P / 2;         // 2x2 slots
    static constexpr bool ODD = (P & 1) != 0;
    static constexpr int NT = P * (P + 1) / 2;

    double D[NT];  // upper triangle of the symmetric D = P - V
    double z[P];
    double g[P];   // P b^H in the real basis (before division by var)
    double var, mean;

    static __host__ __device__ constexpr int idx(int i, int j) { return i * P - (i * (i - 1)) / 2 + (j - i); }

    CARMA_HD void reset(const RealParams<P>& prm, double e2_0) {
#pragma unroll
        for (int i = 0; i < NT; i++) D[i] = 0.0;
#pragma unroll
        for (int i = 0; i < P; i++) { z[i] = 0.0; g[i] = prm.h[i]; }
        mean = 0.0;
        var = prm.v0 + prm.scale * e2_0;
    }

    // One Update(): condition on the residual `innov` (= y_i - mu - mean_i) observed with predictive
    // variance `var`, move forward by dt, and form mean/var for the next point (measurement variance e2n).
    // ALLC = true: every 2x2 slot is a conjugate pair (compile time; the per-lane selections vanish);
    // ALLC = false: conjugate and real pairs mixed per lane -- same instruction sequence, operands selected.
    template <bool ALLC, class Tab>
    CARMA_HD void advance(const RealParams<P>& prm, const Tab& tb, double innov, double inv_var, double dt, double e2n) {
        measurement_update(innov, inv_var);
        predict_observe<ALLC>(prm, tb, dt, e2n);
    }

    // z += g innov/var ;  D -= g g^T / var   (kfilter.cpp:191-197)
    CARMA_HD void measurement_update(double innov, double inv_var) {
        const double w = innov * inv_var;
        double gi[P];
#pragma unroll
        for (int i = 0; i < P; i++) {
            z[i] = fma(g[i], w, z[i]);
            gi[i] = g[i] * inv_var;
        }
#pragma unroll
        for (int i = 0; i < P; i++)
#pragma unroll
            for (int j = i; j < P; j++) D[idx(i, j)] = fma(-gi[i], g[j], D[idx(i, j)]);
    }

    // the transition blocks [[A, sB],[B, A]] of all slots and the factor of the odd root
    template <bool ALLC, class Tab>
    static CARMA_HD void transition(const RealParams<P>& prm, const Tab& tb, double dt, double* fa, double* fb,
                                    double* fsb, double* fo) {
#pragma unroll
        for (int s = 0; s < NS; s++) {
            const bool is_c = ALLC || ((prm.cmask >> s) & 1u);
            const double e = exp_scaled(prm.le[s], dt, tb);
            double s2, c2;
            rot_scaled<ALLC>(prm.ls[s], dt, is_c, tb, &s2, &c2);
            fa[s] = e * c2;
            fb[s] = e * s2;
            if (ALLC) fsb[s] = -fb[s];
            else fsb[s] = is_c ? -fb[s] : fb[s];
        }
        *fo = 1.0;
        if (ODD) *fo = exp_scaled(prm.le[NS], dt, tb);
    }

    // transition by dt and predicted observation of the next point (kfilter.cpp:200-210)
    template <bool ALLC, class Tab>
    CARMA_HD void predict_observe(const RealParams<P>& prm, const Tab& tb, double dt, double e2n) {
        double fa[NS > 0 ? NS : 1], fb[NS > 0 ? NS : 1], fsb[NS > 0 ? NS : 1], fo;
        transition<ALLC>(prm, tb, dt, fa, fb, fsb, &fo);
        propagate(prm, fa, fb, fsb, fo, e2n);
    }

    // v <- Phi v for an extra state-like vector (Predict's linear coefficients, kfilter.cpp:290-337)
    static CARMA_HD void propagate_vec(const double* fa, const double* fb, const double* fsb, double fo, double* v) {
#pragma unroll
        for (int s = 0; s < NS; s++) {
            const double u = v[2 * s], w = v[2 * s + 1];
            v[2 * s] = fma(fa[s], u, fsb[s] * w);
            v[2 * s + 1] = fma(fb[s], u, fa[s] * w);
        }
        if (ODD) v[P - 1] *= fo;
    }
    // c . v with the observation row c = (1,0,1,0,...[,1])
    static CARMA_HD double observe_vec(const double* v) {
        double m = v[0];
#pragma unroll
        for (int i = 2; i < P; i++)
            if ((i & 1) == 0) m += v[i];
        return m;
    }
    // g = D c + h, var = c.g + scale e2, mean = c.z for the CURRENT (z, D): what predict_observe ends with
    CARMA_HD void observe(const RealParams<P>& prm, double e2) {
#pragma unroll
        for (int i = 0; i < P; i++) {
            double acc = prm.h[i];
#pragma unroll
            for (int j = 0; j < P; j++)
                if ((j & 1) == 0) acc += D[(i <= j) ? idx(i, j) : idx(j, i)];
            g[i] = acc;
        }
        var = fma(prm.scale, e2, observe_vec(g));
        mean = observe_vec(z);
    }

    // state / covariance prediction with given transition blocks, then the predicted observation
    CARMA_HD void propagate(const RealParams<P>& prm, const double* fa, const double* fb, const double* fsb, double fo,
                            double e2n) {

        // ---- predict state
#pragma unroll
        for (int s = 0; s < NS; s++) {
            const double u = z[2 * s], v = z[2 * s + 1];
            z[2 * s] = fma(fa[s], u, fsb[s] * v);
            z[2 * s + 1] = fma(fb[s], u, fa[s] * v);
        }
        if (ODD) z[P - 1] *= fo;

        // ---- predict covariance: D <- Phi D Phi^T, block by block
#pragma unroll
        for (int a = 0; a < NS; a++) {
            const int i = 2 * a;
            const double A = fa[a], B = fb[a], SB = fsb[a];
            {   // diagonal block (symmetric 2x2)
                const double d00 = D[idx(i, i)], d01 = D[idx(i, i + 1)], d11 = D[idx(i + 1, i + 1)];
                const double m00 = fma(A, d00, SB * d01), m01 = fma(A, d01, SB * d11);
                const double m10 = fma(B, d00, A * d01), m11 = fma(B, d01, A * d11);
                D[idx(i, i)] = fma(m00, A, m01 * SB);
                D[idx(i, i + 1)] = fma(m00, B, m01 * A);
                D[idx(i + 1, i + 1)] = fma(m10, B, m11 * A);
            }
#pragma unroll
            for (int b = a + 1; b < NS; b++) {  // off-diagonal 2x2 block
                const int j = 2 * b;
                const double A2 = fa[b], B2 = fb[b], SB2 = fsb[b];
                const double d00 = D[idx(i, j)], d01 = D[idx(i, j + 1)], d10 = D[idx(i + 1, j)], d11 = D[idx(i + 1, j + 1)];
                const double m00 = fma(A, d00, SB * d10), m01 = fma(A, d01, SB * d11);
                const double m10 = fma(B, d00, A * d10), m11 = fma(B, d01, A * d11);
                D[idx(i, j)] = fma(m00, A2, m01 * SB2);
                D[idx(i, j + 1)] = fma(m00, B2, m01 * A2);
                D[idx(i + 1, j)] = fma(m10, A2, m11 * SB2);
                D[idx(i + 1, j + 1)] = fma(m10, B2, m11 * A2);
            }
            if (ODD) {  // 2x1 block against the odd real root
                const double d0 = D[idx(i, P - 1)] * fo, d1 = D[idx(i + 1, P - 1)] * fo;
                D[idx(i, P - 1)] = fma(A, d0, SB * d1);
                D[idx(i + 1, P - 1)] = fma(B, d0, A * d1);
            }
        }
        if (ODD) D[idx(P - 1, P - 1)] *= fo * fo;

        // ---- predicted observation: g = D c + h, var = c.g + e2, mean = c.z with c = (1,0,1,0,...[,1])
        double m = z[0];
#pragma unroll
        for (int i = 0; i < P; i++) {
            double acc = prm.h[i];
#pragma unroll
            for (int j = 0; j < P; j++)
                if ((j & 1) == 0) acc += D[(i <= j) ? idx(i, j) : idx(j, i)];
            g[i] = acc;
        }
        double vv = fma(prm.scale, e2n, g[0]);  // var = scale e2 + g_0 + g_2 + ...
#pragma unroll
        for (int i = 2; i < P; i++)
            if ((i & 1) == 0) vv += g[i];
#pragma unroll
        for (int i = 2; i < P; i++)
            if ((i & 1) == 0) m += z[i];
        var = vv;
        mean = m;
    }

    // ---- the smoother's adjoint recursion (multi_smooth_kernel, survey.cu): lambda (P) and the symmetric Lambda (upper
    // triangle, D's layout) run backwards through the transposed transitions.
    // v <- Phi^T v: the blocks of Phi^T are [[A, B],[sB, A]], Phi's with B and sB swapped
    static CARMA_HD void propagate_vec_t(const double* fa, const double* fb, const double* fsb, double fo, double* v) {
        propagate_vec(fa, fsb, fb, fo, v);
    }
    // M <- Phi^T M Phi for a symmetric M: the covariance part of propagate with B and sB swapped
    static CARMA_HD void congruence_t(double* M, const double* fa, const double* fb, const double* fsb, double fo) {
#pragma unroll
        for (int a = 0; a < NS; a++) {
            const int i = 2 * a;
            const double A = fa[a], B = fsb[a], SB = fb[a];
            {
                const double d00 = M[idx(i, i)], d01 = M[idx(i, i + 1)], d11 = M[idx(i + 1, i + 1)];
                const double m00 = fma(A, d00, SB * d01), m01 = fma(A, d01, SB * d11);
                const double m10 = fma(B, d00, A * d01), m11 = fma(B, d01, A * d11);
                M[idx(i, i)] = fma(m00, A, m01 * SB);
                M[idx(i, i + 1)] = fma(m00, B, m01 * A);
                M[idx(i + 1, i + 1)] = fma(m10, B, m11 * A);
            }
#pragma unroll
            for (int b = a + 1; b < NS; b++) {
                const int j = 2 * b;
                const double A2 = fa[b], B2 = fsb[b], SB2 = fb[b];
                const double d00 = M[idx(i, j)], d01 = M[idx(i, j + 1)], d10 = M[idx(i + 1, j)], d11 = M[idx(i + 1, j + 1)];
                const double m00 = fma(A, d00, SB * d10), m01 = fma(A, d01, SB * d11);
                const double m10 = fma(B, d00, A * d10), m11 = fma(B, d01, A * d11);
                M[idx(i, j)] = fma(m00, A2, m01 * SB2);
                M[idx(i, j + 1)] = fma(m00, B2, m01 * A2);
                M[idx(i + 1, j)] = fma(m10, A2, m11 * SB2);
                M[idx(i + 1, j + 1)] = fma(m10, B2, m11 * A2);
            }
            if (ODD) {
                const double d0 = M[idx(i, P - 1)] * fo, d1 = M[idx(i + 1, P - 1)] * fo;
                M[idx(i, P - 1)] = fma(A, d0, SB * d1);
                M[idx(i + 1, P - 1)] = fma(B, d0, A * d1);
            }
        }
        if (ODD) M[idx(P - 1, P - 1)] *= fo * fo;
    }
    // out = M v for a symmetric M
    static CARMA_HD void sym_mul(const double* M, const double* v, double* out) {
#pragma unroll
        for (int i = 0; i < P; i++) {
            double acc = 0.0;
#pragma unroll
            for (int j = 0; j < P; j++) acc = fma(M[(i <= j) ? idx(i, j) : idx(j, i)], v[j], acc);
            out[i] = acc;
        }
    }
    static CARMA_HD double dot(const double* a, const double* b) {
        double s = 0.0;
#pragma unroll
        for (int i = 0; i < P; i++) s = fma(a[i], b[i], s);
        return s;
    }
    // Lambda <- c c^T / S + (I - K c)^T Lambda (I - K c) = Lambda - c u^T - u c^T + dk c c^T, given u = Lambda K and
    // dk = 1/S + K^T u: a symmetric update of rank two along the fixed observation row, O(P^2)
    static CARMA_HD void info_update(double* M, const double* u, double dk) {
#pragma unroll
        for (int i = 0; i < P; i++)
#pragma unroll
            for (int j = i; j < P; j++) {
                double v = M[idx(i, j)];
                if ((i & 1) == 0) v -= u[j];
                if ((j & 1) == 0) v -= u[i];
                if ((i & 1) == 0 && (j & 1) == 0) v += dk;
                M[idx(i, j)] = v;
            }
    }
};

// Running sum of -1/2 log(var_i) - 1/2 innov_i^2 / var_i with the logs folded into one log of a product of
// mantissas (exponent fields summed as integers): log() leaves the time loop, and so does every branch -- a var
// that is not a positive normal number only sets a sticky flag; the caller then recomputes that evaluation with
// loglik_exact_slow (same recursion, one log() per point), which gives NaN / -inf in the same class as the reference.
struct LogLikAcc {
    double quad;    // sum innov^2 / var
    double prod;    // product of mantissas of var (renormalise at least every 1000 points)
    int esum;       // sum of biased exponent fields
    int npts;
    unsigned hmin, hmax;  // range of the high words of var seen so far (as unsigned: a set sign bit is "huge")
    CARMA_HD void init() { quad = 0.0; prod = 1.0; esum = 0; npts = 0; hmin = 0x3ff00000u; hmax = 0x3ff00000u; }
    // some var was zero, negative, subnormal, infinite or NaN: exponent field 0 or 2047, or sign set
    CARMA_HD bool bad() const { return hmin < 0x00100000u || hmax >= 0x7ff00000u; }
    CARMA_HD void add(double var, double innov, double inv_var) {
        quad = fma(innov, innov * inv_var, quad);  // innov * inv_var is also the gain factor of the measurement update
        const int hi = hi32(var);
        prod *= mk64((hi & 0x000fffff) | 0x3ff00000, lo32(var));
        esum += (int)((unsigned)hi >> 20);
        hmin = min((unsigned)hi, hmin);
        hmax = max((unsigned)hi, hmax);
    }
    // call at least once every 1000 add()s: prod < 2^1000
    CARMA_HD void renorm(int added) {
        npts += added;
        const int hi = hi32(prod);
        esum += (int)(((unsigned)hi >> 20) & 0x7ffu) - 1023;
        prod = mk64((hi & 0x800fffff) | 0x3ff00000, lo32(prod));
    }
    CARMA_HD double value() const {
        return -0.5 * (log(prod) + (double)(esum - 1023 * npts) * 0.693147180559945309417232121458) - 0.5 * quad;
    }
};

// ---- where the time loop reads the light curve from
#ifdef __CUDACC__
// shared memory: dt[i] at a + 8 i, y[i] at a + yoff + 8 i, next-point yerr^2 at a + eoff + 8 i (device only)
struct SeriesSmem {
    uint32_t a, yoff, eoff;
    __device__ __forceinline__ void get(int i, double* dt, double* y, double* e) const {
#ifdef __CUDA_ARCH__
        const uint32_t p = a + 8u * (uint32_t)i;
        asm("ld.shared.f64 %0, [%1];" : "=d"(*dt) : "r"(p));
        asm("ld.shared.f64 %0, [%1];" : "=d"(*y) : "r"(p + yoff));
        asm("ld.shared.f64 %0, [%1];" : "=d"(*e) : "r"(p + eoff));
#endif
    }
    __device__ __forceinline__ double get_y(int i) const {
        double y = 0.0;
#ifdef __CUDA_ARCH__
        asm("ld.shared.f64 %0, [%1];" : "=d"(y) : "r"(a + yoff + 8u * (uint32_t)i));
#endif
        return y;
    }
};
#endif
// global (or host) memory
struct SeriesPtr {
    const double* dt;
    const double* y;
    const double* e;
    CARMA_HD void get(int i, double* dt_, double* y_, double* e_) const { *dt_ = dt[i]; *y_ = y[i]; *e_ = e[i]; }
    CARMA_HD double get_y(int i) const { return y[i]; }
};

constexpr int RENORM_EVERY = 512;

// Run the recursion over `len` points (dt, y, next-point yerr^2); the last `len - nadv` (0 or 1) points are
// only scored, not advanced past (end of the light curve).
// PF = true: the three operands of step i+1 are loaded while step i is computed (software prefetch);
// used when the series is read straight from global memory (K4, K5), pointless for shared memory.
template <int P, bool ALLC, bool PF, class Src, class Tab>
CARMA_HD void filter_span_impl(KalmanReal<P>& kf, LogLikAcc& acc, const RealParams<P>& prm, const Tab& tb,
                               const Src& src, int len, int nadv) {
    double y_c = 0.0, dt_c = 0.0, e_c = 0.0;
    if (PF && nadv > 0) src.get(0, &dt_c, &y_c, &e_c);
    else if (PF && len > 0) y_c = src.get_y(0);
    for (int i0 = 0; i0 < nadv; i0 += RENORM_EVERY) {
        const int i1 = (nadv - i0 < RENORM_EVERY) ? nadv : i0 + RENORM_EVERY;
        for (int i = i0; i < i1; i++) {
            double y_i, dt_i, e_i;
            if (PF) {
                y_i = y_c; dt_i = dt_c; e_i = e_c;
                const int j = i + 1;  // j <= nadv <= len - 1 whenever the last point is only scored
                if (j < nadv) src.get(j, &dt_c, &y_c, &e_c);
                else if (j < len) y_c = src.get_y(j);
            } else {
                src.get(i, &dt_i, &y_i, &e_i);
            }
            const double innov = (y_i - prm.mu) - kf.mean;
            const double inv = rcp_fast(kf.var);
            acc.add(kf.var, innov, inv);
            kf.template advance<ALLC>(prm, tb, innov, inv, dt_i, e_i);
        }
        acc.renorm(i1 - i0);
    }
    if (nadv < len) {
        const double y_l = PF ? y_c : src.get_y(len - 1);
        const double innov = (y_l - prm.mu) - kf.mean;
        const double inv = rcp_fast(kf.var);
        acc.add(kf.var, innov, inv);
        acc.renorm(1);
    }
}

// Software-pipelined form for launches with ONE OR TWO warps per SM (a single PT ensemble: the reference's own use,
// BASELINE config 1), where nothing hides latency: the transition blocks of step i + 1 -- table lookups and ~70 FP64
// instructions that depend only on dt, not on the filter state -- are computed in the same basic block as the state
// update of step i, so their latency no longer sits on the recursion's critical path (rcp -> gain -> D update ->
// predict -> observe).  Same operations, same results, bit for bit.  Costs ~10 registers.  Measured: no gain once the
// SM holds >= 8 warps (config 3: 4.09 vs 4.11e6 ensemble-iterations/s), so pt_kernel selects it only for small grids.
// Requires src.get(nadv) to be readable (the staged series is padded: dt[ny-1] = 0).
template <int P, bool ALLC, class Src, class Tab>
CARMA_HD void filter_span_pipelined(KalmanReal<P>& kf, LogLikAcc& acc, const RealParams<P>& prm, const Tab& tb,
                                    const Src& src, int len, int nadv) {
    constexpr int NS = KalmanReal<P>::NS;
    double fa[NS > 0 ? NS : 1], fb[NS > 0 ? NS : 1], fsb[NS > 0 ? NS : 1], fo = 1.0;
    double y_c = 0.0, dt_c = 0.0, e_c = 0.0;
    if (len > 0) src.get(0, &dt_c, &y_c, &e_c);
    if (nadv > 0) KalmanReal<P>::template transition<ALLC>(prm, tb, dt_c, fa, fb, fsb, &fo);
    for (int i0 = 0; i0 < nadv; i0 += RENORM_EVERY) {
        const int i1 = (nadv - i0 < RENORM_EVERY) ? nadv : i0 + RENORM_EVERY;
        for (int i = i0; i < i1; i++) {
            double na[NS > 0 ? NS : 1], nb[NS > 0 ? NS : 1], nsb[NS > 0 ? NS : 1], no;
            double y_n, dt_n, e_n;
            src.get(i + 1, &dt_n, &y_n, &e_n);
            KalmanReal<P>::template transition<ALLC>(prm, tb, dt_n, na, nb, nsb, &no);
            const double innov = (y_c - prm.mu) - kf.mean;
            const double inv = rcp_fast(kf.var);
            acc.add(kf.var, innov, inv);
            kf.measurement_update(innov, inv);
            kf.propagate(prm, fa, fb, fsb, fo, e_c);
#pragma unroll
            for (int s = 0; s < NS; s++) { fa[s] = na[s]; fb[s] = nb[s]; fsb[s] = nsb[s]; }
            fo = no;
            y_c = y_n; e_c = e_n;
        }
        acc.renorm(i1 - i0);
    }
    if (nadv < len) {
        const double innov = (y_c - prm.mu) - kf.mean;
        const double inv = rcp_fast(kf.var);
        acc.add(kf.var, innov, inv);
        acc.renorm(1);
    }
}

template <int P, bool PF, class Src, class Tab>
CARMA_HD void filter_span_any(KalmanReal<P>& kf, LogLikAcc& acc, const RealParams<P>& prm, const Tab& tb,
                              const Src& src, int len, int nadv) {
    constexpr unsigned ALL = (P / 2 > 0) ? ((1u << (P / 2)) - 1u) : 0u;
#ifdef __CUDA_ARCH__
    // Warp-uniform choice: the all-conjugate-pairs loop (no per-lane selections) only when EVERY active lane of
    // the warp qualifies; otherwise all lanes run the generic loop.  Both round identically on a conjugate pair,
    // so a result never depends on which lanes share a warp.
    const bool all_c = __all_sync(__activemask(), prm.cmask == ALL);
#else
    const bool all_c = prm.cmask == ALL;
#endif
    if (all_c) filter_span_impl<P, true, PF>(kf, acc, prm, tb, src, len, nadv);
    else filter_span_impl<P, false, PF>(kf, acc, prm, tb, src, len, nadv);
}

template <int P, class Src, class Tab>
CARMA_HD void filter_span_any_pipelined(KalmanReal<P>& kf, LogLikAcc& acc, const RealParams<P>& prm, const Tab& tb,
                                        const Src& src, int len, int nadv) {
    constexpr unsigned ALL = (P / 2 > 0) ? ((1u << (P / 2)) - 1u) : 0u;
#ifdef __CUDA_ARCH__
    const bool all_c = __all_sync(__activemask(), prm.cmask == ALL);
#else
    const bool all_c = prm.cmask == ALL;
#endif
    if (all_c) filter_span_pipelined<P, true>(kf, acc, prm, tb, src, len, nadv);
    else filter_span_pipelined<P, false>(kf, acc, prm, tb, src, len, nadv);
}

// K4's loop: every thread streams ITS OWN light curve from global memory.  With one 8-byte load per array and step the
// 32 lanes of a warp touch 32 different sectors per load, four times per sector, and the loads of a step are issued one
// step ahead only: ncu showed the warps waiting on them (long-scoreboard 5.0 stalls per issue, FP64 pipe 53 %).  Here a
// thread fetches FOUR steps of an array with one 256-bit access (a whole sector: a quarter of the L1 wavefronts) and
// the block after the current one is in flight while the current one is computed (prefetch distance 4 to 7 steps).
// dt, y: the curve's arrays; E: its yerr^2 array UNSHIFTED (step i uses E[i + 1], the next point's variance).
// A misaligned curve start is peeled with up to three scalar steps.  Same operations in the same order as
// filter_span_impl: bitwise equal results.
#ifdef __CUDACC__
struct Dbl4 { double a, b, c, d; };
__device__ __forceinline__ Dbl4 ldg4(const double* q) {   // q 32-byte aligned
    Dbl4 v;
#ifdef __CUDA_ARCH__
    // one 256-bit access per sector (sm_100); the curve is read exactly once, so it does not need a line in L1
    asm volatile("ld.global.nc.L1::no_allocate.v4.f64 {%0, %1, %2, %3}, [%4];" : "=d"(v.a), "=d"(v.b), "=d"(v.c), "=d"(v.d) : "l"(q));
#else
    v.a = q[0]; v.b = q[1]; v.c = q[2]; v.d = q[3];
#endif
    return v;
}
template <int P, bool ALLC, class Tab>
__device__ void filter_span_blocks(KalmanReal<P>& kf, LogLikAcc& acc, const RealParams<P>& prm, const Tab& tb,
                                   const double* __restrict__ dt, const double* __restrict__ y,
                                   const double* __restrict__ E, int len) {
    const int nadv = len - 1;
    int since = 0;
    auto step = [&](double dt_i, double y_i, double e_i) {
        const double innov = (y_i - prm.mu) - kf.mean;
        const double inv = rcp_fast(kf.var);
        acc.add(kf.var, innov, inv);
        kf.template advance<ALLC>(prm, tb, innov, inv, dt_i, e_i);
    };
    int i = 0;
    const int head = min(nadv, (int)((4u - (unsigned)(((size_t)dt >> 3) & 3u)) & 3u));
    for (; i < head; i++) step(dt[i], y[i], E[i + 1]);
    since = head;
    if (i + 4 <= nadv) {
        Dbl4 cdt = ldg4(dt + i), cy = ldg4(y + i), cE = ldg4(E + i);
        for (;;) {
            const bool nx = i + 8 <= len;   // the next block lies inside this curve
            Dbl4 ndt = cdt, ny_ = cy, nE = cE;
            double e_last;
            if (nx) {
                ndt = ldg4(dt + i + 4); ny_ = ldg4(y + i + 4); nE = ldg4(E + i + 4);
                e_last = nE.a;
            } else {
                e_last = E[i + 4];          // i + 4 <= nadv = len - 1
            }
            step(cdt.a, cy.a, cE.b);
            step(cdt.b, cy.b, cE.c);
            step(cdt.c, cy.c, cE.d);
            step(cdt.d, cy.d, e_last);
            i += 4;
            since += 4;
            if (since >= RENORM_EVERY - 8) { acc.renorm(since); since = 0; }
            if (!nx || i + 4 > nadv) break;
            cdt = ndt; cy = ny_; cE = nE;
        }
    }
    for (; i < nadv; i++, since++) step(dt[i], y[i], E[i + 1]);
    if (since) acc.renorm(since);
    {   // the last point is only scored
        const double innov = (y[len - 1] - prm.mu) - kf.mean;
        const double inv = rcp_fast(kf.var);
        acc.add(kf.var, innov, inv);
        acc.renorm(1);
    }
}
template <int P, class Tab>
__device__ void filter_span_blocks_any(KalmanReal<P>& kf, LogLikAcc& acc, const RealParams<P>& prm, const Tab& tb,
                                       const double* dt, const double* y, const double* E, int len) {
    constexpr unsigned ALL = (P / 2 > 0) ? ((1u << (P / 2)) - 1u) : 0u;
    const bool all_c = __all_sync(__activemask(), prm.cmask == ALL);
    if (all_c) filter_span_blocks<P, true>(kf, acc, prm, tb, dt, y, E, len);
    else filter_span_blocks<P, false>(kf, acc, prm, tb, dt, y, E, len);
}
#endif

// KalmanFilterp::Predict (kfilter.cpp:218-337) of one query time t*, resumed from the forward filter's state.
// ip: number of data times strictly before t*; st_z / st_D: the state (z, D) predicted at point ip - 1 (not read when
// ip == 0); gap_before = t* - t[ip-1], gap_after = t[ip] - t* (each only read where it exists).  The curve is read
// through y(i), dt(i) (gap from point i to i + 1) and e2(i) (yerr^2 of point i).  The linear-coefficient pass runs over
// the ny - ip points behind the query.  Outputs: predictive mean (without mu) and variance.
template <int P, class Tab, class Y, class DT, class E2>
__device__ __forceinline__ void predict_resume(const RealParams<P>& prm, const Tab& tb, const double* st_z,
                                               const double* st_D, int ip, int ny, double gap_before, double gap_after,
                                               Y y, DT dt, E2 e2, double* qmean, double* qvar) {
    constexpr int NS = P / 2, NT = P * (P + 1) / 2;
    KalmanReal<P> kf;
    double fa[NS > 0 ? NS : 1], fb[NS > 0 ? NS : 1], fsb[NS > 0 ? NS : 1], fo;
    double pmean, pvar;
    if (ip == 0) {
        kf.reset(prm, 0.0);       // stationary law: mean 0, variance Re(b V b^H), g = V b^H
        pmean = 0.0;
        pvar = prm.v0;
    } else {
#pragma unroll
        for (int i = 0; i < P; i++) kf.z[i] = st_z[i];
#pragma unroll
        for (int i = 0; i < NT; i++) kf.D[i] = st_D[i];
        kf.observe(prm, e2(ip - 1));
        const double innov = (y(ip - 1) - prm.mu) - kf.mean;
        kf.template advance<false>(prm, tb, innov, 1.0 / kf.var, gap_before, 0.0);  // no noise at t*
        pmean = kf.mean;
        pvar = kf.var;
    }
    if (ip == ny) { *qmean = pmean; *qvar = pvar; return; }   // forecast: nothing behind the query
    // InitializeCoefs (kfilter.cpp:290-312): y* enters as a noiseless pseudo-observation with the predictive law
    double prec = 1.0 / pvar, pm = pmean * prec;
    double zs[P];
    {
        const double inv = 1.0 / pvar;
#pragma unroll
        for (int i = 0; i < P; i++) zs[i] = kf.g[i] * inv;            // state_slope = K
        kf.measurement_update(-pmean, inv);                           // state_const = x - K ymean ; P -= yvar K K^H
        KalmanReal<P>::template transition<false>(prm, tb, gap_after, fa, fb, fsb, &fo);
        KalmanReal<P>::propagate_vec(fa, fb, fsb, fo, zs);
        kf.propagate(prm, fa, fb, fsb, fo, e2(ip));                   // kf.mean = yconst, kf.var = var[ip]
    }
    double yslope = KalmanReal<P>::observe_vec(zs);
    prec += yslope * yslope / kf.var;
    pm += yslope * ((y(ip) - prm.mu) - kf.mean) / kf.var;
    for (int i = ip + 1; i < ny; i++) {                               // UpdateCoefs (kfilter.cpp:316-337)
        const double inv = 1.0 / kf.var;
        const double sl = yslope * inv;
#pragma unroll
        for (int j = 0; j < P; j++) zs[j] = fma(-kf.g[j], sl, zs[j]);  // state_slope -= K yslope
        kf.measurement_update((y(i - 1) - prm.mu) - kf.mean, inv);     // state_const += K (y - yconst) ; P -= var K K^H
        KalmanReal<P>::template transition<false>(prm, tb, dt(i - 1), fa, fb, fsb, &fo);
        KalmanReal<P>::propagate_vec(fa, fb, fsb, fo, zs);
        kf.propagate(prm, fa, fb, fsb, fo, e2(i));
        yslope = KalmanReal<P>::observe_vec(zs);
        prec += yslope * yslope / kf.var;
        pm += yslope * ((y(i) - prm.mu) - kf.mean) / kf.var;
    }
    pvar = 1.0 / prec;
    *qmean = pm * pvar;
    *qvar = pvar;
}

// Conditional simulation, prior part (carma_simulate's sim_prior_kernel, the survey's condsim_prior_kernel): an
// unconditional path of the noise-free process on the merged grid of data and requested times, drawn point by point
// from the innovations form of the filter (kf built with prm.scale = 0).  Merged point k of path `path` uses the Philox
// counters (seed, path, STREAM_CONDSIM, k, block).
enum { STREAM_CONDSIM = 5 };

// Draw f at the current merged point: returns f = mean + innov; rr * sn is a second, independent normal (the
// measurement noise of a data point).
template <int P>
__device__ __forceinline__ double condsim_draw(const KalmanReal<P>& kf, unsigned long long seed, uint32_t path, uint32_t k,
                                               uint32_t block, double* innov, double* rr, double* sn) {
    double u0, u1;
    uniforms2(seed, path, STREAM_CONDSIM, k, block, &u0, &u1);
    *rr = sqrt(-2.0 * log(u0));
    double cs;
    sincos(6.283185307179586476925286766559 * u1, sn, &cs);
    const double var = fmax(kf.var, 0.0);
    *innov = sqrt(var) * *rr * cs;
    return kf.mean + *innov;
}

// Condition on the drawn value and move to the next merged point, dt ahead.
template <int P, class Tab>
__device__ __forceinline__ void condsim_next(KalmanReal<P>& kf, const RealParams<P>& prm, const Tab& tb, double innov,
                                             double dt) {
    // a point that coincides with the previous one (var = 0) carries no new information
    const double inv = kf.var > 1e-300 ? 1.0 / kf.var : 0.0;
    kf.measurement_update(innov, inv);
    kf.template predict_observe<false>(prm, tb, dt, 0.0);
}

// Exact (slow) evaluation of the log-likelihood of one theta: the same recursion with one log() per point.
// Only reached when LogLikAcc::bad was raised (var not a positive normal number somewhere).
template <int P, class Src, class Tab>
__host__ __device__ __noinline__ double loglik_exact_slow(const RealParams<P>& prm, const Tab& tb, const Src& src,
                                                          int ny, double e2_0) {
    KalmanReal<P> kf;
    kf.reset(prm, e2_0);
    double ll = 0.0;
    for (int i = 0; i < ny; i++) {
        double dt_i = 0.0, y_i, e_i = 0.0;
        if (i + 1 < ny) src.get(i, &dt_i, &y_i, &e_i);
        else y_i = src.get_y(i);
        const double innov = (y_i - prm.mu) - kf.mean;
        ll += -0.5 * log(kf.var) - 0.5 * innov * innov / kf.var;
        if (ll != ll) return ll;   // NaN stays NaN whatever follows (a negative or NaN variance): no need to finish the series
        if (i + 1 < ny) kf.template advance<false>(prm, tb, innov, 1.0 / kf.var, dt_i, e_i);
    }
    return ll;
}

// ---- Kalman smoother of one curve (Bryson-Frazier adjoint form; the survey's multi_smooth_kernel, DESIGN.md K-smooth).
// Records, field-major: field f of point i at rp[f * ps + i] -- g[P] = P^- c, the predictive mean (without mu), the
// predictive variance S -- and field f of the curve's sorted query k at rq[f * qs + k - k0] -- w[P] = Phi(t[ip] - t*) g*,
// mean^-(t*), v^-(t*), ip (number of data times strictly before t*, as a double).  Queries are on the curve's own axis
// (running sum of dt from 0), sorted; qmean / qvar are written at perm[k].
//
// Forward: K4's steps in K4's order (the log-density is bitwise K4's: renormalising LogLikAcc at other points only
// rescales its mantissa product by powers of two), the point records, and for each query the state filtered at point
// ip - 1 moved to t* without noise (predict_resume's first half); forecasts (ip = ny) are final here.
template <int P, bool ALLC, class Tab>
CARMA_HD void smooth_forward(KalmanReal<P>& kf, LogLikAcc& acc, const RealParams<P>& prm, const Tab& tb, const double* dt,
                             const double* y, const double* E, int ny, double* rp, size_t ps, long long k, long long k1,
                             const double* qtq, double* rq, size_t qs, const long long* perm, double* qmean, double* qvar) {
    constexpr int NS = P / 2;
    double fa[NS > 0 ? NS : 1], fb[NS > 0 ? NS : 1], fsb[NS > 0 ? NS : 1], fo;
    double t = 0.0;
    for (; k < k1 && !(qtq[k] > t); k++) {   // at or before the first point (ip = 0): the stationary law, g* = h
        double w[P];
#pragma unroll
        for (int j = 0; j < P; j++) w[j] = prm.h[j];
        KalmanReal<P>::template transition<false>(prm, tb, t - qtq[k], fa, fb, fsb, &fo);
        KalmanReal<P>::propagate_vec(fa, fb, fsb, fo, w);
#pragma unroll
        for (int j = 0; j < P; j++) rq[j * qs] = w[j];
        rq[P * qs] = 0.0;
        rq[(P + 1) * qs] = prm.v0;
        rq[(P + 2) * qs] = 0.0;
        rq++;
    }
    int since = 0;
    for (int i = 0; i < ny; i++) {
        const bool last = i + 1 == ny;
        const double dt_i = last ? 0.0 : dt[i];
        const double tn = t + dt_i;
        const double innov = (y[i] - prm.mu) - kf.mean;
        const double inv = rcp_fast(kf.var);
        acc.add(kf.var, innov, inv);
#pragma unroll
        for (int j = 0; j < P; j++) rp[j * ps + i] = kf.g[j];
        rp[P * ps + i] = kf.mean;
        rp[(P + 1) * ps + i] = kf.var;
        for (; k < k1 && (last || !(qtq[k] > tn)); k++) {   // t[i] < t* <= t[i+1], or past the last point: ip = i + 1
            KalmanReal<P> kq = kf;
            kq.template advance<false>(prm, tb, innov, 1.0 / kf.var, qtq[k] - t, 0.0);   // no noise at t*
            if (last) {
                qmean[perm[k]] = kq.mean;
                qvar[perm[k]] = kq.var;
            } else {
                KalmanReal<P>::template transition<false>(prm, tb, tn - qtq[k], fa, fb, fsb, &fo);
                KalmanReal<P>::propagate_vec(fa, fb, fsb, fo, kq.g);
#pragma unroll
                for (int j = 0; j < P; j++) rq[j * qs] = kq.g[j];
                rq[P * qs] = kq.mean;
                rq[(P + 1) * qs] = kq.var;
            }
            rq[(P + 2) * qs] = (double)(i + 1);
            rq++;
        }
        if (last) break;
        kf.template advance<ALLC>(prm, tb, innov, inv, dt_i, E[i + 1]);
        if (++since == RENORM_EVERY) { acc.renorm(since); since = 0; }
        t = tn;
    }
    acc.renorm(since + 1);
}

// Backward, from the last point with lambda = Lambda = 0 (K_i = g_i / S_i):
//   lambda^_i = Phi_i^T lambda_{i+1},  Lambda^_i = Phi_i^T Lambda_{i+1} Phi_i
//   u_i = e_i / S_i - K_i^T lambda^_i,  d_i = 1 / S_i + K_i^T Lambda^_i K_i
//   loo: y_i - mu given the rest has mean (y_i - mu) - u_i / d_i and variance 1 / d_i
//   lambda_i = c u_i + lambda^_i,  Lambda_i = c c^T / S_i + (I - K_i c)^T Lambda^_i (I - K_i c)
//   smoothed f(t_i): mean_i + g_i^T lambda_i, c.g_i - g_i^T Lambda_i g_i;  query with ip = i: mean^- + w^T lambda_i,
//   v^- - w^T Lambda_i w.  Outputs (the curve's own slices) without mu.
template <int P, class Tab>
CARMA_HD void smooth_backward(const RealParams<P>& prm, const Tab& tb, const double* dt, const double* y, int ny,
                              const double* rp, size_t ps, long long k0, long long k1, const double* rq, size_t qs,
                              const long long* perm, double* mean, double* var, double* loo_mean, double* loo_var,
                              double* qmean, double* qvar) {
    using KR = KalmanReal<P>;
    constexpr int NS = P / 2, NT = KR::NT;
    double lam[P], Lam[NT];
#pragma unroll
    for (int j = 0; j < P; j++) lam[j] = 0.0;
#pragma unroll
    for (int j = 0; j < NT; j++) Lam[j] = 0.0;
    const double* qip = rq + (P + 2) * qs - k0;
    long long k = k1 - 1;
    while (k >= k0 && qip[k] == (double)ny) k--;   // forecasts are done
    double fa[NS > 0 ? NS : 1], fb[NS > 0 ? NS : 1], fsb[NS > 0 ? NS : 1], fo;
    for (int i = ny - 1; i >= 0; i--) {
        if (i + 1 < ny) {
            KR::template transition<false>(prm, tb, dt[i], fa, fb, fsb, &fo);
            KR::propagate_vec_t(fa, fb, fsb, fo, lam);
            KR::congruence_t(Lam, fa, fb, fsb, fo);
        }
        double g[P], K[P], u[P];
#pragma unroll
        for (int j = 0; j < P; j++) g[j] = rp[j * ps + i];
        const double m = rp[P * ps + i], S = rp[(P + 1) * ps + i];
        const double inv = 1.0 / S, yc = y[i] - prm.mu;
#pragma unroll
        for (int j = 0; j < P; j++) K[j] = g[j] * inv;
        KR::sym_mul(Lam, K, u);
        const double ui = (yc - m) * inv - KR::dot(K, lam);
        const double di = inv + KR::dot(K, u);
        loo_var[i] = 1.0 / di;
        loo_mean[i] = yc - ui / di;
#pragma unroll
        for (int j = 0; j < P; j += 2) lam[j] += ui;
        KR::info_update(Lam, u, di);
        double Lg[P];
        KR::sym_mul(Lam, g, Lg);
        mean[i] = m + KR::dot(g, lam);
        var[i] = KR::observe_vec(g) - KR::dot(g, Lg);
        for (; k >= k0 && qip[k] == (double)i; k--) {
            double w[P], Lw[P];
#pragma unroll
            for (int j = 0; j < P; j++) w[j] = rq[j * qs + (k - k0)];
            KR::sym_mul(Lam, w, Lw);
            qmean[perm[k]] = rq[P * qs + (k - k0)] + KR::dot(w, lam);
            qvar[perm[k]] = rq[(P + 1) * qs + (k - k0)] - KR::dot(w, Lw);
        }
    }
}

}  // namespace carma
