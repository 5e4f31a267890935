// laplace.cuh -- the per-curve arithmetic of carma_multi_laplace (importance sampling from the Laplace approximation):
// the Cholesky factor of the proposal covariance and the pieces of the weight summaries (weight ESS, the
// generalised-Pareto k-hat of PSIS, systematic resampling).  Host-device code: survey.cu runs it in
// multi_laplace_factor_kernel / multi_laplace_summary_kernel, and tests/host_check/laplacecheck.cu compiles it for the
// host.  The formulas are documented at carma_multi_laplace in
// include/carma_b200.h.
#pragma once
#include <math.h>
#include <float.h>

#include "theta_transform.cuh"

namespace carma {

enum { STREAM_LAPLACE = 6, STREAM_LAPLACE_RESAMPLE = 7 };

constexpr double LAP_LOG_2PI = 1.8378770664093453;            // np.log(2 * np.pi)
constexpr double LAP_LOG_DBL_MIN = -708.3964185322641;        // np.log(np.finfo(float).tiny)

// one rounded product / difference: the device would otherwise contract them into FMAs, the host does not
__host__ __device__ __forceinline__ double lap_mul(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
__host__ __device__ __forceinline__ double lap_sub(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dsub_rn(a, b);
#else
    return a - b;
#endif
}

// Lower Cholesky factor L (d x d, row-major, upper triangle set to 0) of cov, reading only cov's lower triangle, and
// log|L| = sum_i log L_ii.  Returns CARMA_LAPLACE_OK, or CARMA_LAPLACE_BAD_COV (L and logdet NaN) when the centre row
// or the lower triangle is not finite or a pivot is not positive.
__host__ __device__ inline int lap_cholesky(int d, const double* centre, const double* cov, double* L, double* logdet) {
    bool ok = true;
    for (int i = 0; i < d; i++) {
        ok = ok && isfinite(centre[i]);
        for (int j = 0; j <= i; j++) ok = ok && isfinite(cov[i * d + j]);
    }
    double ld = 0.0;
    for (int j = 0; j < d && ok; j++) {
        double s = cov[j * d + j];
        for (int k = 0; k < j; k++) s = lap_sub(s, lap_mul(L[j * d + k], L[j * d + k]));
        if (!(s > 0.0) || !isfinite(s)) { ok = false; break; }
        const double ljj = sqrt(s);
        L[j * d + j] = ljj;
        for (int i = j + 1; i < d; i++) {
            double t = cov[i * d + j];
            for (int k = 0; k < j; k++) t = lap_sub(t, lap_mul(L[i * d + k], L[j * d + k]));
            L[i * d + j] = t / ljj;
        }
        for (int i = 0; i < j; i++) L[i * d + j] = 0.0;
        ld += log(ljj);
    }
    if (!ok) {
        for (int i = 0; i < d * d; i++) L[i] = NAN;
        *logdet = NAN;
        return CARMA_LAPLACE_BAD_COV;
    }
    *logdet = ld;
    return CARMA_LAPLACE_OK;
}

// M of the tail: ceil(min(0.2 S, 3 sqrt(S)))
__host__ __device__ inline size_t psis_tail_len(size_t S) {
    return (size_t)ceil(fmin(0.2 * (double)S, 3.0 * sqrt((double)S)));
}

// the m = 30 + floor(sqrt(n)) trial b_i of the generalised-Pareto fit to the ascending tail x (n values), i = 1 .. m
__host__ __device__ inline int gpd_m(int n) { return 30 + (int)sqrt((double)n); }
__host__ __device__ inline double gpd_b(int i, int m, const double* x, int n) {
    const double xq = x[(int)((double)n / 4.0 + 0.5) - 1];
    return (1.0 - sqrt((double)m / ((double)i - 0.5))) / (3.0 * xq) + 1.0 / x[n - 1];
}
// the profile log-likelihood L_i = n (log(-b / k) - k - 1) of b with k = mean_t log1p(-b x_t)
__host__ __device__ inline double gpd_profile(int n, double b, double k) { return n * (log(-(b / k)) - k - 1.0); }
// the weight w_i = 1 / sum_l exp(L_l - L_i) of trial b_i (L of m entries), 0 where it is below 10 eps (dropped)
__host__ __device__ inline double gpd_weight(int i, int m, const double* Lp) {
    double s = 0.0;
    for (int l = 0; l < m; l++) s += exp(Lp[l] - Lp[i]);
    const double w = 1.0 / s;
    return w >= 10.0 * DBL_EPSILON ? w : 0.0;
}
// bbar = sum_i b_i w_i / sum_l w_l, the posterior mean of b
__host__ __device__ inline double gpd_bbar(int m, const double* b, const double* w) {
    double tot = 0.0, bbar = 0.0;
    for (int i = 0; i < m; i++) tot += w[i];
    for (int i = 0; i < m; i++) bbar += b[i] * (w[i] / tot);
    return bbar;
}
// k-hat from the mean k = mean_t log1p(-bbar x_t) over the n tail values: the weakly informative prior of _gpdfit
__host__ __device__ inline double gpd_khat(int n, double k) { return (n * k + 5.0) / (n + 10.0); }

// target of systematic resample i: ((i + u) / S) T
__host__ __device__ inline double resample_target(size_t i, double u, size_t S, double T) {
    return ((double)i + u) / (double)S * T;
}
// the first j with C[j] > target, capped at S - 1 (C ascending: running sums of the weights)
__host__ __device__ inline size_t resample_find(const double* C, size_t S, double target) {
    size_t lo = 0, hi = S - 1;   // the answer lies in [lo, hi]
    while (lo < hi) {
        const size_t mid = lo + (hi - lo) / 2;
        if (C[mid] > target) hi = mid;
        else lo = mid + 1;
    }
    return lo;
}

}  // namespace carma
