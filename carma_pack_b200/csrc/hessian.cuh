// hessian.cuh -- the finite-difference stencil of carma_multi_hessian and its assembly into the gradient, Hessian and
// covariance of one curve's log-density.  Host-device code: multi_hessian_eval_kernel builds the stencil rows on the
// device, multi_hessian_assemble_kernel runs hess_assemble one thread per curve, and tests/host_check/hesscheck.cu
// compiles both for the host.
//
// Steps h_i = rel_step * s_i with s = (theta_0, theta_1, theta_0, 1, 1, ...): sigma_y and measerr_scale take relative
// steps, mu a step in units of sigma_y, and every coordinate from 3 on (log or logit) an absolute step.  The
// d^2 + d + 1 points of a curve, in this order:
//   k = 0                     the centre;
//   k = 1 .. d                theta + h_i e_i           (i = k - 1);
//   k = d + 1 .. 2d           theta - h_i e_i           (i = k - d - 1);
//   k = 2d + 1 + 2r (+ 1)     theta + h_i e_i + h_j e_j (then theta - h_i e_i - h_j e_j) for the r-th pair i < j in
//                             row-major order (0,1), (0,2), ..., (0,d-1), (1,2), ...
// Every perturbed coordinate is one rounded add theta_i +- h_i, so numpy reproduces each row bit for bit.
#pragma once
#include <math.h>

#include "theta_transform.cuh"

namespace carma {

__host__ __device__ inline int hess_points(int d) { return d * d + d + 1; }

// s_i of the row (theta_0, theta_1, ...); the step is the one rounded product rel_step * s_i
__host__ __device__ inline double hess_scale(double th0, double th1, int i) {
    return i == 1 ? th1 : (i == 0 || i == 2) ? th0 : 1.0;
}

// The coordinates stencil point k moves: a (sign sa) and b (sign sb), -1 where none.
__host__ __device__ inline void hess_point_dirs(int k, int d, int* a, double* sa, int* b, double* sb) {
    *a = -1; *b = -1; *sa = 0.0; *sb = 0.0;
    if (k == 0) return;
    if (k <= d) { *a = k - 1; *sa = 1.0; return; }
    if (k <= 2 * d) { *a = k - d - 1; *sa = -1.0; return; }
    const int r = k - 2 * d - 1;
    int pair = r >> 1, i = 0;
    while (pair >= d - 1 - i) { pair -= d - 1 - i; i++; }
    *a = i; *b = i + 1 + pair;
    *sa = *sb = (r & 1) ? -1.0 : 1.0;
}

// One curve: f its hess_points(d) stencil values, h its d steps.  Writes g (d), H (d x d) and cov (d x d, row-major)
// and returns the CARMA_HESS_* status; outputs the status declares invalid are NaN.  H_ij (i < j) is formed once and
// mirrored, so H is exactly symmetric; cov = (-H)^-1 through the Cholesky factor L of -H (cov = L^-T L^-1).
__host__ __device__ inline int hess_assemble(int d, const double* f, const double* h, double* g, double* H, double* cov) {
    const int n = hess_points(d);
    int status = CARMA_HESS_OK;
    if (f[0] == -INFINITY) status = CARMA_HESS_REJECTED;
    else {
        for (int k = 0; k < n; k++)
            if (!isfinite(f[k])) status = CARMA_HESS_NONFINITE;
        for (int i = 0; i < d; i++)
            if (!isfinite(h[i]) || h[i] == 0.0) status = CARMA_HESS_NONFINITE;
    }
    if (status != CARMA_HESS_OK) {
        for (int i = 0; i < d; i++) g[i] = NAN;
        for (int i = 0; i < d * d; i++) H[i] = cov[i] = NAN;
        return status;
    }
    const double f0 = f[0];
    const double* fp = f + 1;       // theta + h_i e_i
    const double* fm = f + 1 + d;   // theta - h_i e_i
    for (int i = 0; i < d; i++) {
        g[i] = (fp[i] - fm[i]) / (2.0 * h[i]);
        H[i * d + i] = (fp[i] - 2.0 * f0 + fm[i]) / (h[i] * h[i]);
    }
    const double* fpair = f + 1 + 2 * d;
    for (int i = 0, r = 0; i < d; i++)
        for (int j = i + 1; j < d; j++, r++) {
            const double num = fpair[2 * r] - fp[i] - fp[j] + 2.0 * f0 - fm[i] - fm[j] + fpair[2 * r + 1];
            H[i * d + j] = H[j * d + i] = num / (2.0 * h[i] * h[j]);
        }
    // Cholesky factor L of -H (lower triangle), W = L^-1, cov = W^T W
    double L[MAX_D * MAX_D];
    for (int j = 0; j < d; j++) {
        double s = -H[j * d + j];
        for (int k = 0; k < j; k++) s -= L[j * MAX_D + k] * L[j * MAX_D + k];
        if (!(s > 0.0) || !isfinite(s)) {
            for (int i = 0; i < d * d; i++) cov[i] = NAN;
            return CARMA_HESS_NOT_NEGDEF;
        }
        const double ljj = sqrt(s);
        L[j * MAX_D + j] = ljj;
        for (int i = j + 1; i < d; i++) {
            double t = -H[i * d + j];
            for (int k = 0; k < j; k++) t -= L[i * MAX_D + k] * L[j * MAX_D + k];
            L[i * MAX_D + j] = t / ljj;
        }
    }
    double W[MAX_D * MAX_D];
    for (int j = 0; j < d; j++) {
        W[j * MAX_D + j] = 1.0 / L[j * MAX_D + j];
        for (int i = j + 1; i < d; i++) {
            double t = 0.0;
            for (int k = j; k < i; k++) t += L[i * MAX_D + k] * W[k * MAX_D + j];
            W[i * MAX_D + j] = -t / L[i * MAX_D + i];
        }
    }
    for (int i = 0; i < d; i++)
        for (int j = i; j < d; j++) {
            double t = 0.0;
            for (int k = j; k < d; k++) t += W[k * MAX_D + i] * W[k * MAX_D + j];
            cov[i * d + j] = cov[j * d + i] = t;
        }
    return CARMA_HESS_OK;
}

}  // namespace carma
