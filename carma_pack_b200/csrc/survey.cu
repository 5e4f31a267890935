// survey.cu -- the KalmanFilterp outputs for every light curve of a multi-series, taking one theta row per curve the
// way carma_multi_loglik does:
//   multi_filter_kernel<P>     one thread = one curve: K4's recursion (same operations, so the log-density is bitwise
//                              K4's) that also stores the one-step predictive mean and variance of every point;
//   residual_acf_kernel        one warp = one curve: moments and autocorrelation of the standardised residuals
//                              (the numeric part of CarmaSample.assess_fit_values) without sending them to the host;
//   predict_forward_kernel<P>  one thread = one curve: the same recursion with a cursor over the curve's (time-sorted)
//   predict_query_kernel<P>    queries, parking the state in front of each; then one thread = one query resumes from it
//                              (predict_resume, shared with the single-series predict_real_kernel);
//   condsim_prior_kernel<P>    one thread = one (curve, path): the prior draw of conditional simulation (Matheron's rule,
//                              as carma_simulate); the two predict kernels then run on every path's residual data;
//   multi_smooth_kernel<P>     one thread = one curve: K4's recursion forward, storing per-point and per-query records,
//                              then the adjoint (Bryson-Frazier) recursion backward: smoothed values, leave-one-out laws
//                              and queries in O(ny + nq) steps;
//   multi_hessian_eval_kernel<P>  one thread = one (curve, stencil point): K4's body on a finite-difference row;
//   multi_hessian_assemble_kernel one thread = one curve: gradient, Hessian and covariance from its stencil values;
//   multi_laplace_factor_kernel   one thread = one curve: Cholesky factor of its proposal covariance (laplace.cuh);
//   multi_laplace_eval_kernel<P>  one thread = one (curve, draw): the proposal draw, then K4's body on it;
//   multi_laplace_summary_kernel  one block = one curve: weight ESS, Pareto k-hat and systematic resampling.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <string>
#include <vector>

#include "hessian.cuh"
#include "kalman_real.cuh"
#include "laplace.cuh"
#include "select.cuh"
#include "series.h"

namespace carma {

constexpr int SF_BLOCK = 64;

__device__ __forceinline__ void stg4(double* q, double a, double b, double c, double d) {   // q 32-byte aligned
    asm volatile("st.global.v4.f64 [%0], {%1, %2, %3, %4};" ::"l"(q), "d"(a), "d"(b), "d"(c), "d"(d) : "memory");
}

// filter_span_blocks (kalman_real.cuh) with the predictive mean / variance of every point stored to mo / vo.  The same
// loads and the same steps in the same order, so the accumulated log-density is bitwise K4's.  Each thread writes its
// own curve: with one 8-byte store per point a warp store touches 32 sectors.  BLKST: the four points of a block are
// written with one 32-byte store per array (mo / vo sit like dt within a sector; the head and tail peel with scalar
// stores); otherwise one scalar store per point and array.
template <int P, bool ALLC, bool BLKST, class Tab>
__device__ void filter_span_emit(KalmanReal<P>& kf, LogLikAcc& acc, const RealParams<P>& prm, const Tab& tb,
                                 const double* __restrict__ dt, const double* __restrict__ y,
                                 const double* __restrict__ E, int len, double* __restrict__ mo,
                                 double* __restrict__ vo) {
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
    for (; i < head; i++) {
        mo[i] = kf.mean; vo[i] = kf.var;
        step(dt[i], y[i], E[i + 1]);
    }
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
            const double m0 = kf.mean, v0 = kf.var;
            step(cdt.a, cy.a, cE.b);
            const double m1 = kf.mean, v1 = kf.var;
            step(cdt.b, cy.b, cE.c);
            const double m2 = kf.mean, v2 = kf.var;
            step(cdt.c, cy.c, cE.d);
            const double m3 = kf.mean, v3 = kf.var;
            step(cdt.d, cy.d, e_last);
            if (BLKST) {
                stg4(mo + i, m0, m1, m2, m3);
                stg4(vo + i, v0, v1, v2, v3);
            } else {
                mo[i] = m0; mo[i + 1] = m1; mo[i + 2] = m2; mo[i + 3] = m3;
                vo[i] = v0; vo[i + 1] = v1; vo[i + 2] = v2; vo[i + 3] = v3;
            }
            i += 4;
            since += 4;
            if (since >= RENORM_EVERY - 8) { acc.renorm(since); since = 0; }
            if (!nx || i + 4 > nadv) break;
            cdt = ndt; cy = ny_; cE = nE;
        }
    }
    for (; i < nadv; i++, since++) {
        mo[i] = kf.mean; vo[i] = kf.var;
        step(dt[i], y[i], E[i + 1]);
    }
    if (since) acc.renorm(since);
    {   // the last point is only scored
        mo[len - 1] = kf.mean; vo[len - 1] = kf.var;
        const double innov = (y[len - 1] - prm.mu) - kf.mean;
        const double inv = rcp_fast(kf.var);
        acc.add(kf.var, innov, inv);
        acc.renorm(1);
    }
}

template <int P, bool BLKST>
__global__ void __launch_bounds__(SF_BLOCK, P <= 3 ? 8 : 1)   // K4's bounds
multi_filter_kernel(const double* __restrict__ dt, const double* __restrict__ y, const double* __restrict__ e2,
                    const long long* __restrict__ off, size_t ncurves, double dt_max, int kind, int q, int d,
                    unsigned flags, const carma_prior_t* __restrict__ priors, const double* __restrict__ theta,
                    double* __restrict__ mean, double* __restrict__ var, double* __restrict__ out /* may be null */) {
    MathTab tb;
    tb.load();
    const size_t c = (size_t)blockIdx.x * SF_BLOCK + threadIdx.x;
    if (c >= ncurves) return;
    const long long o0 = off[c], o1 = off[c + 1];
    const int ny = (int)(o1 - o0);
    double th[MAX_D];
#pragma unroll
    for (int j = 0; j < MAX_D; j++) th[j] = (j < d) ? theta[c * (size_t)d + j] : 0.0;
    RealParams<P> prm;
    carma_prior_t pr = priors[c];
    if (transform_theta<P>(kind, q, flags, pr, th, dt_max, prm) != TT_OK) {
        for (int i = 0; i < ny; i++) { mean[o0 + i] = NAN; var[o0 + i] = NAN; }
        if (out) out[c] = -INFINITY;
        return;
    }
    KalmanReal<P> kf;
    LogLikAcc acc;
    kf.reset(prm, e2[o0]);
    acc.init();
    constexpr unsigned ALL = (P / 2 > 0) ? ((1u << (P / 2)) - 1u) : 0u;
    if (__all_sync(__activemask(), prm.cmask == ALL))   // warp-uniform, as filter_span_blocks_any
        filter_span_emit<P, true, BLKST>(kf, acc, prm, tb, dt + o0, y + o0, e2 + o0, ny, mean + o0, var + o0);
    else
        filter_span_emit<P, false, BLKST>(kf, acc, prm, tb, dt + o0, y + o0, e2 + o0, ny, mean + o0, var + o0);
    if (out) {
        const SeriesPtr src{dt + o0, y + o0, e2 + o0 + 1};
        out[c] = (acc.bad() ? loglik_exact_slow<P>(prm, tb, src, ny, e2[o0]) : acc.value()) + prm.logprior;
    }
}

// One warp per curve.  Pass 1 turns mean into the standardised residuals r = (y - (mean + mu)) / sqrt(var) in place and
// sums r and r^2; pass 2: lane k sums (r_i - rbar)(r_{i+L} - rbar) over i in index order for its lags L = k, k + 32, ...
// (r and r^2), with r_i read by every lane and r_{i+L} adjacent across lanes.  Fixed summation order: deterministic.
// out row (3 + 2 nlags): loglik, mean(r), population std(r), acf(r)[1..nlags], acf(r^2)[1..nlags] (mean-subtracted,
// normalised by lag 0).
constexpr int ACF_BLOCK = 128;
__global__ void __launch_bounds__(ACF_BLOCK)
residual_acf_kernel(const double* __restrict__ y, const long long* __restrict__ off, size_t ncurves,
                    const double* __restrict__ theta, int d, const double* __restrict__ loglik, double* mean,
                    const double* __restrict__ var, int nlags, double* __restrict__ out) {
    const size_t c = ((size_t)blockIdx.x * ACF_BLOCK + threadIdx.x) / 32;
    const int lane = threadIdx.x & 31;
    if (c >= ncurves) return;   // uniform over the warp
    const long long o0 = off[c];
    const int ny = (int)(off[c + 1] - o0);
    const double mu = theta[c * (size_t)d + 2];
    double* r = mean + o0;
    double s1 = 0.0, s2 = 0.0;
    for (int i = lane; i < ny; i += 32) {
        const double ri = (y[o0 + i] - (r[i] + mu)) / sqrt(var[o0 + i]);
        r[i] = ri;
        s1 += ri;
        s2 += ri * ri;
    }
#pragma unroll
    for (int k = 16; k >= 1; k >>= 1) {
        s1 += __shfl_xor_sync(0xffffffffu, s1, k);
        s2 += __shfl_xor_sync(0xffffffffu, s2, k);
    }
    __syncwarp();   // the residuals of every lane are visible to the warp
    const double rbar = s1 / ny, qbar = s2 / ny;
    const int w = 3 + 2 * nlags;
    double* o = out + c * (size_t)w;
    double c0r = 0.0, c0q = 0.0;
    for (int L = lane; L <= nlags; L += 32) {
        double ar = 0.0, aq = 0.0;
        for (int i = 0; i + L < ny; i++) {
            const double a = r[i], b = r[i + L];
            ar += (a - rbar) * (b - rbar);
            aq += (a * a - qbar) * (b * b - qbar);
        }
        if (L == 0) { c0r = ar; c0q = aq; }
        else { o[2 + L] = ar; o[2 + nlags + L] = aq; }
    }
    c0r = __shfl_sync(0xffffffffu, c0r, 0);
    c0q = __shfl_sync(0xffffffffu, c0q, 0);
    for (int L = lane; L <= nlags; L += 32) {
        if (L == 0) continue;
        o[2 + L] /= c0r;
        o[2 + nlags + L] /= c0q;
    }
    if (lane == 0) {
        o[0] = loglik[c];
        o[1] = rbar;
        o[2] = sqrt(c0r / ny);
    }
}

// Predict, forward part.  Curve c's queries are qtq[qoff[c] .. qoff[c+1]), sorted by time, on the curve's own axis (the
// running sum of its gaps from 0, as carma_multi_series_get_curve forms it).  For every query the record holds the state
// (z, D) predicted at point ip - 1 (ip = number of data times strictly before t*), then t* - t[ip-1], t[ip] - t* and ip.
template <int P>
struct PredictRec {
    static constexpr int NT = P * (P + 1) / 2, SD = P + NT, R = SD + 3;
};

// The paths one launch of the predict kernels serves when they are instantiated with PATHS = true, for conditional
// simulation: paths j0 .. j0 + B - 1 of every curve; path jj filters its own residual-data row y + jj * ystride
// (centred: mu = 0) with theta row c * rpc + j (rpc = npaths: one row per path) or c (rpc = 1), and the query pass adds
// its mean to the prior draw already stored at path jj's destination jj * nq + perm[k].  Threads are path-minor (curve
// c, path jj at c * B + jj; query k, path jj at k * B + jj), so the lanes of a warp walk the same curve and query and
// share its trip counts.  PATHS = false is predict: one path, the curve's data, theta row c -- the index arithmetic
// folds away and the kernels compile as they did before paths existed.
struct PathSet {
    unsigned B = 1, j0 = 0;
    size_t ystride = 0, rpc = 1;
    __device__ size_t theta_row(size_t c, unsigned jj) const { return c * rpc + (rpc > 1 ? j0 + jj : 0); }
};

template <int P, bool PATHS>
__global__ void __launch_bounds__(SF_BLOCK)
predict_forward_kernel(const double* __restrict__ dt, const double* __restrict__ y, const double* __restrict__ e2,
                       const long long* __restrict__ off, size_t ncurves, double dt_max, int kind, int q, int d,
                       unsigned flags, const carma_prior_t* __restrict__ priors, const double* __restrict__ theta,
                       const long long* __restrict__ qoff, const double* __restrict__ qtq, PathSet ps,
                       double* __restrict__ rec, RealParams<P>* __restrict__ prm_out, int* __restrict__ status_out) {
    using PR = PredictRec<P>;
    MathTab tb;
    tb.load();
    const unsigned B = PATHS ? ps.B : 1u;
    const size_t tid = (size_t)blockIdx.x * SF_BLOCK + threadIdx.x;
    if (tid >= ncurves * B) return;
    const size_t c = tid / B;
    const unsigned jj = (unsigned)(tid - c * B);
    long long k = qoff[c];
    const long long k1 = qoff[c + 1];
    double th[MAX_D];
    const size_t row = PATHS ? ps.theta_row(c, jj) : c;
#pragma unroll
    for (int j = 0; j < MAX_D; j++) th[j] = (j < d) ? theta[row * d + j] : 0.0;
    RealParams<P> prm;
    carma_prior_t pr = priors[c];
    const int status = transform_theta<P>(kind, q, flags, pr, th, dt_max, prm);
    if (PATHS) prm.mu = 0.0;   // the residual data are centred
    prm_out[tid] = prm;      // the query threads of this curve and path read the constants from here
    status_out[tid] = status;
    if (status != TT_OK || k == k1) return;
    const long long o0 = off[c];
    const int ny = (int)(off[c + 1] - o0);
    const double *cdt = dt + o0, *cy = y + (PATHS ? jj * ps.ystride : 0) + o0, *cE = e2 + o0;
    double t = 0.0;
    for (; k < k1 && !(qtq[k] > t); k++) {   // at or before the first point: ip = 0
        double* r = rec + ((size_t)k * B + jj) * PR::R;
        r[PR::SD] = 0.0;
        r[PR::SD + 1] = fabs(t - qtq[k]);
        r[PR::SD + 2] = 0.0;
    }
    KalmanReal<P> kf;
    kf.reset(prm, cE[0]);
    for (int i = 0; i < ny && k < k1; i++) {
        const bool last = i + 1 == ny;
        const double tn = last ? 0.0 : t + cdt[i];
        for (; k < k1 && (last || !(qtq[k] > tn)); k++) {   // t[i] < t* <= t[i+1], or past the last point
            double* r = rec + ((size_t)k * B + jj) * PR::R;
#pragma unroll
            for (int j = 0; j < P; j++) r[j] = kf.z[j];
#pragma unroll
            for (int j = 0; j < PR::NT; j++) r[P + j] = kf.D[j];
            r[PR::SD] = fabs(qtq[k] - t);
            r[PR::SD + 1] = last ? 0.0 : fabs(tn - qtq[k]);
            r[PR::SD + 2] = (double)(i + 1);
        }
        if (last || k == k1) break;
        const double innov = (cy[i] - prm.mu) - kf.mean;
        kf.template advance<false>(prm, tb, innov, 1.0 / kf.var, cdt[i], cE[i + 1]);
        t = tn;
    }
}

// Predict, query part: one thread per query and path (queries sorted curve-major, then by time, so a warp walks one
// curve), result written to the caller's position perm[k] of the path's row.
template <int P, bool PATHS>
__global__ void __launch_bounds__(SF_BLOCK)
predict_query_kernel(const double* __restrict__ dt, const double* __restrict__ y, const double* __restrict__ e2,
                     const long long* __restrict__ off, const int* __restrict__ qcurve, const long long* __restrict__ perm,
                     size_t nq, PathSet ps, const double* __restrict__ rec, const RealParams<P>* __restrict__ prms,
                     const int* __restrict__ status, double* __restrict__ qmean, double* __restrict__ qvar /* may be null */) {
    using PR = PredictRec<P>;
    MathTab tb;
    tb.load();
    const unsigned B = PATHS ? ps.B : 1u;
    const size_t u = (size_t)blockIdx.x * SF_BLOCK + threadIdx.x;
    if (u >= nq * B) return;
    const size_t k = u / B;
    const unsigned jj = (unsigned)(u - k * B);
    const int c = qcurve[k];
    const size_t cp = (size_t)c * B + jj;
    const size_t dst = jj * nq + (size_t)perm[k];
    if (status[cp] != TT_OK) { qmean[dst] = NAN; if (qvar) qvar[dst] = NAN; return; }
    const RealParams<P> prm = prms[cp];
    const double* r = rec + u * PR::R;
    const long long o0 = off[c];
    const int ny = (int)(off[c + 1] - o0);
    const double* cy = y + (PATHS ? jj * ps.ystride : 0) + o0;
    double pm, pv;
    predict_resume<P>(prm, tb, r, r + P, (int)r[PR::SD + 2], ny, r[PR::SD], r[PR::SD + 1],
                      [&](int i) { return cy[i]; }, [&](int i) { return dt[o0 + i]; },
                      [&](int i) { return e2[o0 + i]; }, &pm, &pv);
    qmean[dst] = PATHS ? qmean[dst] + pm : pm;
    if (qvar) qvar[dst] = pv;
}

// Conditional simulation, prior part: one thread per curve and path (path-minor, as PathSet).  The noise-free
// innovations filter (condsim_draw / condsim_next, shared with carma_simulate's sim_prior_kernel) walks the curve's
// merged grid: its data points and its time-sorted queries, a query equal to a data time after it, all on the curve's
// own axis.  Merged point k of global path j uses the Philox counters (seed, j, STREAM_CONDSIM, k, curve_offset + c).
// Writes the residual data (y - mu) - f - sqrt(scale) yerr eps of every point to the path's row yres + jj * ystride
// (CSR layout) and f + mu of every query to out[jj * nq + perm[k]].  A rejected theta row gives NaN queries.
template <int P>
__global__ void __launch_bounds__(SF_BLOCK)
condsim_prior_kernel(const double* __restrict__ dt, const double* __restrict__ y, const double* __restrict__ e2,
                     const long long* __restrict__ off, size_t ncurves, double dt_max, int kind, int q, int d,
                     unsigned flags, const carma_prior_t* __restrict__ priors, const double* __restrict__ theta,
                     const long long* __restrict__ qoff, const double* __restrict__ qtq, const long long* __restrict__ perm,
                     size_t nq, PathSet ps, unsigned long long seed, uint32_t curve_offset, double* __restrict__ yres,
                     double* __restrict__ out) {
    MathTab tb;
    tb.load();
    const size_t tid = (size_t)blockIdx.x * SF_BLOCK + threadIdx.x;
    if (tid >= ncurves * ps.B) return;
    const size_t c = tid / ps.B;
    const unsigned jj = (unsigned)(tid - c * ps.B);
    long long k = qoff[c];
    const long long k1 = qoff[c + 1];
    double* o = out + jj * nq;
    double th[MAX_D];
    const size_t row = ps.theta_row(c, jj);
#pragma unroll
    for (int j = 0; j < MAX_D; j++) th[j] = (j < d) ? theta[row * d + j] : 0.0;
    RealParams<P> prm;
    carma_prior_t pr = priors[c];
    if (transform_theta<P>(kind, q, flags, pr, th, dt_max, prm) != TT_OK) {
        for (; k < k1; k++) o[perm[k]] = NAN;
        return;
    }
    const double mu = prm.mu, sscale = sqrt(prm.scale);
    prm.scale = 0.0;   // the process itself carries no measurement noise
    KalmanReal<P> kf;
    kf.reset(prm, 0.0);
    const long long o0 = off[c];
    const int ny = (int)(off[c + 1] - o0);
    const double *cdt = dt + o0, *cy = y + o0, *cE = e2 + o0;
    double* res = yres + jj * ps.ystride + o0;
    const uint32_t path = ps.j0 + jj, block = curve_offset + (uint32_t)c;
    double td = 0.0, tprev = 0.0, innov = 0.0;   // time of data point i, of the previous merged point
    int i = 0;
    for (uint32_t km = 0; i < ny || k < k1; km++) {
        const bool data = k == k1 || (i < ny && td <= qtq[k]);
        const double tm = data ? td : qtq[k];
        if (km > 0) condsim_next(kf, prm, tb, innov, tm - tprev);
        double rr, sn;
        const double f = condsim_draw(kf, seed, path, km, block, &innov, &rr, &sn);
        if (data) {
            res[i] = (cy[i] - mu) - f - sscale * sqrt(cE[i]) * rr * sn;   // second normal: the measurement noise
            td += cdt[i];
            i++;
        } else {
            o[perm[k]] = f + mu;
            k++;
        }
        tprev = tm;
    }
}

// Smoother: one thread = one curve of a chunk of curves (smooth_forward / smooth_backward, kalman_real.cuh).  The
// records live in scratch, field-major: a curve's point records at rp + (o0 - pbase), aligned like its dt / y / e2 arrays
// (pbase: the chunk's first point rounded down to a multiple of 4, stride pstride), its query records at
// rq + (qoff[c] - qbase) (stride qstride).  Outputs without mu at the curve's CSR positions; a row the transform rejects
// gives NaN everywhere and -inf loglik.
struct SmoothChunk {
    size_t c0 = 0, nc = 0;
    long long pbase = 0, qbase = 0;
    size_t pstride = 0, qstride = 0;
};

template <int P>
__global__ void __launch_bounds__(SF_BLOCK, P <= 3 ? 8 : 1)   // K4's bounds
multi_smooth_kernel(const double* __restrict__ dt, const double* __restrict__ y, const double* __restrict__ e2,
                    const long long* __restrict__ off, SmoothChunk ch, double dt_max, int kind, int q, int d,
                    unsigned flags, const carma_prior_t* __restrict__ priors, const double* __restrict__ theta,
                    const long long* __restrict__ qoff, const double* __restrict__ qtq, const long long* __restrict__ perm,
                    double* __restrict__ rp, double* __restrict__ rq, double* __restrict__ mean, double* __restrict__ var,
                    double* __restrict__ loo_mean, double* __restrict__ loo_var, double* __restrict__ loglik,
                    double* __restrict__ qmean, double* __restrict__ qvar) {
    MathTab tb;
    tb.load();
    const size_t tid = (size_t)blockIdx.x * SF_BLOCK + threadIdx.x;
    if (tid >= ch.nc) return;
    const size_t c = ch.c0 + tid;
    const long long o0 = off[c];
    const int ny = (int)(off[c + 1] - o0);
    const long long k0 = qoff[c], k1 = qoff[c + 1];
    double th[MAX_D];
#pragma unroll
    for (int j = 0; j < MAX_D; j++) th[j] = (j < d) ? theta[c * (size_t)d + j] : 0.0;
    RealParams<P> prm;
    carma_prior_t pr = priors[c];
    if (transform_theta<P>(kind, q, flags, pr, th, dt_max, prm) != TT_OK) {
        for (int i = 0; i < ny; i++) { mean[o0 + i] = NAN; var[o0 + i] = NAN; loo_mean[o0 + i] = NAN; loo_var[o0 + i] = NAN; }
        for (long long k = k0; k < k1; k++) { qmean[perm[k]] = NAN; qvar[perm[k]] = NAN; }
        loglik[c] = -INFINITY;
        return;
    }
    const double *cdt = dt + o0, *cy = y + o0, *cE = e2 + o0;
    double* crp = rp + (o0 - ch.pbase);
    double* crq = rq + (k0 - ch.qbase);
    {
        KalmanReal<P> kf;
        LogLikAcc acc;
        kf.reset(prm, cE[0]);
        acc.init();
        constexpr unsigned ALL = (P / 2 > 0) ? ((1u << (P / 2)) - 1u) : 0u;
        if (__all_sync(__activemask(), prm.cmask == ALL))   // warp-uniform, as filter_span_blocks_any
            smooth_forward<P, true>(kf, acc, prm, tb, cdt, cy, cE, ny, crp, ch.pstride, k0, k1, qtq, crq, ch.qstride,
                                    perm, qmean, qvar);
        else
            smooth_forward<P, false>(kf, acc, prm, tb, cdt, cy, cE, ny, crp, ch.pstride, k0, k1, qtq, crq, ch.qstride,
                                     perm, qmean, qvar);
        const SeriesPtr src{cdt, cy, cE + 1};
        loglik[c] = (acc.bad() ? loglik_exact_slow<P>(prm, tb, src, ny, cE[0]) : acc.value()) + prm.logprior;
    }
    smooth_backward<P>(prm, tb, cdt, cy, ny, crp, ch.pstride, k0, k1, crq, ch.qstride, perm, mean + o0, var + o0,
                       loo_mean + o0, loo_var + o0, qmean, qvar);
}

// Hessian, evaluation: one thread per (curve, stencil point) of the curves c0 .. c0 + nc - 1, stencil-minor (thread u:
// curve c0 + u / npts, point u % npts; hessian.cuh), so the lanes of a warp walk the same curve: each 32-byte block of it
// is fetched once per warp and its length does not diverge inside the warp.  The step is one rounded product and the
// row one rounded add or subtract (no contraction), as numpy forms them.  After the row, the body is
// multi_loglik_kernel's (same transform and rate clamp, block loads, slow fallback, log-prior), so fval[u] is what
// carma_multi_loglik returns for that row.
template <int P>
__global__ void __launch_bounds__(SF_BLOCK, P <= 3 ? 8 : 1)   // K4's bounds
multi_hessian_eval_kernel(const double* __restrict__ dt, const double* __restrict__ y, const double* __restrict__ e2,
                          const long long* __restrict__ off, size_t c0, size_t nc, int npts, double dt_max, int kind,
                          int q, int d, unsigned flags, const carma_prior_t* __restrict__ priors,
                          const double* __restrict__ theta, double rel_step, double* __restrict__ fval) {
    MathTab tb;
    tb.load();
    const size_t u = (size_t)blockIdx.x * SF_BLOCK + threadIdx.x;
    if (u >= nc * npts) return;
    const size_t cl = u / npts;
    const int k = (int)(u - cl * npts);
    const size_t c = c0 + cl;
    const long long o0 = off[c], o1 = off[c + 1];
    const int ny = (int)(o1 - o0);
    const double* row = theta + c * (size_t)d;
    const double th0 = row[0], th1 = row[1];
    int a, b;
    double sa, sb;
    hess_point_dirs(k, d, &a, &sa, &b, &sb);
    double th[MAX_D];
#pragma unroll
    for (int j = 0; j < MAX_D; j++) {
        const double v = (j < d) ? row[j] : 0.0;
        const double h = __dmul_rn(rel_step, hess_scale(th0, th1, j));
        const double s = (j == a) ? sa : (j == b) ? sb : 0.0;
        th[j] = (s > 0.0) ? __dadd_rn(v, h) : (s < 0.0) ? __dsub_rn(v, h) : v;
    }
    RealParams<P> prm;
    carma_prior_t pr = priors[c];
    if (transform_theta<P>(kind, q, flags, pr, th, dt_max, prm) != TT_OK) {
        fval[u] = -INFINITY;
        return;
    }
    KalmanReal<P> kf;
    LogLikAcc acc;
    kf.reset(prm, e2[o0]);
    acc.init();
    const SeriesPtr src{dt + o0, y + o0, e2 + o0 + 1};
    filter_span_blocks_any<P>(kf, acc, prm, tb, dt + o0, y + o0, e2 + o0, ny);
    fval[u] = (acc.bad() ? loglik_exact_slow<P>(prm, tb, src, ny, e2[o0]) : acc.value()) + prm.logprior;
}

// Hessian, assembly: one thread per curve of the chunk, hess_assemble on its npts stencil values; outputs at the curve's
// global index.
__global__ void __launch_bounds__(SF_BLOCK)
multi_hessian_assemble_kernel(const double* __restrict__ fval, size_t c0, size_t nc, int d,
                              const double* __restrict__ theta, double rel_step, double* __restrict__ loglik,
                              double* __restrict__ grad, double* __restrict__ hess, double* __restrict__ cov,
                              int* __restrict__ status) {
    const size_t cl = (size_t)blockIdx.x * SF_BLOCK + threadIdx.x;
    if (cl >= nc) return;
    const size_t c = c0 + cl;
    const double* row = theta + c * (size_t)d;
    double h[MAX_D];
    for (int i = 0; i < d; i++) h[i] = __dmul_rn(rel_step, hess_scale(row[0], row[1], i));
    const double* f = fval + cl * (size_t)hess_points(d);
    loglik[c] = f[0];
    status[c] = hess_assemble(d, f, h, grad + c * d, hess + c * d * d, cov + c * d * d);
}

// Laplace importance sampling, factor: one thread per curve of the chunk; L (d x d), log|L| and the CARMA_LAPLACE_OK /
// BAD_COV status at the curve's chunk index.
__global__ void __launch_bounds__(SF_BLOCK)
multi_laplace_factor_kernel(const double* __restrict__ theta, const double* __restrict__ cov, size_t c0, size_t nc,
                            int d, double* __restrict__ L, double* __restrict__ logdet, int* __restrict__ fstat) {
    const size_t cl = (size_t)blockIdx.x * SF_BLOCK + threadIdx.x;
    if (cl >= nc) return;
    const size_t c = c0 + cl;
    fstat[cl] = lap_cholesky(d, theta + c * d, cov + c * d * d, L + cl * d * d, logdet + cl);
}

// Laplace importance sampling, evaluation: one thread per (curve, draw) of the chunk, draw-minor (thread u: chunk curve
// u / S, draw u % S), so the lanes of a warp walk the same curve with broadcast loads, as multi_hessian_eval_kernel.
// The draw (Philox pairs, Box-Muller, the row theta + L z with every product and sum rounded on its own) and its
// proposal log-density, then multi_loglik_kernel's body (same transform and rate clamp, block loads, slow fallback,
// log-prior), so logpost[u] is what carma_multi_loglik returns for the row.  A BAD_COV curve gets NaN rows.
template <int P>
__global__ void __launch_bounds__(SF_BLOCK, P <= 3 ? 8 : 1)   // K4's bounds
multi_laplace_eval_kernel(const double* __restrict__ dt, const double* __restrict__ y, const double* __restrict__ e2,
                          const long long* __restrict__ off, size_t c0, size_t nc, size_t S, double dt_max, int kind,
                          int q, int d, unsigned flags, const carma_prior_t* __restrict__ priors,
                          const double* __restrict__ theta, const double* __restrict__ L,
                          const double* __restrict__ logdet, const int* __restrict__ fstat, unsigned long long seed,
                          uint32_t curve_offset, double* __restrict__ draws, double* __restrict__ logpost,
                          double* __restrict__ logq) {
    MathTab tb;
    tb.load();
    const size_t u = (size_t)blockIdx.x * SF_BLOCK + threadIdx.x;
    if (u >= nc * S) return;
    const size_t cl = u / S;
    const uint32_t j = (uint32_t)(u - cl * S);
    const size_t c = c0 + cl;
    double* out = draws + u * d;
    if (fstat[cl] != CARMA_LAPLACE_OK) {
        for (int i = 0; i < d; i++) out[i] = NAN;
        logpost[u] = NAN;
        logq[u] = NAN;
        return;
    }
    const uint32_t block = curve_offset + (uint32_t)c;
    double z[MAX_D + 1];
    double zz = 0.0;
#pragma unroll
    for (int k = 0; k < MAX_D; k += 2) {
        z[k] = z[k + 1] = 0.0;
        if (k < d) {
            double u0, u1, sn, cs;
            uniforms2(seed, j, STREAM_LAPLACE, (uint32_t)(k / 2), block, &u0, &u1);
            const double r = sqrt(-2.0 * log(u0));
            sincos(6.283185307179586476925286766559 * u1, &sn, &cs);
            z[k] = __dmul_rn(r, cs);
            z[k + 1] = __dmul_rn(r, sn);
            zz = __dadd_rn(zz, __dmul_rn(z[k], z[k]));
            if (k + 1 < d) zz = __dadd_rn(zz, __dmul_rn(z[k + 1], z[k + 1]));
        }
    }
    logq[u] = -0.5 * zz - logdet[cl] - 0.5 * d * LAP_LOG_2PI;
    const double* Lc = L + cl * d * d;
    const double* row = theta + c * (size_t)d;
    double th[MAX_D];
#pragma unroll
    for (int i = 0; i < MAX_D; i++) {
        th[i] = 0.0;
        if (i < d) {
            double s = 0.0;
#pragma unroll
            for (int k = 0; k <= i; k++) s = __dadd_rn(s, __dmul_rn(Lc[i * d + k], z[k]));
            th[i] = __dadd_rn(row[i], s);
            out[i] = th[i];
        }
    }
    RealParams<P> prm;
    carma_prior_t pr = priors[c];
    if (transform_theta<P>(kind, q, flags, pr, th, dt_max, prm) != TT_OK) {
        logpost[u] = -INFINITY;
        return;
    }
    const long long o0 = off[c], o1 = off[c + 1];   // read here rather than first: P = 5 then spills half as much
    const int ny = (int)(o1 - o0);
    KalmanReal<P> kf;
    LogLikAcc acc;
    kf.reset(prm, e2[o0]);
    acc.init();
    const SeriesPtr src{dt + o0, y + o0, e2 + o0 + 1};
    filter_span_blocks_any<P>(kf, acc, prm, tb, dt + o0, y + o0, e2 + o0, ny);
    logpost[u] = (acc.bad() ? loglik_exact_slow<P>(prm, tb, src, ny, e2[o0]) : acc.value()) + prm.logprior;
}

// Fixed-order block reductions of LAP_THREADS threads (xor butterflies, then warp 0 over the warp partials): the same
// inputs give the same bits on every run.
constexpr int LAP_THREADS = 256;
constexpr int LAP_TAIL_MAX = 4096;   // >= psis_tail_len(CARMA_LAPLACE_MAX_DRAWS) = 3072; a power of two for the sort
static_assert(3 * 1024 <= LAP_TAIL_MAX, "the Pareto tail must fit the shared sort");

template <bool MAX>
__device__ __forceinline__ double lap_block_reduce(double v, double* sh) {
#pragma unroll
    for (int k = 16; k >= 1; k >>= 1) {
        const double o = __shfl_xor_sync(0xffffffffu, v, k);
        v = MAX ? fmax(v, o) : v + o;
    }
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    __syncthreads();   // sh is free
    if (lane == 0) sh[w] = v;
    __syncthreads();
    if (w == 0) {
        v = lane < LAP_THREADS / 32 ? sh[lane] : (MAX ? -INFINITY : 0.0);
#pragma unroll
        for (int k = 16; k >= 1; k >>= 1) {
            const double o = __shfl_xor_sync(0xffffffffu, v, k);
            v = MAX ? fmax(v, o) : v + o;
        }
        if (lane == 0) sh[LAP_THREADS / 32] = v;
    }
    __syncthreads();
    return sh[LAP_THREADS / 32];
}

// Laplace importance sampling, summary: one block per curve of the chunk.  W (S doubles per curve) holds the log
// weights lw, then exp(lw - max), then their running sums.  The cut a_(S-M-1) comes from the radix select of select.cuh
// on lw (a = lw - max is monotone in lw), the tail (at most M <= 3072 values) is sorted in shared memory, and the
// generalised-Pareto fit spreads its trial b_i over the warps.  Outputs at the curve's chunk index.
__global__ void __launch_bounds__(LAP_THREADS)
multi_laplace_summary_kernel(size_t c0, size_t S, const int* __restrict__ fstat, const double* __restrict__ logpost,
                             const double* __restrict__ logq, double* __restrict__ W, unsigned long long seed,
                             uint32_t curve_offset, int32_t* __restrict__ resample, double* __restrict__ ess,
                             double* __restrict__ khat, int* __restrict__ status) {
    __shared__ double tail[LAP_TAIL_MAX];
    __shared__ double red[LAP_THREADS / 32 + 1];
    __shared__ double gb[128], gl[128], gw[128];
    __shared__ SelectSmem sm;
    __shared__ unsigned ntail;
    const size_t cl = blockIdx.x;
    const int tid = threadIdx.x;
    const double* lp = logpost + cl * S;
    const double* lq = logq + cl * S;
    double* w = W + cl * S;
    int32_t* rs = resample + cl * S;
    auto reject = [&](int st) {
        for (size_t i = tid; i < S; i += LAP_THREADS) rs[i] = -1;
        if (tid == 0) { ess[cl] = 0.0; khat[cl] = NAN; status[cl] = st; }
    };
    if (fstat[cl] != CARMA_LAPLACE_OK) { reject(CARMA_LAPLACE_BAD_COV); return; }
    double mx = -INFINITY;
    for (size_t i = tid; i < S; i += LAP_THREADS) {
        const double a = lp[i];
        const double v = isfinite(a) ? a - lq[i] : -INFINITY;
        w[i] = v;
        mx = fmax(mx, v);
    }
    mx = lap_block_reduce<true>(mx, red);
    if (mx == -INFINITY) { reject(CARMA_LAPLACE_NO_WEIGHT); return; }
    // weight ESS
    double s1 = 0.0, s2 = 0.0;
    for (size_t i = tid; i < S; i += LAP_THREADS) {
        const double e = exp(w[i] - mx);
        s1 += e;
        s2 += e * e;
    }
    s1 = lap_block_reduce<false>(s1, red);
    s2 = lap_block_reduce<false>(s2, red);
    // k-hat
    double kh = INFINITY;
    if (S >= 2) {
        const size_t M = psis_tail_len(S);
        unsigned long long ka, kb;
        block_select_pair(w, S, S - M - 1, sm, &ka, &kb);
        const double cut = fmax(key_value(ka) - mx, LAP_LOG_DBL_MIN), ecut = exp(cut);
        if (tid == 0) ntail = 0;
        __syncthreads();
        for (size_t i = tid; i < S; i += LAP_THREADS) {
            const double a = w[i] - mx;
            if (a > cut) {
                const unsigned k = atomicAdd(&ntail, 1u);
                if (k < LAP_TAIL_MAX) tail[k] = exp(a) - ecut;
            }
        }
        __syncthreads();
        const int n = (int)min(ntail, (unsigned)LAP_TAIL_MAX);
        if (n > 4) {
            int n2 = 1;
            while (n2 < n) n2 <<= 1;
            for (int i = n + tid; i < n2; i += LAP_THREADS) tail[i] = INFINITY;
            __syncthreads();
            for (int k = 2; k <= n2; k <<= 1)   // bitonic sort, ascending
                for (int jj = k >> 1; jj > 0; jj >>= 1) {
                    for (int i = tid; i < n2; i += LAP_THREADS) {
                        const int l = i ^ jj;
                        if (l > i) {
                            const double a = tail[i], b = tail[l];
                            if (((i & k) == 0) == (a > b)) { tail[i] = b; tail[l] = a; }
                        }
                    }
                    __syncthreads();
                }
            const int m = gpd_m(n), wp = tid >> 5, lane = tid & 31;
            for (int i = wp; i < m; i += LAP_THREADS / 32) {   // warp wp: trial b_(i+1)
                const double b = gpd_b(i + 1, m, tail, n);
                double s = 0.0;
                for (int t = lane; t < n; t += 32) s += log1p(-b * tail[t]);
#pragma unroll
                for (int k = 16; k >= 1; k >>= 1) s += __shfl_xor_sync(0xffffffffu, s, k);
                if (lane == 0) { gb[i] = b; gl[i] = gpd_profile(n, b, s / n); }
            }
            __syncthreads();
            for (int i = tid; i < m; i += LAP_THREADS) gw[i] = gpd_weight(i, m, gl);
            __syncthreads();
            const double bbar = gpd_bbar(m, gb, gw);   // every thread, same order
            double s = 0.0;
            for (int t = tid; t < n; t += LAP_THREADS) s += log1p(-bbar * tail[t]);
            s = lap_block_reduce<false>(s, red);
            kh = gpd_khat(n, s / n);
        }
    }
    // systematic resampling: running sums of e over contiguous per-thread ranges, then the ranges' offsets in order
    const size_t per = (S + LAP_THREADS - 1) / LAP_THREADS, i0 = min(S, tid * per), i1 = min(S, i0 + per);
    double part = 0.0;
    for (size_t i = i0; i < i1; i++) {
        const double e = exp(w[i] - mx);
        w[i] = e;
        part += e;
    }
    __syncthreads();
    tail[tid] = part;   // the tail is no longer needed
    __syncthreads();
    if (tid == 0)
        for (int t = 1; t < LAP_THREADS; t++) tail[t] += tail[t - 1];
    __syncthreads();
    double run = tid == 0 ? 0.0 : tail[tid - 1];
    for (size_t i = i0; i < i1; i++) {
        run += w[i];
        w[i] = run;
    }
    __syncthreads();
    const double T = w[S - 1];
    double u0, u1;
    uniforms2(seed, 0u, STREAM_LAPLACE_RESAMPLE, 0u, curve_offset + (uint32_t)(c0 + cl), &u0, &u1);
    for (size_t i = tid; i < S; i += LAP_THREADS) rs[i] = (int32_t)resample_find(w, S, resample_target(i, u0, S, T));
    if (tid == 0) {
        ess[cl] = s1 * s1 / s2;
        khat[cl] = kh;
        status[cl] = CARMA_LAPLACE_OK;
    }
}

// ---- launchers ---------------------------------------------------------------------------------------------------
static bool alike32(const void* a, const void* b) { return (((size_t)a ^ (size_t)b) & 31u) == 0; }

static cudaError_t launch_multi_filter(const carma_multi_series* m, int kind, int p, int q, unsigned flags,
                                       const carma_prior_t* d_priors, const double* d_theta, double* d_mean,
                                       double* d_var, double* d_out, cudaStream_t st) {
    const int d = model_dim(kind, p, q);
    const unsigned grid = (unsigned)((m->ncurves + SF_BLOCK - 1) / SF_BLOCK);
    // block stores need mean / var to sit like the curve arrays within a 32-byte sector; CARMA_MULTI_FILTER_STORES=scalar
    // selects one store per point (kept for comparison; read at every call so both can be timed in one process)
    const char* env = getenv("CARMA_MULTI_FILTER_STORES");
    const bool blk = !(env && !strcmp(env, "scalar")) && alike32(m->d_dt, d_mean) && alike32(m->d_dt, d_var);
#define LAUNCH_SF(PP)                                                                                                  \
    if (blk) multi_filter_kernel<PP, true><<<grid, SF_BLOCK, 0, st>>>(m->d_dt, m->d_y, m->d_e2, m->d_off, m->ncurves,   \
                                                                     m->dt_max, kind, q, d, flags, d_priors, d_theta,  \
                                                                     d_mean, d_var, d_out);                            \
    else multi_filter_kernel<PP, false><<<grid, SF_BLOCK, 0, st>>>(m->d_dt, m->d_y, m->d_e2, m->d_off, m->ncurves,      \
                                                                  m->dt_max, kind, q, d, flags, d_priors, d_theta,     \
                                                                  d_mean, d_var, d_out)
    switch (p) {
        case 1: LAUNCH_SF(1); break;
        case 2: LAUNCH_SF(2); break;
        case 3: LAUNCH_SF(3); break;
        case 4: LAUNCH_SF(4); break;
        case 5: LAUNCH_SF(5); break;
        case 6: LAUNCH_SF(6); break;
        case 7: LAUNCH_SF(7); break;
        default: return cudaErrorInvalidValue;
    }
#undef LAUNCH_SF
    return cudaGetLastError();
}

template <int P, bool PATHS>
static cudaError_t launch_predict_p(const carma_multi_series* m, int kind, int q, unsigned flags, double dt_max,
                                    const carma_prior_t* d_priors, const double* d_theta, const double* d_y,
                                    const PathSet& ps, const long long* d_qoff, const double* d_qtq, const int* d_qcurve,
                                    const long long* d_perm, size_t nq, double* d_rec, void* d_prm, int* d_status,
                                    double* d_qm, double* d_qv, cudaStream_t st) {
    const int d = model_dim(kind, P, q);
    predict_forward_kernel<P, PATHS><<<(unsigned)((m->ncurves * ps.B + SF_BLOCK - 1) / SF_BLOCK), SF_BLOCK, 0, st>>>(
        m->d_dt, d_y, m->d_e2, m->d_off, m->ncurves, dt_max, kind, q, d, flags, d_priors, d_theta, d_qoff, d_qtq, ps,
        d_rec, (RealParams<P>*)d_prm, d_status);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    predict_query_kernel<P, PATHS><<<(unsigned)((nq * ps.B + SF_BLOCK - 1) / SF_BLOCK), SF_BLOCK, 0, st>>>(
        m->d_dt, d_y, m->d_e2, m->d_off, d_qcurve, d_perm, nq, ps, d_rec, (const RealParams<P>*)d_prm, d_status, d_qm,
        d_qv);
    return cudaGetLastError();
}

// one chunk of conditional-simulation paths: prior draws, then the predict kernels on their residual data
template <int P>
static cudaError_t launch_simulate_p(const carma_multi_series* m, int kind, int q, unsigned flags, double dt_max,
                                     const carma_prior_t* d_priors, const double* d_theta, const PathSet& ps,
                                     unsigned long long seed, uint32_t curve_offset, const long long* d_qoff,
                                     const double* d_qtq, const int* d_qcurve, const long long* d_perm, size_t nq,
                                     double* d_yres, double* d_rec, void* d_prm, int* d_status, double* d_out,
                                     cudaStream_t st) {
    const int d = model_dim(kind, P, q);
    condsim_prior_kernel<P><<<(unsigned)((m->ncurves * ps.B + SF_BLOCK - 1) / SF_BLOCK), SF_BLOCK, 0, st>>>(
        m->d_dt, m->d_y, m->d_e2, m->d_off, m->ncurves, dt_max, kind, q, d, flags, d_priors, d_theta, d_qoff, d_qtq,
        d_perm, nq, ps, seed, curve_offset, d_yres, d_out);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    return launch_predict_p<P, true>(m, kind, q, flags, dt_max, d_priors, d_theta, d_yres, ps, d_qoff, d_qtq, d_qcurve, d_perm,
                               nq, d_rec, d_prm, d_status, d_out, nullptr, st);
}

// upload the priors (NULL: the population-variance defaults) and `rows` theta rows into the multi-series' scratch
static int upload_rows(carma_multi_series* m, int kind, int p, int q, const carma_prior_t* priors, const double* theta,
                       size_t rows, cudaStream_t st) {
    const size_t d = (size_t)model_dim(kind, p, q), n = m->ncurves;
    if (!m->scratch_in.reserve(rows * d * sizeof(double)) || !m->scratch_pr.reserve(n * sizeof(carma_prior_t)))
        return CARMA_ERR_CUDA;
    const carma_prior_t* hp = priors ? priors : m->priors_pop.data();
    if (!cuda_ok(cudaMemcpyAsync(m->scratch_pr.p, hp, n * sizeof(carma_prior_t), cudaMemcpyHostToDevice, st), "H2D priors") ||
        !cuda_ok(cudaMemcpyAsync(m->scratch_in.p, theta, rows * d * sizeof(double), cudaMemcpyHostToDevice, st), "H2D theta"))
        return CARMA_ERR_CUDA;
    return CARMA_OK;
}

// Sort every curve's queries by time, on the curve's own axis (t - t0[c]): perm[k] is the caller's position of sorted
// query k, qtq its time on the axis, qcurve its curve.  Returns the rate clamp of the call, which must cover its longest
// transition: the data gaps, forecasts past the last point and backcasts before the first.
static double sort_queries(const carma_multi_series* m, const int64_t* q_offsets, const double* tq,
                           std::vector<long long>& perm, std::vector<double>& qtq, std::vector<int>& qcurve) {
    const size_t nc = m->ncurves, nq = (size_t)q_offsets[nc];
    perm.resize(nq);
    qtq.resize(nq);
    qcurve.resize(nq);
    double dt_max = m->dt_max;
    for (size_t c = 0; c < nc; c++) {
        const size_t k0 = (size_t)q_offsets[c], k1 = (size_t)q_offsets[c + 1];
        std::iota(perm.begin() + k0, perm.begin() + k1, (long long)k0);
        std::stable_sort(perm.begin() + k0, perm.begin() + k1, [&](long long a, long long b) { return tq[a] < tq[b]; });
        const double tspan = m->info[c].tspan;
        for (size_t k = k0; k < k1; k++) {
            qtq[k] = tq[perm[k]] - m->t0[c];
            qcurve[k] = (int)c;
            dt_max = std::max(dt_max, std::max(qtq[k] - tspan, -qtq[k]));
        }
    }
    return dt_max;
}

static size_t round32(size_t n) { return (n + 31) & ~(size_t)31; }   // doubles: keeps 256-byte alignment

template <int P>
static cudaError_t launch_smooth_p(const carma_multi_series* m, int kind, int q, unsigned flags, double dt_max,
                                   const carma_prior_t* d_priors, const double* d_theta, const long long* d_qoff,
                                   const double* d_qtq, const long long* d_perm, const SmoothChunk& ch, double* d_rp,
                                   double* d_rq, double* const* d_pt, double* d_ll, double* d_qm, double* d_qv,
                                   cudaStream_t st) {
    multi_smooth_kernel<P><<<(unsigned)((ch.nc + SF_BLOCK - 1) / SF_BLOCK), SF_BLOCK, 0, st>>>(
        m->d_dt, m->d_y, m->d_e2, m->d_off, ch, dt_max, kind, q, model_dim(kind, P, q), flags, d_priors, d_theta, d_qoff,
        d_qtq, d_perm, d_rp, d_rq, d_pt[0], d_pt[1], d_pt[2], d_pt[3], d_ll, d_qm, d_qv);
    return cudaGetLastError();
}

template <int P>
static cudaError_t launch_hessian_eval_p(const carma_multi_series* m, int kind, int q, unsigned flags,
                                         const carma_prior_t* d_priors, const double* d_theta, double rel_step,
                                         size_t c0, size_t nc, double* d_f, cudaStream_t st) {
    const int d = model_dim(kind, P, q), npts = hess_points(d);
    multi_hessian_eval_kernel<P><<<(unsigned)((nc * npts + SF_BLOCK - 1) / SF_BLOCK), SF_BLOCK, 0, st>>>(
        m->d_dt, m->d_y, m->d_e2, m->d_off, c0, nc, npts, m->dt_max, kind, q, d, flags, d_priors, d_theta, rel_step, d_f);
    return cudaGetLastError();
}

// one chunk of carma_multi_laplace's draws: curves c0 .. c0 + nc - 1, S draws each
struct LaplaceChunk {
    double *L, *logdet, *w, *draws, *logpost, *logq, *ess, *khat;
    int *fstat, *status;
    int32_t* resample;
};

template <int P>
static cudaError_t launch_laplace_eval_p(const carma_multi_series* m, int kind, int q, unsigned flags,
                                         const carma_prior_t* d_priors, const double* d_theta, size_t c0, size_t nc,
                                         size_t S, unsigned long long seed, uint32_t curve_offset, const LaplaceChunk& ch,
                                         cudaStream_t st) {
    multi_laplace_eval_kernel<P><<<(unsigned)((nc * S + SF_BLOCK - 1) / SF_BLOCK), SF_BLOCK, 0, st>>>(
        m->d_dt, m->d_y, m->d_e2, m->d_off, c0, nc, S, m->dt_max, kind, q, model_dim(kind, P, q), flags, d_priors,
        d_theta, ch.L, ch.logdet, ch.fstat, seed, curve_offset, ch.draws, ch.logpost, ch.logq);
    return cudaGetLastError();
}

}  // namespace carma

using namespace carma;

extern "C" {

int carma_multi_filter_dev(carma_multi_series_t m, int kind, int p, int q, const carma_prior_t* d_priors,
                           const double* d_theta, unsigned flags, double* d_mean, double* d_var, double* d_loglik,
                           void* stream) {
    if (!m || !d_priors || !d_theta || !d_mean || !d_var) { set_error("carma_multi_filter_dev: null argument"); return CARMA_ERR_ARG; }
    if (!valid_model(kind, p, q)) { set_error("carma_multi_filter_dev: invalid (kind,p,q)"); return CARMA_ERR_ARG; }
    if (!alike32(m->d_dt, m->d_y) || !alike32(m->d_dt, m->d_e2)) { set_error("carma_multi_filter_dev: curve arrays not sector-aligned"); return CARMA_ERR_ARG; }
    if (!cuda_ok(launch_multi_filter(m, kind, p, q, flags, d_priors, d_theta, d_mean, d_var, d_loglik, (cudaStream_t)stream),
                 "multi_filter_kernel launch"))
        return CARMA_ERR_CUDA;
    return CARMA_OK;
}

// the filter of every curve into the multi-series' scratch: mean at scratch_pts, var behind it, loglik in scratch_out
static int multi_filter_to_scratch(carma_multi_series* m, int kind, int p, int q, const carma_prior_t* priors,
                                   const double* theta, unsigned flags, cudaStream_t st, double** d_mean, double** d_var) {
    if (!cuda_ok(cudaSetDevice(m->device), "cudaSetDevice")) return CARMA_ERR_CUDA;
    const size_t stride = round32(m->total);
    if (!m->scratch_pts.reserve(2 * stride * sizeof(double)) || !m->scratch_out.reserve(m->ncurves * sizeof(double)))
        return CARMA_ERR_CUDA;
    int rc = upload_rows(m, kind, p, q, priors, theta, m->ncurves, st);
    if (rc) return rc;
    *d_mean = (double*)m->scratch_pts.p;
    *d_var = *d_mean + stride;
    return carma_multi_filter_dev(m, kind, p, q, (const carma_prior_t*)m->scratch_pr.p, (const double*)m->scratch_in.p,
                                  flags, *d_mean, *d_var, (double*)m->scratch_out.p, st);
}

int carma_multi_filter(carma_multi_series_t m, int kind, int p, int q, const carma_prior_t* priors, const double* theta,
                       unsigned flags, double* mean, double* var, double* loglik) {
    if (!m || !theta || !mean || !var) { set_error("carma_multi_filter: null argument"); return CARMA_ERR_ARG; }
    if (!valid_model(kind, p, q)) { set_error("carma_multi_filter: invalid (kind,p,q)"); return CARMA_ERR_ARG; }
    cudaStream_t st = 0;
    double *d_mean = nullptr, *d_var = nullptr;
    int rc = multi_filter_to_scratch(m, kind, p, q, priors, theta, flags, st, &d_mean, &d_var);
    if (rc) return rc;
    const size_t n = m->total;
    if (!cuda_ok(cudaMemcpyAsync(mean, d_mean, n * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H mean") ||
        !cuda_ok(cudaMemcpyAsync(var, d_var, n * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H var"))
        return CARMA_ERR_CUDA;
    if (loglik && !cuda_ok(cudaMemcpyAsync(loglik, m->scratch_out.p, m->ncurves * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H loglik"))
        return CARMA_ERR_CUDA;
    if (!cuda_ok(cudaStreamSynchronize(st), "multi_filter sync")) return CARMA_ERR_CUDA;
    return CARMA_OK;
}

int carma_multi_assess_fit(carma_multi_series_t m, int kind, int p, int q, const carma_prior_t* priors,
                           const double* theta, unsigned flags, int nlags, double* out) {
    if (nlags < 1) { set_error("carma_multi_assess_fit: nlags must be >= 1"); return CARMA_ERR_ARG; }
    if (!m || !theta || !out) { set_error("carma_multi_assess_fit: null argument"); return CARMA_ERR_ARG; }
    if (!valid_model(kind, p, q)) { set_error("carma_multi_assess_fit: invalid (kind,p,q)"); return CARMA_ERR_ARG; }
    long long min_ny = m->off[1] - m->off[0];
    for (size_t c = 1; c < m->ncurves; c++) min_ny = std::min(min_ny, m->off[c + 1] - m->off[c]);
    if ((long long)nlags >= min_ny) {
        set_error("carma_multi_assess_fit: nlags must be below the shortest curve's length (" + std::to_string(min_ny) + ")");
        return CARMA_ERR_ARG;
    }
    cudaStream_t st = 0;
    double *d_mean = nullptr, *d_var = nullptr;
    int rc = multi_filter_to_scratch(m, kind, p, q, priors, theta, flags, st, &d_mean, &d_var);
    if (rc) return rc;
    const size_t w = 3 + 2 * (size_t)nlags, n = m->ncurves;
    if (!m->scratch_misc.reserve(n * w * sizeof(double))) return CARMA_ERR_CUDA;
    const unsigned grid = (unsigned)((n * 32 + ACF_BLOCK - 1) / ACF_BLOCK);
    residual_acf_kernel<<<grid, ACF_BLOCK, 0, st>>>(m->d_y, m->d_off, n, (const double*)m->scratch_in.p,
                                                    model_dim(kind, p, q), (const double*)m->scratch_out.p, d_mean,
                                                    d_var, nlags, (double*)m->scratch_misc.p);
    if (!cuda_ok(cudaGetLastError(), "residual_acf_kernel launch")) return CARMA_ERR_CUDA;
    if (!cuda_ok(cudaMemcpyAsync(out, m->scratch_misc.p, n * w * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H assess_fit") ||
        !cuda_ok(cudaStreamSynchronize(st), "multi_assess_fit sync"))
        return CARMA_ERR_CUDA;
    return CARMA_OK;
}

int carma_multi_predict(carma_multi_series_t m, int kind, int p, int q, const carma_prior_t* priors,
                        const double* theta, unsigned flags, const int64_t* q_offsets, const double* tq, double* qmean,
                        double* qvar) {
    if (q_offsets && q_offsets[0] != 0) { set_error("carma_multi_predict: q_offsets must start at 0"); return CARMA_ERR_ARG; }
    if (!m || !theta || !q_offsets) { set_error("carma_multi_predict: null argument"); return CARMA_ERR_ARG; }
    if (!valid_model(kind, p, q)) { set_error("carma_multi_predict: invalid (kind,p,q)"); return CARMA_ERR_ARG; }
    const size_t nc = m->ncurves;
    for (size_t c = 0; c < nc; c++)
        if (q_offsets[c + 1] < q_offsets[c]) { set_error("carma_multi_predict: q_offsets must be non-decreasing"); return CARMA_ERR_ARG; }
    const size_t nq = (size_t)q_offsets[nc];
    if (nq == 0) return CARMA_OK;
    if (!tq || !qmean || !qvar) { set_error("carma_multi_predict: null argument"); return CARMA_ERR_ARG; }
    for (size_t k = 0; k < nq; k++)
        if (!std::isfinite(tq[k])) { set_error("carma_multi_predict: non-finite query time"); return CARMA_ERR_ARG; }
    std::vector<long long> perm;
    std::vector<double> qtq;
    std::vector<int> qcurve;
    const double dt_max = sort_queries(m, q_offsets, tq, perm, qtq, qcurve);
    if (!cuda_ok(cudaSetDevice(m->device), "cudaSetDevice")) return CARMA_ERR_CUDA;
    cudaStream_t st = 0;
    int rc = upload_rows(m, kind, p, q, priors, theta, nc, st);
    if (rc) return rc;
    // scratch_q: records | qtq | qm | qv | perm | qoff | prm | status | qcurve, each on a 256-byte boundary
    const size_t R = (size_t)(p + p * (p + 1) / 2 + 3);
    const size_t b_rec = round32(nq * R), b_q = round32(nq), b_off = round32(nc + 1),
                 b_prm = round32((nc * sizeof(RealParams<MAX_P>) + 7) / 8), b_st = round32((nc + 1) / 2), b_qc = round32((nq + 1) / 2);
    if (!m->scratch_q.reserve((b_rec + 4 * b_q + b_off + b_prm + b_st + b_qc) * sizeof(double))) return CARMA_ERR_CUDA;
    double* d_rec = (double*)m->scratch_q.p;
    double* d_qtq = d_rec + b_rec;
    double* d_qm = d_qtq + b_q;
    double* d_qv = d_qm + b_q;
    long long* d_perm = (long long*)(d_qv + b_q);
    long long* d_qoff = (long long*)((double*)d_perm + b_q);
    void* d_prm = (double*)d_qoff + b_off;
    int* d_status = (int*)((double*)d_prm + b_prm);
    int* d_qcurve = (int*)((double*)d_status + b_st);
    bool ok = cuda_ok(cudaMemcpyAsync(d_qtq, qtq.data(), nq * sizeof(double), cudaMemcpyHostToDevice, st), "H2D tq") &&
              cuda_ok(cudaMemcpyAsync(d_perm, perm.data(), nq * sizeof(long long), cudaMemcpyHostToDevice, st), "H2D perm") &&
              cuda_ok(cudaMemcpyAsync(d_qoff, q_offsets, (nc + 1) * sizeof(long long), cudaMemcpyHostToDevice, st), "H2D q_offsets") &&
              cuda_ok(cudaMemcpyAsync(d_qcurve, qcurve.data(), nq * sizeof(int), cudaMemcpyHostToDevice, st), "H2D qcurve");
    if (!ok) return CARMA_ERR_CUDA;
    const carma_prior_t* d_pr = (const carma_prior_t*)m->scratch_pr.p;
    const double* d_th = (const double*)m->scratch_in.p;
    cudaError_t e;
#define LAUNCH_PQ(PP) e = launch_predict_p<PP, false>(m, kind, q, flags, dt_max, d_pr, d_th, m->d_y, PathSet{}, d_qoff, d_qtq, \
                                                d_qcurve, d_perm, nq, d_rec, d_prm, d_status, d_qm, d_qv, st)
    switch (p) {
        case 1: LAUNCH_PQ(1); break;
        case 2: LAUNCH_PQ(2); break;
        case 3: LAUNCH_PQ(3); break;
        case 4: LAUNCH_PQ(4); break;
        case 5: LAUNCH_PQ(5); break;
        case 6: LAUNCH_PQ(6); break;
        default: LAUNCH_PQ(7); break;
    }
#undef LAUNCH_PQ
    if (!cuda_ok(e, "predict kernels launch")) return CARMA_ERR_CUDA;
    if (!cuda_ok(cudaMemcpyAsync(qmean, d_qm, nq * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H qmean") ||
        !cuda_ok(cudaMemcpyAsync(qvar, d_qv, nq * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H qvar") ||
        !cuda_ok(cudaStreamSynchronize(st), "multi_predict sync"))
        return CARMA_ERR_CUDA;
    return CARMA_OK;
}

int carma_multi_simulate(carma_multi_series_t m, int kind, int p, int q, const carma_prior_t* priors,
                         const double* theta, size_t theta_rows, unsigned flags, const int64_t* s_offsets,
                         const double* tsim, size_t npaths, uint64_t seed, uint32_t curve_offset, double* ysim) {
    if (s_offsets && s_offsets[0] != 0) { set_error("carma_multi_simulate: s_offsets must start at 0"); return CARMA_ERR_ARG; }
    if (!m || !theta || !s_offsets) { set_error("carma_multi_simulate: null argument"); return CARMA_ERR_ARG; }
    if (!valid_model(kind, p, q)) { set_error("carma_multi_simulate: invalid (kind,p,q)"); return CARMA_ERR_ARG; }
    const size_t nc = m->ncurves;
    for (size_t c = 0; c < nc; c++)
        if (s_offsets[c + 1] < s_offsets[c]) { set_error("carma_multi_simulate: s_offsets must be non-decreasing"); return CARMA_ERR_ARG; }
    const size_t nq = (size_t)s_offsets[nc];
    if (npaths == 0 || nq == 0) return CARMA_OK;
    if (!tsim || !ysim) { set_error("carma_multi_simulate: null argument"); return CARMA_ERR_ARG; }
    if (theta_rows != nc && theta_rows != nc * npaths) {
        set_error("carma_multi_simulate: theta_rows must be ncurves or ncurves * npaths");
        return CARMA_ERR_ARG;
    }
    if ((uint64_t)curve_offset + nc > ((uint64_t)1 << 32) || (uint64_t)npaths > ((uint64_t)1 << 32)) {
        set_error("carma_multi_simulate: curve_offset + ncurves and npaths must not exceed 2^32 (32-bit Philox counters)");
        return CARMA_ERR_ARG;
    }
    for (size_t k = 0; k < nq; k++)
        if (!std::isfinite(tsim[k])) { set_error("carma_multi_simulate: non-finite time"); return CARMA_ERR_ARG; }
    std::vector<long long> perm;
    std::vector<double> qtq;
    std::vector<int> qcurve;
    const double dt_max = sort_queries(m, s_offsets, tsim, perm, qtq, qcurve);
    if (!cuda_ok(cudaSetDevice(m->device), "cudaSetDevice")) return CARMA_ERR_CUDA;
    cudaStream_t st = 0;
    int rc = upload_rows(m, kind, p, q, priors, theta, theta_rows, st);
    if (rc) return rc;
    // Paths go in chunks of B whose scratch fits the budget (CARMA_MULTI_SIMULATE_BUDGET bytes, read at every call so
    // that a test can force several chunks): per path a residual-data row, the query records, the output row and the
    // constants of every curve.  A draw depends only on its curve, path and theta row, so chunking changes no bit.
    const size_t R = (size_t)(p + p * (p + 1) / 2 + 3), ystride = round32(m->total);
    const size_t prm_d = (sizeof(RealParams<MAX_P>) + 7) / 8;
    const size_t per_path = ystride + nq * (R + 1) + nc * (prm_d + 1);
    size_t budget = (size_t)4 << 30;
    if (const char* env = getenv("CARMA_MULTI_SIMULATE_BUDGET")) budget = (size_t)std::strtoull(env, nullptr, 10);
    const size_t B = std::max<size_t>(1, std::min(npaths, budget / (per_path * sizeof(double))));
    // scratch_pts: B residual-data rows; scratch_q: records | out | qtq | perm | qoff | prm | status | qcurve
    const size_t b_rec = round32(nq * B * R), b_out = round32(nq * B), b_q = round32(nq), b_off = round32(nc + 1),
                 b_prm = round32(nc * B * prm_d), b_st = round32((nc * B + 1) / 2), b_qc = round32((nq + 1) / 2);
    if (!m->scratch_pts.reserve(B * ystride * sizeof(double)) ||
        !m->scratch_q.reserve((b_rec + b_out + 2 * b_q + b_off + b_prm + b_st + b_qc) * sizeof(double)))
        return CARMA_ERR_CUDA;
    double* d_yres = (double*)m->scratch_pts.p;
    double* d_rec = (double*)m->scratch_q.p;
    double* d_out = d_rec + b_rec;
    double* d_qtq = d_out + b_out;
    long long* d_perm = (long long*)(d_qtq + b_q);
    long long* d_qoff = (long long*)((double*)d_perm + b_q);
    void* d_prm = (double*)d_qoff + b_off;
    int* d_status = (int*)((double*)d_prm + b_prm);
    int* d_qcurve = (int*)((double*)d_status + b_st);
    bool ok = cuda_ok(cudaMemcpyAsync(d_qtq, qtq.data(), nq * sizeof(double), cudaMemcpyHostToDevice, st), "H2D tsim") &&
              cuda_ok(cudaMemcpyAsync(d_perm, perm.data(), nq * sizeof(long long), cudaMemcpyHostToDevice, st), "H2D perm") &&
              cuda_ok(cudaMemcpyAsync(d_qoff, s_offsets, (nc + 1) * sizeof(long long), cudaMemcpyHostToDevice, st), "H2D s_offsets") &&
              cuda_ok(cudaMemcpyAsync(d_qcurve, qcurve.data(), nq * sizeof(int), cudaMemcpyHostToDevice, st), "H2D qcurve");
    if (!ok) return CARMA_ERR_CUDA;
    const carma_prior_t* d_pr = (const carma_prior_t*)m->scratch_pr.p;
    const double* d_th = (const double*)m->scratch_in.p;
    for (size_t j0 = 0; j0 < npaths; j0 += B) {
        PathSet ps;
        ps.B = (unsigned)std::min(B, npaths - j0);
        ps.j0 = (unsigned)j0;
        ps.ystride = ystride;
        ps.rpc = theta_rows / nc;
        cudaError_t e;
#define LAUNCH_SIM(PP) e = launch_simulate_p<PP>(m, kind, q, flags, dt_max, d_pr, d_th, ps, seed, curve_offset, d_qoff, d_qtq, \
                                                 d_qcurve, d_perm, nq, d_yres, d_rec, d_prm, d_status, d_out, st)
        switch (p) {
            case 1: LAUNCH_SIM(1); break;
            case 2: LAUNCH_SIM(2); break;
            case 3: LAUNCH_SIM(3); break;
            case 4: LAUNCH_SIM(4); break;
            case 5: LAUNCH_SIM(5); break;
            case 6: LAUNCH_SIM(6); break;
            default: LAUNCH_SIM(7); break;
        }
#undef LAUNCH_SIM
        if (!cuda_ok(e, "simulate kernels launch")) return CARMA_ERR_CUDA;
        if (!cuda_ok(cudaMemcpyAsync(ysim + j0 * nq, d_out, ps.B * nq * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H ysim"))
            return CARMA_ERR_CUDA;
    }
    if (!cuda_ok(cudaStreamSynchronize(st), "multi_simulate sync")) return CARMA_ERR_CUDA;
    return CARMA_OK;
}

int carma_multi_smooth(carma_multi_series_t m, int kind, int p, int q, const carma_prior_t* priors, const double* theta,
                       unsigned flags, double* mean, double* var, double* loo_mean, double* loo_var, double* loglik,
                       const int64_t* q_offsets, const double* tq, double* qmean, double* qvar) {
    if (q_offsets && q_offsets[0] != 0) { set_error("carma_multi_smooth: q_offsets must start at 0"); return CARMA_ERR_ARG; }
    if (!m || !theta) { set_error("carma_multi_smooth: null argument"); return CARMA_ERR_ARG; }
    if (!valid_model(kind, p, q)) { set_error("carma_multi_smooth: invalid (kind,p,q)"); return CARMA_ERR_ARG; }
    const size_t nc = m->ncurves;
    std::vector<int64_t> no_queries;
    if (!q_offsets) {
        no_queries.assign(nc + 1, 0);
        q_offsets = no_queries.data();
    }
    for (size_t c = 0; c < nc; c++)
        if (q_offsets[c + 1] < q_offsets[c]) { set_error("carma_multi_smooth: q_offsets must be non-decreasing"); return CARMA_ERR_ARG; }
    const size_t nq = (size_t)q_offsets[nc];
    if (nq > 0 && !tq) { set_error("carma_multi_smooth: null argument (tq)"); return CARMA_ERR_ARG; }
    for (size_t k = 0; k < nq; k++)
        if (!std::isfinite(tq[k])) { set_error("carma_multi_smooth: non-finite query time"); return CARMA_ERR_ARG; }
    std::vector<long long> perm;
    std::vector<double> qtq;
    std::vector<int> qcurve;
    const double dt_max = sort_queries(m, q_offsets, tq, perm, qtq, qcurve);
    if (!cuda_ok(cudaSetDevice(m->device), "cudaSetDevice")) return CARMA_ERR_CUDA;
    cudaStream_t st = 0;
    int rc = upload_rows(m, kind, p, q, priors, theta, nc, st);
    if (rc) return rc;
    // Curves go in chunks whose records fit the budget (CARMA_MULTI_SMOOTH_BUDGET bytes, read at every call so that a
    // test can force several chunks).  Every output depends only on its curve, so chunking changes no bit.
    const size_t PF = (size_t)p + 2, QF = (size_t)p + 3;
    size_t budget = (size_t)4 << 30;
    if (const char* env = getenv("CARMA_MULTI_SMOOTH_BUDGET")) budget = (size_t)std::strtoull(env, nullptr, 10);
    std::vector<SmoothChunk> chunks;
    size_t rec_max = 0;   // doubles of the largest chunk's records
    for (size_t c = 0; c < nc;) {
        SmoothChunk ch;
        ch.c0 = c;
        ch.pbase = m->off[c] & ~3ll;
        ch.qbase = q_offsets[c];
        size_t need = 0;
        for (size_t e = c + 1; e <= nc; e++) {
            const size_t ps = round32((size_t)(m->off[e] - ch.pbase)), qs = round32((size_t)(q_offsets[e] - ch.qbase));
            const size_t n = PF * ps + QF * qs;
            if (e > c + 1 && n * sizeof(double) > budget) break;
            ch.nc = e - c;
            ch.pstride = ps;
            ch.qstride = qs;
            need = n;
        }
        rec_max = std::max(rec_max, need);
        chunks.push_back(ch);
        c += ch.nc;
    }
    // scratch_pts: mean | var | loo_mean | loo_var (total each); scratch_misc: one chunk's point and query records;
    // scratch_q: qm | qv | qtq | perm | qoff; scratch_out: loglik
    const size_t b_pt = round32(m->total), b_q = round32(nq), b_off = round32(nc + 1);
    if (!m->scratch_pts.reserve(4 * b_pt * sizeof(double)) || !m->scratch_misc.reserve(std::max<size_t>(rec_max, 1) * sizeof(double)) ||
        !m->scratch_q.reserve((4 * b_q + b_off) * sizeof(double)) || !m->scratch_out.reserve(nc * sizeof(double)))
        return CARMA_ERR_CUDA;
    double* d_pt[4];
    for (int j = 0; j < 4; j++) d_pt[j] = (double*)m->scratch_pts.p + j * b_pt;
    double* d_qm = (double*)m->scratch_q.p;
    double* d_qv = d_qm + b_q;
    double* d_qtq = d_qv + b_q;
    long long* d_perm = (long long*)(d_qtq + b_q);
    long long* d_qoff = (long long*)((double*)d_perm + b_q);
    double* d_ll = (double*)m->scratch_out.p;
    bool ok = cuda_ok(cudaMemcpyAsync(d_qoff, q_offsets, (nc + 1) * sizeof(long long), cudaMemcpyHostToDevice, st), "H2D q_offsets");
    if (ok && nq > 0)
        ok = cuda_ok(cudaMemcpyAsync(d_qtq, qtq.data(), nq * sizeof(double), cudaMemcpyHostToDevice, st), "H2D tq") &&
             cuda_ok(cudaMemcpyAsync(d_perm, perm.data(), nq * sizeof(long long), cudaMemcpyHostToDevice, st), "H2D perm");
    if (!ok) return CARMA_ERR_CUDA;
    const carma_prior_t* d_pr = (const carma_prior_t*)m->scratch_pr.p;
    const double* d_th = (const double*)m->scratch_in.p;
    for (const SmoothChunk& ch : chunks) {
        double* d_rp = (double*)m->scratch_misc.p;
        double* d_rq = d_rp + PF * ch.pstride;
        cudaError_t e;
#define LAUNCH_SM(PP) e = launch_smooth_p<PP>(m, kind, q, flags, dt_max, d_pr, d_th, d_qoff, d_qtq, d_perm, ch, d_rp, d_rq, \
                                              d_pt, d_ll, d_qm, d_qv, st)
        switch (p) {
            case 1: LAUNCH_SM(1); break;
            case 2: LAUNCH_SM(2); break;
            case 3: LAUNCH_SM(3); break;
            case 4: LAUNCH_SM(4); break;
            case 5: LAUNCH_SM(5); break;
            case 6: LAUNCH_SM(6); break;
            default: LAUNCH_SM(7); break;
        }
#undef LAUNCH_SM
        if (!cuda_ok(e, "multi_smooth_kernel launch")) return CARMA_ERR_CUDA;
    }
    double* const host_pt[4] = {mean, var, loo_mean, loo_var};
    const char* what[4] = {"D2H mean", "D2H var", "D2H loo_mean", "D2H loo_var"};
    for (int j = 0; j < 4; j++)
        if (host_pt[j] && !cuda_ok(cudaMemcpyAsync(host_pt[j], d_pt[j], m->total * sizeof(double), cudaMemcpyDeviceToHost, st), what[j]))
            return CARMA_ERR_CUDA;
    if (loglik && !cuda_ok(cudaMemcpyAsync(loglik, d_ll, nc * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H loglik"))
        return CARMA_ERR_CUDA;
    if (nq > 0 && qmean && !cuda_ok(cudaMemcpyAsync(qmean, d_qm, nq * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H qmean"))
        return CARMA_ERR_CUDA;
    if (nq > 0 && qvar && !cuda_ok(cudaMemcpyAsync(qvar, d_qv, nq * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H qvar"))
        return CARMA_ERR_CUDA;
    if (!cuda_ok(cudaStreamSynchronize(st), "multi_smooth sync")) return CARMA_ERR_CUDA;
    return CARMA_OK;
}

int carma_multi_hessian(carma_multi_series_t m, int kind, int p, int q, const carma_prior_t* priors, const double* theta,
                        unsigned flags, double rel_step, double* loglik, double* grad, double* hess, double* cov,
                        int* status) {
    if (!std::isfinite(rel_step)) { set_error("carma_multi_hessian: rel_step must be finite"); return CARMA_ERR_ARG; }
    if (!valid_model(kind, p, q)) { set_error("carma_multi_hessian: invalid (kind,p,q)"); return CARMA_ERR_ARG; }
    if (!m || !theta) { set_error("carma_multi_hessian: null argument"); return CARMA_ERR_ARG; }
    if (rel_step <= 0.0) rel_step = CARMA_HESS_DEFAULT_REL_STEP;
    if (!alike32(m->d_dt, m->d_y) || !alike32(m->d_dt, m->d_e2)) { set_error("carma_multi_hessian: curve arrays not sector-aligned"); return CARMA_ERR_ARG; }
    const size_t nc = m->ncurves, d = (size_t)model_dim(kind, p, q), npts = (size_t)hess_points((int)d);
    if (!cuda_ok(cudaSetDevice(m->device), "cudaSetDevice")) return CARMA_ERR_CUDA;
    cudaStream_t st = 0;
    int rc = upload_rows(m, kind, p, q, priors, theta, nc, st);
    if (rc) return rc;
    // Curves go in chunks of B whose stencil values fit the budget (CARMA_MULTI_HESSIAN_BUDGET bytes, read at every call
    // so that a test can force several chunks).  Every output depends only on its curve, so chunking changes no bit.
    size_t budget = (size_t)4 << 30;
    if (const char* env = getenv("CARMA_MULTI_HESSIAN_BUDGET")) budget = (size_t)std::strtoull(env, nullptr, 10);
    const size_t B = std::max<size_t>(1, std::min(nc, budget / (npts * sizeof(double))));
    // scratch_misc: one chunk's stencil values; scratch_pts: loglik | grad | hess | cov | status
    const size_t b_ll = round32(nc), b_g = round32(nc * d), b_h = round32(nc * d * d), b_st = round32((nc + 1) / 2);
    if (!m->scratch_misc.reserve(B * npts * sizeof(double)) ||
        !m->scratch_pts.reserve((b_ll + b_g + 2 * b_h + b_st) * sizeof(double)))
        return CARMA_ERR_CUDA;
    double* d_f = (double*)m->scratch_misc.p;
    double* d_ll = (double*)m->scratch_pts.p;
    double* d_g = d_ll + b_ll;
    double* d_h = d_g + b_g;
    double* d_cov = d_h + b_h;
    int* d_st = (int*)(d_cov + b_h);
    const carma_prior_t* d_pr = (const carma_prior_t*)m->scratch_pr.p;
    const double* d_th = (const double*)m->scratch_in.p;
    for (size_t c0 = 0; c0 < nc; c0 += B) {
        const size_t n = std::min(B, nc - c0);
        cudaError_t e;
#define LAUNCH_HE(PP) e = launch_hessian_eval_p<PP>(m, kind, q, flags, d_pr, d_th, rel_step, c0, n, d_f, st)
        switch (p) {
            case 1: LAUNCH_HE(1); break;
            case 2: LAUNCH_HE(2); break;
            case 3: LAUNCH_HE(3); break;
            case 4: LAUNCH_HE(4); break;
            case 5: LAUNCH_HE(5); break;
            case 6: LAUNCH_HE(6); break;
            default: LAUNCH_HE(7); break;
        }
#undef LAUNCH_HE
        if (!cuda_ok(e, "multi_hessian_eval_kernel launch")) return CARMA_ERR_CUDA;
        multi_hessian_assemble_kernel<<<(unsigned)((n + SF_BLOCK - 1) / SF_BLOCK), SF_BLOCK, 0, st>>>(
            d_f, c0, n, (int)d, d_th, rel_step, d_ll, d_g, d_h, d_cov, d_st);
        if (!cuda_ok(cudaGetLastError(), "multi_hessian_assemble_kernel launch")) return CARMA_ERR_CUDA;
    }
    struct Out { void* host; const void* dev; size_t bytes; const char* what; };
    const Out outs[5] = {{loglik, d_ll, nc * sizeof(double), "D2H loglik"}, {grad, d_g, nc * d * sizeof(double), "D2H grad"},
                         {hess, d_h, nc * d * d * sizeof(double), "D2H hess"}, {cov, d_cov, nc * d * d * sizeof(double), "D2H cov"},
                         {status, d_st, nc * sizeof(int), "D2H status"}};
    for (const Out& o : outs)
        if (o.host && !cuda_ok(cudaMemcpyAsync(o.host, o.dev, o.bytes, cudaMemcpyDeviceToHost, st), o.what)) return CARMA_ERR_CUDA;
    if (!cuda_ok(cudaStreamSynchronize(st), "multi_hessian sync")) return CARMA_ERR_CUDA;
    return CARMA_OK;
}

int carma_multi_laplace(carma_multi_series_t m, int kind, int p, int q, const carma_prior_t* priors, const double* theta,
                        const double* cov, unsigned flags, size_t ndraws, uint64_t seed, uint32_t curve_offset,
                        double* draws, double* logpost, double* logq, int32_t* resample, double* ess, double* khat,
                        int* status) {
    if (!m || !theta || !cov) { set_error("carma_multi_laplace: null argument"); return CARMA_ERR_ARG; }
    if (!valid_model(kind, p, q)) { set_error("carma_multi_laplace: invalid (kind,p,q)"); return CARMA_ERR_ARG; }
    if (ndraws == 0 || ndraws > CARMA_LAPLACE_MAX_DRAWS) {
        set_error("carma_multi_laplace: ndraws must be in 1 .. CARMA_LAPLACE_MAX_DRAWS (2^20)");
        return CARMA_ERR_ARG;
    }
    if ((unsigned long long)curve_offset + m->ncurves > (1ull << 32)) {
        set_error("carma_multi_laplace: curve_offset + ncurves exceeds 2^32");
        return CARMA_ERR_ARG;
    }
    if (!alike32(m->d_dt, m->d_y) || !alike32(m->d_dt, m->d_e2)) { set_error("carma_multi_laplace: curve arrays not sector-aligned"); return CARMA_ERR_ARG; }
    const size_t nc = m->ncurves, d = (size_t)model_dim(kind, p, q), S = ndraws;
    if (!cuda_ok(cudaSetDevice(m->device), "cudaSetDevice")) return CARMA_ERR_CUDA;
    cudaStream_t st = 0;
    int rc = upload_rows(m, kind, p, q, priors, theta, nc, st);
    if (rc) return rc;
    if (!m->scratch_pts.reserve(nc * d * d * sizeof(double)) ||
        !cuda_ok(cudaMemcpyAsync(m->scratch_pts.p, cov, nc * d * d * sizeof(double), cudaMemcpyHostToDevice, st), "H2D cov"))
        return CARMA_ERR_CUDA;
    // Curves go in chunks of B whose scratch fits the budget (CARMA_MULTI_LAPLACE_BUDGET bytes, read at every call so
    // that a test can force several chunks), and whose threads fit one grid.  Every output depends only on its curve, so
    // chunking changes no bit.
    size_t budget = (size_t)4 << 30;
    if (const char* env = getenv("CARMA_MULTI_LAPLACE_BUDGET")) budget = (size_t)std::strtoull(env, nullptr, 10);
    const size_t per_curve = 8 * S * (d + 3) + 4 * S + 8 * d * d + 32;
    const size_t B = std::max<size_t>(1, std::min(std::min(nc, budget / per_curve), ((size_t)1 << 36) / S));
    // scratch_misc: L | logdet | ess | khat | w | draws | logpost | logq | fstat | status | resample
    const size_t b_L = round32(B * d * d), b_1 = round32(B), b_S = round32(B * S), b_i = round32((B + 1) / 2);
    const size_t b_D = round32(B * S * d), b_r = round32((B * S + 1) / 2);
    if (!m->scratch_misc.reserve((b_L + 3 * b_1 + 3 * b_S + b_D + 2 * b_i + b_r) * sizeof(double))) return CARMA_ERR_CUDA;
    LaplaceChunk ch;
    ch.L = (double*)m->scratch_misc.p;
    ch.logdet = ch.L + b_L;
    ch.ess = ch.logdet + b_1;
    ch.khat = ch.ess + b_1;
    ch.w = ch.khat + b_1;
    ch.draws = ch.w + b_S;
    ch.logpost = ch.draws + b_D;
    ch.logq = ch.logpost + b_S;
    ch.fstat = (int*)(ch.logq + b_S);
    ch.status = (int*)((double*)ch.fstat + b_i);
    ch.resample = (int32_t*)((double*)ch.status + b_i);
    const carma_prior_t* d_pr = (const carma_prior_t*)m->scratch_pr.p;
    const double* d_th = (const double*)m->scratch_in.p;
    const double* d_cov = (const double*)m->scratch_pts.p;
    for (size_t c0 = 0; c0 < nc; c0 += B) {
        const size_t n = std::min(B, nc - c0);
        multi_laplace_factor_kernel<<<(unsigned)((n + SF_BLOCK - 1) / SF_BLOCK), SF_BLOCK, 0, st>>>(
            d_th, d_cov, c0, n, (int)d, ch.L, ch.logdet, ch.fstat);
        if (!cuda_ok(cudaGetLastError(), "multi_laplace_factor_kernel launch")) return CARMA_ERR_CUDA;
        cudaError_t e;
#define LAUNCH_LE(PP) e = launch_laplace_eval_p<PP>(m, kind, q, flags, d_pr, d_th, c0, n, S, seed, curve_offset, ch, st)
        switch (p) {
            case 1: LAUNCH_LE(1); break;
            case 2: LAUNCH_LE(2); break;
            case 3: LAUNCH_LE(3); break;
            case 4: LAUNCH_LE(4); break;
            case 5: LAUNCH_LE(5); break;
            case 6: LAUNCH_LE(6); break;
            default: LAUNCH_LE(7); break;
        }
#undef LAUNCH_LE
        if (!cuda_ok(e, "multi_laplace_eval_kernel launch")) return CARMA_ERR_CUDA;
        multi_laplace_summary_kernel<<<(unsigned)n, LAP_THREADS, 0, st>>>(
            c0, S, ch.fstat, ch.logpost, ch.logq, ch.w, seed, curve_offset, ch.resample, ch.ess, ch.khat, ch.status);
        if (!cuda_ok(cudaGetLastError(), "multi_laplace_summary_kernel launch")) return CARMA_ERR_CUDA;
        struct Out { void* host; const void* dev; size_t bytes; const char* what; };
        const Out outs[7] = {
            {draws ? draws + c0 * S * d : nullptr, ch.draws, n * S * d * sizeof(double), "D2H draws"},
            {logpost ? logpost + c0 * S : nullptr, ch.logpost, n * S * sizeof(double), "D2H logpost"},
            {logq ? logq + c0 * S : nullptr, ch.logq, n * S * sizeof(double), "D2H logq"},
            {resample ? resample + c0 * S : nullptr, ch.resample, n * S * sizeof(int32_t), "D2H resample"},
            {ess ? ess + c0 : nullptr, ch.ess, n * sizeof(double), "D2H ess"},
            {khat ? khat + c0 : nullptr, ch.khat, n * sizeof(double), "D2H khat"},
            {status ? status + c0 : nullptr, ch.status, n * sizeof(int), "D2H status"}};
        for (const Out& o : outs)
            if (o.host && !cuda_ok(cudaMemcpyAsync(o.host, o.dev, o.bytes, cudaMemcpyDeviceToHost, st), o.what)) return CARMA_ERR_CUDA;
        // the next chunk reuses the scratch: its outputs must have left
        if (!cuda_ok(cudaStreamSynchronize(st), "multi_laplace sync")) return CARMA_ERR_CUDA;
    }
    return CARMA_OK;
}

}  // extern "C"
