// mle_dev.cu -- the optimiser of get_mle / choose_order ON THE DEVICE: one warp per random start.
//
// carma_mle_batch (mle.cu) keeps the L-BFGS loop on the host and sends every batch of trial points through a K1
// launch: an iteration costs a launch, two PCIe copies and a synchronise on top of the one evaluation of latency it
// really needs, and all starts of a model wait for the slowest at every step.  Here the whole fit of a start runs
// inside one kernel (reference: one scipy.optimize.minimize(L-BFGS-B) per start, src/carmcmc/carma_pack.py:195-252):
//
//   * a warp owns a start; in an evaluation round lane l evaluates trial point l (a complete LogDensity: the same
//     transform_theta + KalmanReal code as K1/K3), so the d forward-difference points of a gradient, or the four
//     step sizes of a backtracking round plus the d difference points around the full step, cost ONE evaluation
//     of latency;
//   * lane 0 runs the O(m d) optimiser arithmetic (two-loop recursion, Armijo test, curvature test, restarts) on
//     the warp's shared-memory work area;
//   * a block is four warps, one per SM sub-partition, and an SM holds one block; the warps share one copy of the
//     light curve in shared memory; after that copy the warps never synchronise again: fits differ tenfold in their iteration
//     counts, so each warp takes its next start from a queue (an atomic counter) when it is done.
//
// carma_mle_grid_device fits SEVERAL models in the same launch (choose_order: 28 models x 100 starts): the queue runs
// over the starts of all jobs, heaviest job first, and a warp dispatches on the order of the job it popped.  One launch
// per model from concurrent host threads was tried first and did not overlap: 16 streams of long-running kernels
// (0.1 - 0.6 s each) delay each other's launches (shared hardware queues: a copy waiting behind a fit blocks the launch
// queued after it; SMs reconfiguring their shared-memory split), 2.5 - 3.2 s for the grid against 0.98 s for 2,800 starts
// of the heaviest model in ONE launch (scripts/mle_probe7.py ... mle_probe11.py, profiles/r03*_mle_*).
//
// The algorithm is lbfgs_core's, decision for decision (projected L-BFGS, history 8 per start, forward differences
// with a backward retry at an infeasible point, speculative gradient at the full step, two history-reset restarts,
// the same stopping rules), lane 0 does its arithmetic with explicitly rounded multiplies and adds, i.e. without FMA
// contraction, like the host compiler, and the trial points are evaluated by K1's arithmetic (the prologue with its
// LU in shared memory, the same filter loop): a fit takes the host fit's path and ends at the same point with the
// same value after the same number of iterations, bit for bit (tested).  Only the evaluation counts differ: a
// backtracking round tries every halving of the step that fits into the warp's free lanes, the host loop four per
// launch; the first candidate that passes is taken either way.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <mutex>
#include <string>
#include <vector>

#include "kalman_real.cuh"
#include "series.h"
#include "theta_transform.cuh"

namespace carma {
namespace {

constexpr int ML_WARPS = 4;              // one warp per SM sub-partition; a warp owns one start at a time (work queue)
// ONE block per SM, i.e. one warp per sub-partition: a second or third warp on a scheduler slows this kernel down by
// more than it adds (28 x 100 starts: 0.67 s with one block per SM, 0.90 with two, 0.75-0.83 with three; 28 x 300
// starts: 1.02 against 1.39-1.43 s, profiles/r03y_mle_blocks_per_sm.txt) -- the warps of different fits run different
// orders' loops and prologues through one instruction cache and keep 3 kB of local memory each in one L1 -- and the
// register allocation is free to use 255 registers.
constexpr int ML_BLOCKS_PER_SM = 1;
constexpr int ML_M = 8;                  // history pairs kept per start
constexpr int ML_D = MAX_D;              // row stride of the work arrays
constexpr double ML_BIG = 1e300;
constexpr size_t ML_SMEM_MAX = 200 * 1024;
constexpr int ML_LU = 2 * MAX_P * MAX_P * 32;   // LU scratch of the prologue per warp, doubles

struct MleDevParams {     // the optimiser's options, common to all jobs of a launch
    int maxiter, history, max_backtrack;
    double gtol, ftol, fd_eps;
    int series_in_smem;
    int njobs;
    unsigned long long total;   // starts of all jobs
};
struct MleJob {           // one model: its starts are rows [first, first + nstart) of the queue
    int kind, p, q, d;
    unsigned flags;
    carma_prior_t prior;
    unsigned long long first, nstart;
    unsigned long long x_off;   // offset (doubles) of its rows in x0 / x_out; bounds at job index * MAX_D
};

// per-warp work area, in doubles
constexpr int ML_AREA = 32 * ML_D /*pts*/ + 32 /*fv*/ + 7 * ML_D /*x g xn gn pg qv dir*/ + 2 * ML_M * ML_D /*S Y*/ +
                        2 * ML_M /*rho alpha*/ + 2 * ML_D /*blocked, retry (ints, one double slot each)*/;

// Multi-curve mode (carma_multi_mle_grid_device): the queue runs over (job, curve, start).  Within a job the rows
// are curve-major in the order of `order` (curve indices, longest curve first); x0 / x_out / f_out / bounds / nit /
// nfev keep the caller's curve order.
struct MleCurve {         // what a fit needs of its curve beside the data: the prior and the curve's own longest gap
    carma_prior_t prior;
    double dt_max;
};
struct MleMulti {
    const double *dt, *y, *e2;          // CSR arrays of the multi-series
    const long long* off;               // ncurves + 1
    const int* order;                   // ncurves: curve indices, longest first
    const MleCurve* curve;              // ncurves
    const unsigned long long* per_curve;   // njobs: starts per curve of each job (device job order)
    unsigned long long ncurves;
};

// IEEE operations that the compiler may not contract into FMAs (see the header comment)
__device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double sub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double dvd(double a, double b) { return __ddiv_rn(a, b); }
__device__ __forceinline__ double max_(double a, double b) { return (a < b) ? b : a; }   // std::max
__device__ __forceinline__ double min_(double a, double b) { return (b < a) ? b : a; }   // std::min

// -LogDensity(theta), non-finite -> BIG (GpuObjective::run of mle.cu)
template <int P>
__device__ __noinline__ double neg_logdensity(const MleDevParams& mp, const MleJob& job, const SeriesView& sv, const MathTab& tb,
                                              const double* th, const double* sdt, const double* sy, const double* se,
                                              double* lu) {
    RealParams<P> prm;
    double lp;
    // the P x P complex LU of the prologue works in the warp's shared-memory scratch ([element][lane]), as in K1
    if (transform_theta<P, false, true>(job.kind, job.q, job.flags, job.prior, th, sv.dt_max, prm, nullptr, lu, 32) != TT_OK) {
        lp = -INFINITY;
    } else {
        KalmanReal<P> kf;
        LogLikAcc acc;
        kf.reset(prm, sv.e2_0);
        acc.init();
        const SeriesPtr gsrc{sv.dt, sv.y, sv.e2n};
        if (mp.series_in_smem) {
            const uint32_t a = smem_u32(sdt);
            const SeriesSmem src{a, smem_u32(sy) - a, smem_u32(se) - a};
            filter_span_any<P, false>(kf, acc, prm, tb, src, sv.ny, sv.ny - 1);
        } else {
            filter_span_any<P, true>(kf, acc, prm, tb, gsrc, sv.ny, sv.ny - 1);
        }
        lp = acc.bad() ? loglik_exact_slow<P>(prm, tb, gsrc, sv.ny, sv.e2_0) + prm.logprior : acc.value() + prm.logprior;
    }
    const double v = -lp;
    return isfinite(v) ? v : ML_BIG;
}

template <int P>
struct WarpFit {
    const MleDevParams& mp;
    const MleJob& job;
    const SeriesView& sv;
    const MathTab& tb;
    const double *sdt, *sy, *se;
    const double *lower, *upper;
    int lane, d;
    double* lu;   // this lane's column of the warp's LU scratch
    // work area
    double *pts, *fv, *x, *g, *xn, *gn, *pg, *qv, *dir, *S, *Y, *rho, *alpha;
    int *blocked, *retry;
    long long nfev;

    __device__ void carve(double* a) {
        pts = a; a += 32 * ML_D;
        fv = a; a += 32;
        x = a; a += ML_D;
        g = a; a += ML_D;
        xn = a; a += ML_D;
        gn = a; a += ML_D;
        pg = a; a += ML_D;
        qv = a; a += ML_D;
        dir = a; a += ML_D;
        S = a; a += ML_M * ML_D;
        Y = a; a += ML_M * ML_D;
        rho = a; a += ML_M;
        alpha = a; a += ML_M;
        blocked = (int*)a; a += ML_D;
        retry = (int*)a;
    }

    // lane l < npts evaluates pts[l]; fv[l] = value
    __device__ void eval(int npts) {
        __syncwarp();
        double v = ML_BIG;
        if (lane < npts) {
            double th[MAX_D];
#pragma unroll
            for (int j = 0; j < MAX_D; j++) th[j] = (j < d) ? pts[lane * ML_D + j] : 0.0;
            v = neg_logdensity<P>(mp, job, sv, tb, th, sdt, sy, se, lu);
        }
        __syncwarp();
        fv[lane] = v;
        nfev += npts;
        __syncwarp();
    }

    __device__ double fd_step(double zj, int j) const { return (add(zj, mp.fd_eps) > upper[j]) ? -mp.fd_eps : mp.fd_eps; }

    // forward-difference gradient at (z, fz) -> gout, with the backward retry of lbfgs_core::grad
    __device__ void grad(const double* z, double fz, double* gout) {
        if (lane == 0)
            for (int j = 0; j < d; j++) {
                for (int k = 0; k < d; k++) pts[j * ML_D + k] = z[k];
                pts[j * ML_D + j] = add(pts[j * ML_D + j], fd_step(z[j], j));
            }
        eval(d);
        int nretry = 0;
        if (lane == 0) {
            for (int j = 0; j < d; j++) {
                const double h = fd_step(z[j], j);
                if (fabs(fv[j]) >= ML_BIG) { gout[j] = 0.0; retry[nretry++] = j; }
                else gout[j] = dvd(sub(fv[j], fz), h);
            }
            for (int k = 0; k < nretry; k++) {
                const int j = retry[k];
                for (int c = 0; c < d; c++) pts[k * ML_D + c] = z[c];
                const double hb = -fd_step(z[j], j);
                const double zb = add(z[j], hb);
                if (zb >= lower[j] && zb <= upper[j]) pts[k * ML_D + j] = zb;
            }
        }
        nretry = __shfl_sync(0xffffffffu, nretry, 0);
        if (nretry == 0) return;
        eval(nretry);
        if (lane == 0)
            for (int k = 0; k < nretry; k++) {
                const int j = retry[k];
                const double hb = -fd_step(z[j], j);
                const double zb = add(z[j], hb);
                const bool stepped = zb >= lower[j] && zb <= upper[j];
                if (stepped && fabs(fv[k]) < ML_BIG) gout[j] = dvd(sub(fv[k], fz), hb);
            }
        __syncwarp();
    }

    // two-loop recursion on the projected gradient -> dir; returns the slope (lane 0 only)
    __device__ double direction(int nh, int h0) {
        const int m = mp.history;
        for (int j = 0; j < d; j++) qv[j] = pg[j];
        for (int h = nh - 1; h >= 0; h--) {
            const int sl = (h0 + h) % m;
            const double *s = S + sl * ML_D, *y = Y + sl * ML_D;
            double sy_ = 0.0, sq = 0.0;
            for (int j = 0; j < d; j++) { sy_ = add(sy_, mul(s[j], y[j])); sq = add(sq, mul(s[j], qv[j])); }
            const double r = dvd(1.0, max_(sy_, 1e-300)), a = mul(r, sq);
            rho[sl] = r;
            alpha[sl] = a;
            for (int j = 0; j < d; j++) qv[j] = sub(qv[j], mul(a, y[j]));
        }
        if (nh > 0) {
            const int sl = (h0 + nh - 1) % m;
            const double *s = S + sl * ML_D, *y = Y + sl * ML_D;
            double sy_ = 0.0, yy = 0.0;
            for (int j = 0; j < d; j++) { sy_ = add(sy_, mul(s[j], y[j])); yy = add(yy, mul(y[j], y[j])); }
            const double gam = min_(max_(dvd(sy_, max_(yy, 1e-300)), 1e-8), 1e8);
            for (int j = 0; j < d; j++) qv[j] = mul(qv[j], gam);
        } else {
            double nrm = 0.0;
            for (int j = 0; j < d; j++) nrm = add(nrm, mul(pg[j], pg[j]));
            const double sc = dvd(1.0, max_(__dsqrt_rn(nrm), 1.0));
            for (int j = 0; j < d; j++) qv[j] = mul(qv[j], sc);
        }
        for (int h = 0; h < nh; h++) {
            const int sl = (h0 + h) % m;
            const double *s = S + sl * ML_D, *y = Y + sl * ML_D;
            double yq = 0.0;
            for (int j = 0; j < d; j++) yq = add(yq, mul(y[j], qv[j]));
            const double b = mul(rho[sl], yq), a = alpha[sl];
            for (int j = 0; j < d; j++) qv[j] = add(qv[j], mul(sub(a, b), s[j]));
        }
        double sl_ = 0.0, pg2 = 0.0;
        for (int j = 0; j < d; j++) {
            dir[j] = blocked[j] ? 0.0 : -qv[j];
            sl_ = add(sl_, mul(dir[j], pg[j]));
            pg2 = add(pg2, mul(pg[j], pg[j]));
        }
        if (!(sl_ < 0)) {
            for (int j = 0; j < d; j++) dir[j] = -pg[j];
            sl_ = -pg2;
        }
        return sl_;
    }

    // the whole fit of one start; returns the iteration count as lbfgs_core would report it for this row alone
    __device__ int run(const double* x0, double* x_out, double* f_out) {
        const int m = mp.history;
        double f = 0.0;
        if (lane == 0) {
            for (int j = 0; j < d; j++) {
                x[j] = min_(max_(x0[j], lower[j]), upper[j]);
                pts[j] = x[j];
            }
        }
        eval(1);
        f = fv[0];
        grad(x, f, g);
        int active = f < ML_BIG;
        int nh = 0, h0 = 0, restarts_left = 2;
        int nit;
        for (nit = 1; nit <= mp.maxiter; nit++) {
            if (lane == 0 && active) {
                double gmax = 0.0;
                for (int j = 0; j < d; j++) {
                    const double xi = x[j], gi = g[j];
                    const bool blk = (xi <= lower[j] && gi > 0) || (xi >= upper[j] && gi < 0);
                    blocked[j] = blk;
                    pg[j] = blk ? 0.0 : gi;
                    gmax = max_(gmax, fabs(pg[j]));
                }
                if (gmax < mp.gtol) active = 0;
            }
            active = __shfl_sync(0xffffffffu, active, 0);
            if (!active) break;
            double slope = 0.0;
            if (lane == 0) slope = direction(nh, h0);
            // ---- batched Armijo backtracking: as many step sizes per round as there are lanes, the first round also
            // carries the d difference points around the full step
            double t = 1.0, fn = f;
            int todo = 1, grad_done = 0, tried = 0;
            if (lane == 0)
                for (int j = 0; j < d; j++) { xn[j] = x[j]; gn[j] = g[j]; }
            for (int round = 0; tried < mp.max_backtrack && todo; round++) {
                // every lane the round leaves free carries a further halving of the step: the candidates are those of
                // the host loop (which tries four per launch), the first one that passes is taken, so the decision is
                // the same -- but a search that has to go below t = 1/8 costs one evaluation of latency, not several
                const bool spec = (round == 0);
                const int nt = min(32 - (spec ? d : 0), mp.max_backtrack - tried);
                const int per_row = nt + (spec ? d : 0);
                if (lane == 0) {
                    double tk = t;
                    for (int c = 0; c < nt; c++, tk = mul(tk, 0.5))
                        for (int j = 0; j < d; j++) pts[c * ML_D + j] = min_(max_(add(x[j], mul(tk, dir[j])), lower[j]), upper[j]);
                    if (spec)
                        for (int j = 0; j < d; j++) {
                            double* pt = pts + (nt + j) * ML_D;
                            for (int k = 0; k < d; k++) pt[k] = pts[k];
                            pt[j] = add(pt[j], fd_step(pts[j], j));
                        }
                }
                eval(per_row);
                if (lane == 0) {
                    double tk = t;
                    int hit = -1;
                    for (int c = 0; c < nt; c++, tk = mul(tk, 0.5))
                        if (fv[c] <= add(f, mul(mul(1e-4, tk), slope))) { hit = c; break; }
                    if (hit >= 0) {
                        for (int j = 0; j < d; j++) xn[j] = pts[hit * ML_D + j];
                        fn = fv[hit];
                        todo = 0;
                        if (spec && hit == 0) {
                            bool all_finite = true;
                            for (int j = 0; j < d; j++) {
                                const double h = fd_step(pts[j], j);
                                const double fvj = fv[nt + j];
                                if (fabs(fvj) >= ML_BIG) all_finite = false;
                                gn[j] = dvd(sub(fvj, fn), h);
                            }
                            grad_done = all_finite;
                        }
                    } else {
                        for (int c = 0; c < nt; c++) t = mul(t, 0.5);
                    }
                }
                todo = __shfl_sync(0xffffffffu, todo, 0);
                tried += nt;
            }
            grad_done = __shfl_sync(0xffffffffu, grad_done, 0);
            fn = __shfl_sync(0xffffffffu, fn, 0);
            const int moved = !todo;
            __syncwarp();
            if (moved && !grad_done) grad(xn, fn, gn);
            if (lane == 0) {
                if (moved) {
                    double sy_ = 0.0;
                    for (int j = 0; j < d; j++) sy_ = add(sy_, mul(sub(xn[j], x[j]), sub(gn[j], g[j])));
                    if (sy_ > 1e-12) {
                        int dst;
                        if (nh == m) { dst = h0; h0 = (h0 + 1) % m; }
                        else { dst = (h0 + nh) % m; nh++; }
                        for (int j = 0; j < d; j++) { S[dst * ML_D + j] = sub(xn[j], x[j]); Y[dst * ML_D + j] = sub(gn[j], g[j]); }
                    }
                }
                const bool small = moved && (sub(f, fn) <= mul(mp.ftol, max_(max_(fabs(f), fabs(fn)), 1.0)));
                if (todo || small) {
                    if (nh > 0 && restarts_left > 0) { nh = 0; h0 = 0; restarts_left--; }
                    else active = 0;
                }
                for (int j = 0; j < d; j++) { x[j] = xn[j]; g[j] = gn[j]; }
            }
            f = fn;
            active = __shfl_sync(0xffffffffu, active, 0);
            __syncwarp();
        }
        if (lane == 0) {
            for (int j = 0; j < d; j++) x_out[j] = x[j];
            *f_out = f;
        }
        return min(nit, mp.maxiter);
    }
};

// the whole fit of one start of `job` by the calling warp
template <int P>
__device__ __noinline__ void fit_start(const MleDevParams& mp, const MleJob& job, const SeriesView& sv, const MathTab& tb,
                                       const double* sdt, const double* sy, const double* se, const double* lower,
                                       const double* upper, double* area, int lane, const double* x0, double* x_out,
                                       double* f_out, int* nit_out, unsigned long long* nfev_out) {
    WarpFit<P> fit{mp, job, sv, tb, sdt, sy, se, lower, upper, lane, job.d, area + ML_AREA + lane};
    fit.carve(area);
    fit.nfev = 0;
    const int nit = fit.run(x0, x_out, f_out);
    if (lane == 0) {
        atomicMax(nit_out, nit);
        atomicAdd(nfev_out, (unsigned long long)fit.nfev);
    }
}

__device__ __forceinline__ void fit_start_p(int p, const MleDevParams& mp, const MleJob& job, const SeriesView& sv, const MathTab& tb,
                                            const double* sdt, const double* sy, const double* se, const double* lo,
                                            const double* hi, double* area, int lane, const double* xs, double* xo,
                                            double* fo, int* nit, unsigned long long* nfev) {
    switch (p) {
        case 1: fit_start<1>(mp, job, sv, tb, sdt, sy, se, lo, hi, area, lane, xs, xo, fo, nit, nfev); break;
        case 2: fit_start<2>(mp, job, sv, tb, sdt, sy, se, lo, hi, area, lane, xs, xo, fo, nit, nfev); break;
        case 3: fit_start<3>(mp, job, sv, tb, sdt, sy, se, lo, hi, area, lane, xs, xo, fo, nit, nfev); break;
        case 4: fit_start<4>(mp, job, sv, tb, sdt, sy, se, lo, hi, area, lane, xs, xo, fo, nit, nfev); break;
        case 5: fit_start<5>(mp, job, sv, tb, sdt, sy, se, lo, hi, area, lane, xs, xo, fo, nit, nfev); break;
        case 6: fit_start<6>(mp, job, sv, tb, sdt, sy, se, lo, hi, area, lane, xs, xo, fo, nit, nfev); break;
        default: fit_start<7>(mp, job, sv, tb, sdt, sy, se, lo, hi, area, lane, xs, xo, fo, nit, nfev); break;
    }
}

// MULTI = false: one series (sv), staged once per block when it fits.  MULTI = true: every row names its curve of
// the multi-series `mm` (sv is unused) and the fit reads the curve from global memory: staging it into the warp's own
// shared-memory slice was measured slower (DESIGN.md, lbfgs_kernel).
template <bool MULTI>
__global__ void __launch_bounds__(ML_WARPS * 32, ML_BLOCKS_PER_SM) lbfgs_kernel(SeriesView sv, MleDevParams mp, const MleJob* __restrict__ jobs,
                                                              const double* __restrict__ x0, const double* __restrict__ bounds,
                                                              double* __restrict__ x_out, double* __restrict__ f_out,
                                                              int* __restrict__ nit_out, unsigned long long* __restrict__ nfev_out,
                                                              unsigned long long* __restrict__ next_row, MleMulti mm) {
    extern __shared__ __align__(16) double smem[];
    MathTab tb;
    tb.load();
    if constexpr (MULTI) {
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
        double* area = smem + (size_t)warp * (ML_AREA + ML_LU);
        for (;;) {
            unsigned long long row = 0;
            if (lane == 0) row = atomicAdd(next_row, 1ull);
            row = __shfl_sync(0xffffffffu, row, 0);
            if (row >= mp.total) break;
            int j = 0;
            while (j + 1 < mp.njobs && row >= jobs[j].first + jobs[j].nstart) j++;
            const unsigned long long ns = mm.per_curve[j], r = row - jobs[j].first;
            const int c = mm.order[r / ns];
            const unsigned long long idx = (unsigned long long)c * ns + r % ns;   // the row's place in the caller's layout
            const long long o0 = mm.off[c];
            const int ny = (int)(mm.off[c + 1] - o0);
            // the curve as a Series built from it would hold it: gaps to the next point, the next point's yerr^2
            SeriesView cv;
            cv.dt = mm.dt + o0;
            cv.y = mm.y + o0;
            cv.e2n = mm.e2 + o0 + 1;
            cv.t = nullptr;
            cv.e2_0 = mm.e2[o0];
            cv.dt_max = mm.curve[c].dt_max;
            cv.ny = ny;
            cv.nyp = ny;
            MleJob job = jobs[j];
            job.prior = mm.curve[c].prior;
            const unsigned long long pc = (unsigned long long)j * mm.ncurves + c;
            const double *lo = bounds + pc * 2 * MAX_D, *hi = lo + MAX_D;
            fit_start_p(job.p, mp, job, cv, tb, nullptr, nullptr, nullptr, lo, hi, area, lane,
                           x0 + job.x_off + idx * job.d, x_out + job.x_off + idx * job.d, f_out + job.first + idx,
                           nit_out + pc, nfev_out + pc);
            __syncwarp();
        }
        return;
    }
    const int nyp = mp.series_in_smem ? sv.nyp : 0;
    double *sdt = smem, *sy = smem + nyp, *se = smem + 2 * (size_t)nyp;
    if (mp.series_in_smem) {
        for (int k = threadIdx.x; k < sv.nyp; k += blockDim.x) {
            sdt[k] = sv.dt[k];
            sy[k] = sv.y[k];
            se[k] = sv.e2n[k];
        }
        __syncthreads();
    }
    // from here on the warps of a block never meet again: each takes the next unfitted start from the queue until
    // none is left
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double* area = smem + 3 * (size_t)nyp + (size_t)warp * (ML_AREA + ML_LU);
    for (;;) {
        unsigned long long row = 0;
        if (lane == 0) row = atomicAdd(next_row, 1ull);
        row = __shfl_sync(0xffffffffu, row, 0);
        if (row >= mp.total) break;
        int j = 0;
        while (j + 1 < mp.njobs && row >= jobs[j].first + jobs[j].nstart) j++;
        const MleJob& job = jobs[j];
        const unsigned long long r = row - job.first;
        const double *lo = bounds + (size_t)j * 2 * MAX_D, *hi = lo + MAX_D;
        const double* xs = x0 + job.x_off + r * (unsigned long long)job.d;
        double* xo = x_out + job.x_off + r * (unsigned long long)job.d;
        switch (job.p) {
            case 1: fit_start<1>(mp, job, sv, tb, sdt, sy, se, lo, hi, area, lane, xs, xo, f_out + row, nit_out + j, nfev_out + j); break;
            case 2: fit_start<2>(mp, job, sv, tb, sdt, sy, se, lo, hi, area, lane, xs, xo, f_out + row, nit_out + j, nfev_out + j); break;
            case 3: fit_start<3>(mp, job, sv, tb, sdt, sy, se, lo, hi, area, lane, xs, xo, f_out + row, nit_out + j, nfev_out + j); break;
            case 4: fit_start<4>(mp, job, sv, tb, sdt, sy, se, lo, hi, area, lane, xs, xo, f_out + row, nit_out + j, nfev_out + j); break;
            case 5: fit_start<5>(mp, job, sv, tb, sdt, sy, se, lo, hi, area, lane, xs, xo, f_out + row, nit_out + j, nfev_out + j); break;
            case 6: fit_start<6>(mp, job, sv, tb, sdt, sy, se, lo, hi, area, lane, xs, xo, f_out + row, nit_out + j, nfev_out + j); break;
            default: fit_start<7>(mp, job, sv, tb, sdt, sy, se, lo, hi, area, lane, xs, xo, f_out + row, nit_out + j, nfev_out + j); break;
        }
        __syncwarp();
    }
}

template <bool MULTI>
cudaError_t lbfgs_attrs() {
    static OncePerDevice once;
    return once.run([] { return cudaFuncSetAttribute(lbfgs_kernel<MULTI>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ML_SMEM_MAX); });
}

// smem: dynamic shared memory of a block, bytes
template <bool MULTI>
cudaError_t launch_lbfgs(const SeriesView& sv, const MleDevParams& mp, const MleJob* jobs, const double* x0, const double* bounds,
                         double* x_out, double* f_out, int* nit, unsigned long long* nfev, unsigned long long* next_row,
                         const MleMulti& mm, size_t smem, cudaStream_t st) {
    const cudaError_t attr_err = lbfgs_attrs<MULTI>();
    if (attr_err != cudaSuccess) return attr_err;
    int nsm = 148, dev = 0;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
    const size_t want = ((size_t)mp.total + ML_WARPS - 1) / ML_WARPS, cap = (size_t)nsm * ML_BLOCKS_PER_SM;
    const unsigned grid = (unsigned)std::min(want, cap);
    lbfgs_kernel<MULTI><<<grid, ML_WARPS * 32, smem, st>>>(sv, mp, jobs, x0, bounds, x_out, f_out, nit, nfev, next_row, mm);
    return cudaGetLastError();
}

// heaviest job first (the long fits start first); stable, so equal weights keep the caller's order
std::vector<int> jobs_heaviest_first(int njobs, const carma_mle_job_t* jobs) {
    std::vector<int> order(njobs);
    for (int j = 0; j < njobs; j++) order[j] = j;
    auto weight = [&](int j) {
        const int d = model_dim(jobs[j].kind, jobs[j].p, jobs[j].q);
        return (double)jobs[j].p * jobs[j].p * (d + 1);
    };
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return weight(a) > weight(b); });
    return order;
}

bool valid_job(const carma_mle_job_t& jb) {
    return !(jb.kind < CARMA_KIND_CAR1 || jb.kind > CARMA_KIND_ZCARMA || jb.p < 1 || jb.p > MAX_P ||
             (jb.kind == CARMA_KIND_CAR1 && jb.p != 1) || (jb.kind == CARMA_KIND_CARMA && !(jb.q >= 0 && jb.q < jb.p)));
}

}  // namespace
}  // namespace carma

using namespace carma;

extern "C" int carma_mle_grid_device(carma_series_t s, int njobs, const carma_mle_job_t* jobs, const double* x0,
                                     const double* lower, const double* upper, const carma_mle_opts_t* opts,
                                     double* x_out, double* f_out, int* nit_out, long long* nfev_out, int slot) {
    if (!s || njobs < 0 || (njobs > 0 && (!jobs || !x0 || !lower || !upper || !x_out || !f_out)) || slot < 0 || slot >= CARMA_N_SLOTS) {
        set_error("carma_mle_grid_device: bad argument");
        return CARMA_ERR_ARG;
    }
    carma_mle_opts_t o;
    if (opts) o = *opts; else carma_mle_default_opts(&o);
    if (o.maxiter < 0 || o.history < 1 || o.history > ML_M || o.max_backtrack < 1 || !(o.fd_eps > 0)) {
        set_error("carma_mle_grid_device: invalid options (1 <= history <= 8)");
        return CARMA_ERR_ARG;
    }
    std::vector<MleJob> dj(njobs);
    std::vector<size_t> f_first(njobs), x_first(njobs);
    size_t total = 0, xdoubles = 0;
    for (int j = 0; j < njobs; j++) {
        const carma_mle_job_t& jb = jobs[j];
        if (!valid_job(jb)) {
            set_error("carma_mle_grid_device: invalid (kind,p,q) in job " + std::to_string(j));
            return CARMA_ERR_ARG;
        }
        f_first[j] = total;
        x_first[j] = xdoubles;
        total += jb.nstart;
        xdoubles += jb.nstart * (size_t)model_dim(jb.kind, jb.p, jb.q);
    }
    for (int j = 0; j < njobs; j++) {
        if (nit_out) nit_out[j] = 0;
        if (nfev_out) nfev_out[j] = 0;
    }
    if (total == 0) return CARMA_OK;
    // the queue serves the jobs in this order
    const std::vector<int> order = jobs_heaviest_first(njobs, jobs);
    // device order: rows of job order[k] follow those of order[k-1] in the queue, in x and in f
    std::vector<double> hx(xdoubles), hb((size_t)njobs * 2 * MAX_D, 0.0);
    size_t qrow = 0, qx = 0;
    for (int k = 0; k < njobs; k++) {
        const int j = order[k];
        const carma_mle_job_t& jb = jobs[j];
        const int d = model_dim(jb.kind, jb.p, jb.q);
        MleJob& m = dj[k];
        m.kind = jb.kind; m.p = jb.p; m.q = jb.q; m.d = d; m.flags = jb.flags; m.prior = jb.prior;
        m.first = qrow; m.nstart = jb.nstart; m.x_off = qx;
        std::copy(x0 + x_first[j], x0 + x_first[j] + jb.nstart * d, hx.begin() + qx);
        std::copy(lower + (size_t)j * CARMA_MAX_DIM, lower + (size_t)j * CARMA_MAX_DIM + d, hb.begin() + (size_t)k * 2 * MAX_D);
        std::copy(upper + (size_t)j * CARMA_MAX_DIM, upper + (size_t)j * CARMA_MAX_DIM + d, hb.begin() + (size_t)k * 2 * MAX_D + MAX_D);
        qrow += jb.nstart;
        qx += jb.nstart * d;
    }
    if (!cuda_ok(cudaSetDevice(s->device), "cudaSetDevice")) return CARMA_ERR_CUDA;
    if (!s->slot_stream[slot] && !cuda_ok(cudaStreamCreateWithFlags(&s->slot_stream[slot], cudaStreamNonBlocking), "cudaStreamCreate")) return CARMA_ERR_CUDA;
    cudaStream_t st = s->slot_stream[slot];
    // slot_in: [ x0 | bounds njobs x 2 x MAX_D | jobs ]   slot_out: [ x | f total | nfev njobs | queue head | nit njobs ]
    const size_t jobs_bytes = (size_t)njobs * sizeof(MleJob);
    const size_t in_bytes = (xdoubles + hb.size()) * sizeof(double) + jobs_bytes;
    const size_t out_bytes = (xdoubles + total + (size_t)njobs + 1) * sizeof(double) + (size_t)njobs * sizeof(int);
    if (in_bytes > s->slot_in[slot].cap || out_bytes > s->slot_out[slot].cap) {
        if (!cuda_ok(cudaStreamSynchronize(st), "slot sync")) return CARMA_ERR_CUDA;
        if (!s->slot_in[slot].reserve(in_bytes) || !s->slot_out[slot].reserve(out_bytes)) return CARMA_ERR_CUDA;
    }
    double* din = (double*)s->slot_in[slot].p;
    double* dout = (double*)s->slot_out[slot].p;
    double* d_b = din + xdoubles;
    MleJob* d_jobs = (MleJob*)(d_b + hb.size());
    double* d_f = dout + xdoubles;
    unsigned long long* d_nfev = (unsigned long long*)(d_f + total);
    unsigned long long* d_next = d_nfev + njobs;
    int* d_nit = (int*)(d_next + 1);
    if (!cuda_ok(cudaMemcpyAsync(din, hx.data(), xdoubles * sizeof(double), cudaMemcpyHostToDevice, st), "H2D x0") ||
        !cuda_ok(cudaMemcpyAsync(d_b, hb.data(), hb.size() * sizeof(double), cudaMemcpyHostToDevice, st), "H2D bounds") ||
        !cuda_ok(cudaMemcpyAsync(d_jobs, dj.data(), jobs_bytes, cudaMemcpyHostToDevice, st), "H2D jobs") ||
        !cuda_ok(cudaMemsetAsync(d_nfev, 0, ((size_t)njobs + 1) * sizeof(double) + (size_t)njobs * sizeof(int), st), "memset counters"))
        return CARMA_ERR_CUDA;
    SeriesView sv = s->view();
    MleDevParams mp{};
    mp.maxiter = o.maxiter; mp.history = o.history; mp.max_backtrack = o.max_backtrack;
    mp.gtol = o.gtol; mp.ftol = o.ftol; mp.fd_eps = o.fd_eps;
    mp.njobs = njobs;
    mp.total = total;
    mp.series_in_smem = ((3 * (size_t)sv.nyp + (size_t)ML_WARPS * (ML_AREA + ML_LU)) * sizeof(double) <= ML_SMEM_MAX) ? 1 : 0;
    const size_t smem = ((mp.series_in_smem ? 3 * (size_t)sv.nyp : 0) + (size_t)ML_WARPS * (ML_AREA + ML_LU)) * sizeof(double);
    if (!cuda_ok(launch_lbfgs<false>(sv, mp, d_jobs, din, d_b, dout, d_f, d_nit, d_nfev, d_next, MleMulti{}, smem, st), "lbfgs_kernel launch"))
        return CARMA_ERR_CUDA;
    std::vector<double> rx(xdoubles), rf(total);
    std::vector<int> rnit(njobs);
    std::vector<unsigned long long> rnfev(njobs);
    if (!cuda_ok(cudaMemcpyAsync(rx.data(), dout, xdoubles * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H x") ||
        !cuda_ok(cudaMemcpyAsync(rf.data(), d_f, total * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H f") ||
        !cuda_ok(cudaMemcpyAsync(rnit.data(), d_nit, (size_t)njobs * sizeof(int), cudaMemcpyDeviceToHost, st), "D2H nit") ||
        !cuda_ok(cudaMemcpyAsync(rnfev.data(), d_nfev, (size_t)njobs * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st), "D2H nfev") ||
        !cuda_ok(cudaStreamSynchronize(st), "mle sync"))
        return CARMA_ERR_CUDA;
    for (int k = 0; k < njobs; k++) {
        const int j = order[k];
        const MleJob& m = dj[k];
        std::copy(rx.begin() + m.x_off, rx.begin() + m.x_off + m.nstart * m.d, x_out + x_first[j]);
        std::copy(rf.begin() + m.first, rf.begin() + m.first + m.nstart, f_out + f_first[j]);
        if (nit_out) nit_out[j] = rnit[k];
        if (nfev_out) nfev_out[j] = (long long)rnfev[k];
    }
    return CARMA_OK;
}

extern "C" int carma_mle_batch_device(carma_series_t s, int kind, int p, int q, const carma_prior_t* prior, unsigned flags,
                                      size_t nstart, const double* x0, const double* lower, const double* upper,
                                      const carma_mle_opts_t* opts, double* x_out, double* f_out, int* nit_out,
                                      long long* nfev_out, int slot) {
    if (!s || !prior || !x0 || !lower || !upper || !x_out || !f_out || slot < 0 || slot >= CARMA_N_SLOTS) {
        set_error("carma_mle_batch_device: bad argument");
        return CARMA_ERR_ARG;
    }
    if (nit_out) *nit_out = 0;
    if (nfev_out) *nfev_out = 0;
    carma_mle_job_t jb{};
    jb.kind = kind; jb.p = p; jb.q = q; jb.flags = flags; jb.prior = *prior; jb.nstart = nstart;
    if (kind < CARMA_KIND_CAR1 || kind > CARMA_KIND_ZCARMA || p < 1 || p > MAX_P || (kind == CARMA_KIND_CAR1 && p != 1) ||
        (kind == CARMA_KIND_CARMA && !(q >= 0 && q < p))) {
        set_error("carma_mle_batch_device: invalid (kind,p,q)");
        return CARMA_ERR_ARG;
    }
    const int d = model_dim(kind, p, q);
    double lo[CARMA_MAX_DIM] = {}, hi[CARMA_MAX_DIM] = {};
    std::copy(lower, lower + d, lo);
    std::copy(upper, upper + d, hi);
    return carma_mle_grid_device(s, 1, &jb, x0, lo, hi, opts, x_out, f_out, nit_out, nfev_out, slot);
}

extern "C" int carma_multi_mle_grid_device(carma_multi_series_t m, int njobs, const carma_mle_job_t* jobs,
                                           const carma_prior_t* priors, const double* x0, const double* lower,
                                           const double* upper, const carma_mle_opts_t* opts, double* x_out,
                                           double* f_out, int* nit_out, long long* nfev_out) {
    if (!m || njobs < 0 || (njobs > 0 && (!jobs || !x0 || !lower || !upper || !x_out || !f_out))) {
        set_error("carma_multi_mle_grid_device: bad argument");
        return CARMA_ERR_ARG;
    }
    carma_mle_opts_t o;
    if (opts) o = *opts; else carma_mle_default_opts(&o);
    if (o.maxiter < 0 || o.history < 1 || o.history > ML_M || o.max_backtrack < 1 || !(o.fd_eps > 0)) {
        set_error("carma_multi_mle_grid_device: invalid options (1 <= history <= 8)");
        return CARMA_ERR_ARG;
    }
    const size_t nc = m->ncurves;
    std::vector<size_t> f_first(njobs), x_first(njobs);
    size_t total = 0, xdoubles = 0;
    for (int j = 0; j < njobs; j++) {
        if (!valid_job(jobs[j])) {
            set_error("carma_multi_mle_grid_device: invalid (kind,p,q) in job " + std::to_string(j));
            return CARMA_ERR_ARG;
        }
        f_first[j] = total;
        x_first[j] = xdoubles;
        total += nc * jobs[j].nstart;
        xdoubles += nc * jobs[j].nstart * (size_t)model_dim(jobs[j].kind, jobs[j].p, jobs[j].q);
    }
    for (size_t k = 0; k < (size_t)njobs * nc; k++) {
        if (nit_out) nit_out[k] = 0;
        if (nfev_out) nfev_out[k] = 0;
    }
    if (total == 0) return CARMA_OK;
    const std::vector<int> order = jobs_heaviest_first(njobs, jobs);
    // within a job the longest curves first: a fit's latency scales with ny and the launch lasts as long as its slowest fit
    std::vector<int> corder(nc);
    for (size_t c = 0; c < nc; c++) corder[c] = (int)c;
    std::stable_sort(corder.begin(), corder.end(), [&](int a, int b) { return m->off[a + 1] - m->off[a] > m->off[b + 1] - m->off[b]; });
    std::vector<MleCurve> hc(nc);
    for (size_t c = 0; c < nc; c++) {
        hc[c].prior = priors ? priors[c] : m->info[c].prior;
        hc[c].dt_max = m->info[c].dt_max;
    }
    // device job order; per job the rows keep the caller's (curve-major) layout, bounds are (job, curve) rows
    std::vector<MleJob> dj(njobs);
    std::vector<unsigned long long> per_curve(njobs);
    std::vector<double> hx(xdoubles), hb((size_t)njobs * nc * 2 * MAX_D, 0.0);
    size_t qrow = 0, qx = 0;
    for (int k = 0; k < njobs; k++) {
        const int j = order[k];
        const carma_mle_job_t& jb = jobs[j];
        const int d = model_dim(jb.kind, jb.p, jb.q);
        MleJob& mj = dj[k];
        mj.kind = jb.kind; mj.p = jb.p; mj.q = jb.q; mj.d = d; mj.flags = jb.flags; mj.prior = jb.prior;
        mj.first = qrow; mj.nstart = nc * jb.nstart; mj.x_off = qx;
        per_curve[k] = jb.nstart;
        std::copy(x0 + x_first[j], x0 + x_first[j] + nc * jb.nstart * d, hx.begin() + qx);
        for (size_t c = 0; c < nc; c++) {
            const double* lo = lower + ((size_t)j * nc + c) * CARMA_MAX_DIM;
            const double* hi = upper + ((size_t)j * nc + c) * CARMA_MAX_DIM;
            double* b = hb.data() + ((size_t)k * nc + c) * 2 * MAX_D;
            std::copy(lo, lo + d, b);
            std::copy(hi, hi + d, b + MAX_D);
        }
        qrow += nc * jb.nstart;
        qx += nc * jb.nstart * d;
    }
    if (!cuda_ok(cudaSetDevice(m->device), "cudaSetDevice")) return CARMA_ERR_CUDA;
    // scratch_in: [ x0 | bounds | jobs | per_curve | curves | order ]   scratch_out: [ x | f | nfev | queue head | nit ]
    const size_t nb = (size_t)njobs * nc;
    const size_t in_bytes = (xdoubles + hb.size()) * sizeof(double) + (size_t)njobs * (sizeof(MleJob) + sizeof(unsigned long long)) +
                            nc * (sizeof(MleCurve) + sizeof(int));
    const size_t out_bytes = (xdoubles + total + nb + 1) * sizeof(double) + nb * sizeof(int);
    if (!m->scratch_in.reserve(in_bytes) || !m->scratch_out.reserve(out_bytes)) return CARMA_ERR_CUDA;
    double* din = (double*)m->scratch_in.p;
    double* d_b = din + xdoubles;
    MleJob* d_jobs = (MleJob*)(d_b + hb.size());
    unsigned long long* d_pc = (unsigned long long*)(d_jobs + njobs);
    MleCurve* d_curve = (MleCurve*)(d_pc + njobs);
    int* d_order = (int*)(d_curve + nc);
    double* dout = (double*)m->scratch_out.p;
    double* d_f = dout + xdoubles;
    unsigned long long* d_nfev = (unsigned long long*)(d_f + total);
    unsigned long long* d_next = d_nfev + nb;
    int* d_nit = (int*)(d_next + 1);
    cudaStream_t st = 0;
    if (!cuda_ok(cudaMemcpyAsync(din, hx.data(), xdoubles * sizeof(double), cudaMemcpyHostToDevice, st), "H2D x0") ||
        !cuda_ok(cudaMemcpyAsync(d_b, hb.data(), hb.size() * sizeof(double), cudaMemcpyHostToDevice, st), "H2D bounds") ||
        !cuda_ok(cudaMemcpyAsync(d_jobs, dj.data(), njobs * sizeof(MleJob), cudaMemcpyHostToDevice, st), "H2D jobs") ||
        !cuda_ok(cudaMemcpyAsync(d_pc, per_curve.data(), njobs * sizeof(unsigned long long), cudaMemcpyHostToDevice, st), "H2D per_curve") ||
        !cuda_ok(cudaMemcpyAsync(d_curve, hc.data(), nc * sizeof(MleCurve), cudaMemcpyHostToDevice, st), "H2D curves") ||
        !cuda_ok(cudaMemcpyAsync(d_order, corder.data(), nc * sizeof(int), cudaMemcpyHostToDevice, st), "H2D curve order") ||
        !cuda_ok(cudaMemsetAsync(d_nfev, 0, (nb + 1) * sizeof(double) + nb * sizeof(int), st), "memset counters"))
        return CARMA_ERR_CUDA;
    MleDevParams mp{};
    mp.maxiter = o.maxiter; mp.history = o.history; mp.max_backtrack = o.max_backtrack;
    mp.gtol = o.gtol; mp.ftol = o.ftol; mp.fd_eps = o.fd_eps;
    mp.series_in_smem = 0;
    mp.njobs = njobs;
    mp.total = total;
    MleMulti mm{};
    mm.dt = m->d_dt; mm.y = m->d_y; mm.e2 = m->d_e2; mm.off = m->d_off;
    mm.order = d_order; mm.curve = d_curve; mm.per_curve = d_pc; mm.ncurves = nc;
    const size_t smem = (size_t)ML_WARPS * (ML_AREA + ML_LU) * sizeof(double);
    if (!cuda_ok(launch_lbfgs<true>(SeriesView{}, mp, d_jobs, din, d_b, dout, d_f, d_nit, d_nfev, d_next, mm, smem, st),
                 "lbfgs_kernel launch"))
        return CARMA_ERR_CUDA;
    std::vector<double> rx(xdoubles), rf(total);
    std::vector<int> rnit(nb);
    std::vector<unsigned long long> rnfev(nb);
    if (!cuda_ok(cudaMemcpyAsync(rx.data(), dout, xdoubles * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H x") ||
        !cuda_ok(cudaMemcpyAsync(rf.data(), d_f, total * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H f") ||
        !cuda_ok(cudaMemcpyAsync(rnit.data(), d_nit, nb * sizeof(int), cudaMemcpyDeviceToHost, st), "D2H nit") ||
        !cuda_ok(cudaMemcpyAsync(rnfev.data(), d_nfev, nb * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st), "D2H nfev") ||
        !cuda_ok(cudaStreamSynchronize(st), "multi mle sync"))
        return CARMA_ERR_CUDA;
    for (int k = 0; k < njobs; k++) {
        const int j = order[k];
        const MleJob& mj = dj[k];
        std::copy(rx.begin() + mj.x_off, rx.begin() + mj.x_off + mj.nstart * mj.d, x_out + x_first[j]);
        std::copy(rf.begin() + mj.first, rf.begin() + mj.first + mj.nstart, f_out + f_first[j]);
        for (size_t c = 0; c < nc; c++) {
            if (nit_out) nit_out[(size_t)j * nc + c] = rnit[(size_t)k * nc + c];
            if (nfev_out) nfev_out[(size_t)j * nc + c] = (long long)rnfev[(size_t)k * nc + c];
        }
    }
    return CARMA_OK;
}
