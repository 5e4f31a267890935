/* carma_b200.h -- C ABI of the B200-native CARMA(p,q) Kalman log-likelihood / PT-MCMC path.
 *
 * This is the drop-in boundary for ONE hot path of brandonckelly/carma_pack:
 *   KalmanFilterp::Reset/Update/Filter/Predict      (src/kfilter.cpp:138-337, src/include/kfilter.hpp:126-132)
 *   CARMA_Base<>::LogDensity / LogPrior / bounds     (src/include/carpack.hpp:118-191)
 *   CARp/CARMA/ZCARMA theta -> (roots, MA, sigma^2)  (src/carpack.cpp:137-172, 314-409, 522-580, 687-698)
 *   AdaptiveMetro / ExchangeStep / Sampler::Run      (src/steps.cpp:24-131, src/include/steps.hpp:318-362,
 *                                                     src/samplers.cpp:57-124, src/carmcmc.cpp:30-177)
 * Each entry point cites the reference interface it replaces.  Plain pointers and sizes only:
 * no C++ types, no torch types, no exceptions.  All arithmetic is FP64 on the GPU; there is no
 * CPU fallback: every compute entry point returns CARMA_ERR_CUDA when no device is usable.
 *
 * Conventions
 *   - return value: 0 = CARMA_OK, otherwise a CARMA_ERR_* code; carma_last_error() gives text.
 *   - -inf / NaN log-densities are VALUES (prior violated, singular model), never errors
 *     (reference: src/include/carpack.hpp:134-138, 154-164; src/steps.cpp:41-46).
 *   - `*_dev` entry points take DEVICE pointers and a cudaStream_t (passed as void*), do no
 *     synchronisation and no host<->device copies; the plain variants take HOST pointers,
 *     copy in/out and synchronise before returning.
 *   - a series object owns device scratch buffers: calls on ONE object must not run concurrently
 *     (host calls from several threads, or `*_dev` calls on different streams without ordering);
 *     different objects are independent.  carma_last_error() is thread-local.
 *   - theta rows are laid out as the reference's value_ vectors (src/include/carpack.hpp:131-176):
 *       CAR1  : [sigma_y, measerr_scale, mu, log(omega)]                        d = 4
 *       CARp  : [sigma_y, measerr_scale, mu, log-quad AR terms (p)]             d = 3+p
 *       CARMA : [..., log-quad AR terms (p), log-quad MA terms (q)]             d = 3+p+q
 *       ZCAR  : as CARp (the reference evaluates ZCAR as CAR(p), see DESIGN.md) d = 3+p
 *       ZCARMA: [..., AR terms (p), logit(kappa_normalised)]                    d = 4+p
 */
#ifndef CARMA_B200_H
#define CARMA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CARMA_B200_ABI_VERSION 5

enum {
    CARMA_OK = 0,
    CARMA_ERR_ARG = 1,    /* bad argument (null pointer, p out of range, unsorted times, ...) */
    CARMA_ERR_CUDA = 2,   /* CUDA runtime/driver failure, or no device */
    CARMA_ERR_ALLOC = 3,  /* host or device allocation failure */
    CARMA_ERR_START = 4   /* no finite starting value found within max_start_attempts */
};

/* model classes of src/include/carpack.hpp:251-461 */
enum {
    CARMA_KIND_CAR1 = 0,
    CARMA_KIND_CARP = 1,
    CARMA_KIND_CARMA = 2,
    CARMA_KIND_ZCAR = 3,
    CARMA_KIND_ZCARMA = 4
};

/* flags for the log-density entry points */
enum {
    CARMA_IGNORE_BOUNDS = 1u, /* SetMLE(true): skip CheckPriorBounds (src/include/carpack.hpp:180, 230) */
    CARMA_LOGLIK_ONLY = 2u    /* do not add LogPrior (new; the reference always adds it, SURVEY Q2) */
};

#define CARMA_MAX_P 7
#define CARMA_N_SLOTS 4   /* pipeline slots of a series for the *_async / mle entry points */
#define CARMA_MAX_DIM (3 + 2 * CARMA_MAX_P)   /* >= the parameter count of every model: 3+p+q, 4+p (ZCARMA), 3 (CAR1) */

/* prior / bounds of CARMA_Base::SetPrior (src/include/carpack.hpp:201-207) and the ZCARMA kappa
 * bounds (src/include/carpack.hpp:413-419) */
typedef struct carma_prior {
    double max_stdev;
    double max_freq;
    double min_freq;
    double kappa_low;
    double kappa_high;
    double measerr_dof; /* 50, src/include/carpack.hpp:63 */
} carma_prior_t;

/* One light curve resident in HBM (time, y, yerr of KalmanFilter<>::time_/y_/yerr_,
 * src/include/kfilter.hpp:186-190).  Opaque. */
typedef struct carma_series* carma_series_t;
/* A ragged batch of light curves (CSR offsets) resident in HBM. Opaque. */
typedef struct carma_multi_series* carma_multi_series_t;

const char* carma_last_error(void);
int carma_abi_version(void);
int carma_device_count(int* count);

/* ---- series -------------------------------------------------------------------------------
 * Replaces the data members / init() of KalmanFilter<> (src/include/kfilter.hpp:43-76) and the
 * copies held by CARMA_Base (src/include/carpack.hpp:66-68).  Times must be strictly increasing
 * (the reference sorts and de-duplicates in init(); the Python CarmaModel already guarantees it,
 * src/carmcmc/carma_pack.py:32-43).  Host pointers. */
int carma_series_create(const double* time, const double* y, const double* yerr, size_t ny, int device,
                        carma_series_t* out);
int carma_series_destroy(carma_series_t s);
int carma_series_length(carma_series_t s, size_t* ny);
/* SetPrior(10*sqrt(var(y))) with var = population variance as RunCarmaSampler does
 * (src/carmcmc.cpp:85-89) when population_var != 0, else the N-1 variance of the class
 * constructors (src/include/carpack.hpp:71). */
int carma_series_default_prior(carma_series_t s, int population_var, carma_prior_t* out);

/* ---- hot path: batched CARMA_Base::LogDensity ----------------------------------------------
 * Replaces n calls of Parameter<arma::vec>::LogDensity(theta) (src/include/carpack.hpp:131-176,
 * called from src/steps.cpp:39 and src/boost_python_wrapper.cpp:51-72 getLogDensity).
 * theta: n x d row-major; logpost: n. */
int carma_loglik_batch_dev(carma_series_t s, int kind, int p, int q, const carma_prior_t* prior, size_t n,
                           const double* d_theta, double* d_logpost, unsigned flags, void* stream);
int carma_loglik_batch(carma_series_t s, int kind, int p, int q, const carma_prior_t* prior, size_t n,
                       const double* theta, double* logpost, unsigned flags);
/* Pipelined form of carma_loglik_batch for callers that evaluate batch after batch from host memory
 * (optimisers, samplers driven from the host): enqueue H2D + kernel + D2H on one of CARMA_N_SLOTS internal slots
 * (slot = 0 .. CARMA_N_SLOTS-1, each with its own stream and device buffers) and return at once; the copies of one slot
 * overlap the kernel of the other.  The host buffers must stay valid (and should be pinned) until
 * carma_loglik_batch_wait(s, slot) returns. */
int carma_loglik_batch_async(carma_series_t s, int kind, int p, int q, const carma_prior_t* prior, size_t n,
                             const double* theta, double* logpost, unsigned flags, int slot);
int carma_loglik_batch_wait(carma_series_t s, int slot);
/* CARMA_Base::getLogPrior (src/include/carpack.hpp:221-225): host-side scalar helper. */
int carma_log_prior(int kind, int p, const double* theta, const carma_prior_t* prior, double* out);

/* ---- posterior post-processing ---------------------------------------------------------------
 * Replaces the per-sample Python loops of CarmaSample._ar_roots / _ar_coefs / _ma_coefs / _sigma_noise
 * (src/carmcmc/carma_pack.py:439-546): n theta rows (an MCMC trace) -> n rows of width 6p + 2,
 *   [ AR roots (re, im) x p | AR polynomial coefficients p+1, highest power first | MA coefficients p (beta_0 = 1, zero
 *     beyond q) | sigma of the driving noise | PSD widths p (-Re w / 2pi) | PSD centroids p (|Im w| / 2pi) ],
 * one thread per row, no light curve needed.  prior: only its kappa bounds are read (ZCARMA); may be NULL otherwise. */
int carma_derived_params(int kind, int p, int q, const carma_prior_t* prior, size_t n, const double* theta, double* out,
                         int device);
int carma_derived_params_dev(int kind, int p, int q, const carma_prior_t* prior, size_t n, const double* d_theta,
                             double* d_out, void* stream);
/* Pointwise percentiles of the CARMA power spectrum over the samples of each of ncurves groups (survey form of
 * CarmaSample.psd_credible_band / plot_power_spectrum, carma_pack.py:548-612).  theta: ncurves*nsamples rows of d,
 * curve-major.  freq: freq_rows (1 or ncurves) rows of nfreq frequencies.  pct: npct values in [0, 100].
 *   PSD(f) = sigma^2 |sum_{k<=q} beta_k (2 pi i f)^k|^2 / prod_k |2 pi i f - w_k|^2
 * with the roots w, MA coefficients beta and sigma of carma_derived_params (CAR1: sigma^2 = 2 omega var).
 * out[(c*npct + j)*nfreq + f] = np.percentile(psd[c, :, f], pct[j]) (method "linear"), bitwise, of the values returned in
 * psd_out (NULL, or ncurves*nsamples*nfreq: psd_out[(c*nsamples + s)*nfreq + f]).  A theta row whose PSD is not finite
 * (NaN or inf in theta, a failed derivation) gives NaN there and NaN percentiles in its curve's columns.  An output
 * depends only on its curve's theta rows, frequency row and prior.  priors: ncurves entries, only the kappa bounds read
 * (required for ZCARMA, else may be NULL).  Columns of up to 16384 samples are sorted in shared memory; longer ones are
 * selected by a radix select over a global scratch column (CARMA_PSD_GLOBAL_SELECT=1 forces that path).
 * Curves go in chunks whose device footprint stays within 4 GiB: peak 8 B * (B * (nsamples * (d + 22 + nfreq * (1 +
 * [psd_out])) + npct * nfreq + [freq_rows > 1] nfreq) + npct + nfreq) for a chunk of B curves.  _dev: device pointers, all
 * curves in one pass with 8 B * ncurves * nsamples * (1 + 3p + [long columns] nfreq) of stream-ordered scratch; pct is
 * not checked on the host there, and a percentile outside [0, 100] gives NaN. */
int carma_psd_quantiles(int kind, int p, int q, const carma_prior_t* priors, size_t ncurves, size_t nsamples,
                        const double* theta, const double* freq, size_t freq_rows, size_t nfreq,
                        const double* pct, size_t npct, double* out, double* psd_out, int device);
int carma_psd_quantiles_dev(int kind, int p, int q, const carma_prior_t* d_priors, size_t ncurves, size_t nsamples,
                            const double* d_theta, const double* d_freq, size_t freq_rows, size_t nfreq,
                            const double* d_pct, size_t npct, double* d_out, double* d_psd_out, void* stream);
/* MCMCSample.effective_samples for every column of every series: x (nseries, n, k) row-major, ess (nseries, k).
 * r = x - mean, ac[j] = sum_i r_i r_{i+j} / max(sum r^2, 1e-300), tau = 1 + 2 sum ac[j] while ac[j] > 0.05,
 * ess = n / tau; lags are computed one at a time up to the cutoff, in a fixed summation order.  A column whose values
 * are all equal gets ess = n (its residuals are zero). */
int carma_effective_samples(size_t nseries, size_t n, size_t k, const double* x, double* ess, int device);
int carma_effective_samples_dev(size_t nseries, size_t n, size_t k, const double* d_x, double* d_ess, void* stream);

/* ---- maximum-likelihood fits from many starts ----------------------------------------------
 * Replaces the ntrials scipy L-BFGS-B runs of CarmaModel.get_mle / _get_mle_single / _carma_loglik
 * (src/carmcmc/carma_pack.py:92-129, 195-260): projected L-BFGS with forward-difference gradients over a box,
 * all nstart starts in lock-step, every function value of an iteration evaluated in one batched launch.
 * The objective is  -LogDensity(theta)  with `flags` (CARMA_IGNORE_BOUNDS = SetMLE(true), carma_pack.py:242).
 * lower/upper: d entries, +-infinity allowed.  Outputs: x_out[nstart][d], f_out[nstart] (1e300 where no finite
 * value was ever found); nit_out / nfev_out may be NULL.  slot: the stream slot of the series to use (0 .. CARMA_N_SLOTS-1), so
 * fits driven from different host threads on different series handles overlap on the GPU. */
typedef struct carma_mle_opts {
    int maxiter;        /* 1000: L-BFGS-B stops on maxfun = 15000 evaluations, i.e. ~1000 finite-difference gradients at d = 14 */
    int history;        /* L-BFGS pairs kept, 8 */
    int max_backtrack;  /* Armijo halvings per iteration, 25 */
    int reserved;
    double gtol;        /* projected-gradient infinity norm, 1e-5 (scipy pgtol) */
    double ftol;        /* relative decrease, 2.2e-9 (scipy factr * eps) */
    double fd_eps;      /* forward-difference step, 1e-8 (scipy approx_grad epsilon) */
} carma_mle_opts_t;
void carma_mle_default_opts(carma_mle_opts_t* o);
/* The optimiser core on a caller-supplied objective (host code only, no GPU involved): fn evaluates n points
 * (theta: n x d, row-major) into f and returns 0 on success; non-finite values count as +infinity.  This is the
 * loop carma_mle_batch runs with -LogDensity as the objective; exported so that it can be exercised on its own. */
typedef int (*carma_objective_fn)(const double* theta, size_t n, size_t d, double* f, void* user);
int carma_lbfgs_batch(carma_objective_fn fn, void* user, size_t d, size_t nstart, const double* x0,
                      const double* lower, const double* upper, const carma_mle_opts_t* opts, double* x_out,
                      double* f_out, int* nit_out, long long* nfev_out);
int carma_mle_batch(carma_series_t s, int kind, int p, int q, const carma_prior_t* prior, unsigned flags,
                    size_t nstart, const double* x0, const double* lower, const double* upper,
                    const carma_mle_opts_t* opts, double* x_out, double* f_out, int* nit_out, long long* nfev_out,
                    int slot);
/* The same fits with the optimiser itself on the device (one kernel launch per call): a warp owns a start, its lanes
 * evaluate the trial points of a round (the d difference points of a gradient, the step sizes of a backtracking
 * round) concurrently, lane 0 runs the L-BFGS arithmetic.  Same algorithm, options and outputs as carma_mle_batch
 * (history <= 8) -- x_out, f_out and nit_out are bitwise those of carma_mle_batch, nfev_out is larger (more step
 * sizes tried per round); an iteration costs one evaluation of latency instead of a launch, two copies and a
 * synchronise, and no start waits for another.  nit_out: the largest iteration count over the starts. */
int carma_mle_batch_device(carma_series_t s, int kind, int p, int q, const carma_prior_t* prior, unsigned flags,
                           size_t nstart, const double* x0, const double* lower, const double* upper,
                           const carma_mle_opts_t* opts, double* x_out, double* f_out, int* nit_out,
                           long long* nfev_out, int slot);
/* Several models fitted in ONE launch (choose_order, carma_pack.py:131-192: every (p,q) of the grid from `ntrials`
 * starts): the starts of all jobs form one queue on the device, served heaviest model first, each start fitted by a
 * warp exactly as carma_mle_batch_device fits it (a start's result does not depend on what else is in the launch).
 * x0 / x_out: the jobs' rows one after the other, job j holding nstart_j rows of d_j doubles; f_out: nstart_j values
 * per job in the same order; lower / upper: njobs rows of CARMA_MAX_DIM doubles (the first d_j used); nit_out /
 * nfev_out: njobs entries (may be NULL). */
typedef struct carma_mle_job {
    int kind, p, q;
    unsigned flags;
    carma_prior_t prior;
    size_t nstart;
} carma_mle_job_t;
int carma_mle_grid_device(carma_series_t s, int njobs, const carma_mle_job_t* jobs, const double* x0,
                          const double* lower, const double* upper, const carma_mle_opts_t* opts, double* x_out,
                          double* f_out, int* nit_out, long long* nfev_out, int slot);

/* carma_mle_grid_device over every curve of a multi-series, in ONE launch (survey-scale get_mle / choose_order): job j
 * fits jobs[j].nstart starts PER CURVE.  jobs[j].prior is ignored; the per-curve priors come from `priors` (ncurves
 * entries, or NULL = the population-variance defaults).  Per job, curve-major: x0 / x_out ncurves*nstart_j rows of d_j
 * doubles, f_out ncurves*nstart_j values, lower / upper ncurves rows of CARMA_MAX_DIM doubles; the jobs one after the
 * other.  nit_out / nfev_out: njobs*ncurves entries (largest iteration count / total evaluations of that curve's starts;
 * may be NULL).  A fit reads its curve as a carma_series_t built from that curve would hold it (its own longest gap
 * included), so a start's result depends only on (job, curve, x0 row, bounds row, prior): it equals what
 * carma_mle_batch_device returns for that curve alone.  Blocking; uses the multi-series' own scratch buffers. */
int carma_multi_mle_grid_device(carma_multi_series_t m, int njobs, const carma_mle_job_t* jobs,
                                const carma_prior_t* priors, const double* x0, const double* lower,
                                const double* upper, const carma_mle_opts_t* opts, double* x_out,
                                double* f_out, int* nit_out, long long* nfev_out);

/* ---- multi light-curve batch (one theta per curve) ----------------------------------------
 * The reference loops over objects in Python; this is the survey-scale form of the same
 * LogDensity call.  offsets: ncurves+1 (CSR), host pointers. priors: ncurves or NULL (defaults). */
int carma_multi_series_create(const double* time, const double* y, const double* yerr, const int64_t* offsets,
                              size_t ncurves, int device, carma_multi_series_t* out);
int carma_multi_series_destroy(carma_multi_series_t m);
int carma_multi_series_default_priors(carma_multi_series_t m, int population_var, carma_prior_t* out /* ncurves */);
/* Synthetic survey generated in HBM (BASELINE config 5 at full size without a host round trip): ncurves
 * light curves of ny points drawn from the model theta_true, the recipe of the reference's Python generator
 * (carma_process, src/carmcmc/carma_pack.py:1148-1259: innovations form of the noise-free filter; sampling
 * gaps dt_min + |Cauchy| truncated at dt_max as in cpp_tests/generate_test_data.py:17) plus N(0, yerr^2)
 * measurement noise.  Curve c uses Philox chain curve_offset + c, so a survey does not depend on how it is
 * sharded across GPUs.  prior: bounds used by the theta transform (NULL = wide open; kappa in (0, 1/dt_min)).
 * The handle is an ordinary carma_multi_series_t (default priors and starting-value statistics included). */
int carma_multi_series_simulate(size_t ncurves, size_t ny, int kind, int p, int q, const double* theta_true,
                                const carma_prior_t* prior, double yerr, double dt_min, double dt_max, uint64_t seed,
                                uint32_t curve_offset, int device, carma_multi_series_t* out);
/* Copy curve `curve` back to the host (time measured from 0). capacity: length of the three arrays. */
int carma_multi_series_get_curve(carma_multi_series_t m, size_t curve, double* time, double* y, double* yerr,
                                 size_t capacity, size_t* ny_out);
/* Per-curve statistics of a multi-series (what the optimiser's box and the default priors are built from): mean and
 * population / N-1 variance of y, shortest, median and longest sampling gap, time span, number of points. */
typedef struct carma_curve_stats {
    double y_mean, y_var_pop, y_var_sample, min_dt, median_dt, tspan, dt_max;
    int64_t ny;
} carma_curve_stats_t;
int carma_multi_series_curve_stats(carma_multi_series_t m, carma_curve_stats_t* out /* ncurves */);
int carma_multi_loglik_dev(carma_multi_series_t m, int kind, int p, int q, const carma_prior_t* d_priors,
                           const double* d_theta /* ncurves x d */, double* d_logpost, unsigned flags, void* stream);
int carma_multi_loglik(carma_multi_series_t m, int kind, int p, int q, const carma_prior_t* priors,
                       const double* theta, double* logpost, unsigned flags);
/* KalmanFilterp::Filter + GetMean()/GetVar() (src/kfilter.cpp:138-215) of every curve with its own theta row, in one
 * launch: theta ncurves x d, priors ncurves entries or NULL (population-variance defaults), as carma_multi_loglik.
 * mean / var: the one-step predictive mean (without mu) and variance (with measerr_scale * yerr^2) at every point, in the
 * CSR order of the multi-series (total points); mean[first] = 0 and var[first] = Var(y) + scale * yerr_first^2 for every
 * curve, as carma_filter.  loglik (ncurves, may be NULL): bitwise what carma_multi_loglik returns for the same
 * arguments.  A row the transform rejects gives NaN mean / var for its curve and -inf loglik.  _dev: device pointers and
 * a stream, no synchronisation. */
int carma_multi_filter_dev(carma_multi_series_t m, int kind, int p, int q, const carma_prior_t* d_priors,
                           const double* d_theta, unsigned flags, double* d_mean, double* d_var, double* d_loglik,
                           void* stream);
int carma_multi_filter(carma_multi_series_t m, int kind, int p, int q, const carma_prior_t* priors, const double* theta,
                       unsigned flags, double* mean, double* var, double* loglik);
/* The numeric part of assess_fit (CarmaSample.assess_fit_values) for every curve, without the per-point outputs crossing
 * PCIe: with r = (y - mu - mean) / sqrt(var) the standardised one-step residuals, out holds per curve 3 + 2 nlags
 * doubles: loglik, mean(r), population std(r), acf(r)[1..nlags], acf(r^2)[1..nlags] (mean-subtracted, normalised by
 * lag 0).  1 <= nlags < the shortest curve's length. */
int carma_multi_assess_fit(carma_multi_series_t m, int kind, int p, int q, const carma_prior_t* priors,
                           const double* theta, unsigned flags, int nlags, double* out);
/* KalmanFilterp::Predict (src/kfilter.cpp:218-337) of every curve at its own query times: q_offsets ncurves+1 (CSR)
 * into tq, times absolute (on the axis the curves were created with), in any order, possibly equal to data times.
 * qmean (without mu) / qvar come back in the caller's order.  Forecasts, backcasts and interpolation as carma_predict;
 * a curve's queries cost O(ny - ip) filter steps each (ip: data points before the query). */
int carma_multi_predict(carma_multi_series_t m, int kind, int p, int q, const carma_prior_t* priors,
                        const double* theta, unsigned flags, const int64_t* q_offsets, const double* tq, double* qmean,
                        double* qvar);
/* KalmanFilter<>::Simulate (src/include/kfilter.hpp:135-184) of every curve of a multi-series at its own times, npaths
 * paths per curve, by Matheron's rule as carma_simulate: a draw of the noise-free process at the requested times given
 * the curve's data.  s_offsets (ncurves+1, CSR) and tsim as carma_multi_predict: absolute times, any order, possibly
 * repeated or equal to data times (a requested time equal to a data time follows it on the curve's own axis).
 * theta_rows = ncurves: every path of curve c uses row c; theta_rows = ncurves * npaths: path j of curve c uses row
 * c * npaths + j (posterior predictive: one posterior sample per path).  priors and flags as carma_multi_predict.
 * ysim[path * nsim_total + k] in the caller's order of tsim, mu included.  Draw (curve c, path j) uses the Philox
 * counters of carma_simulate's path j with block word curve_offset + c (0 in carma_simulate): curve c equals a one-curve
 * multi-series of that curve called with curve_offset = c, and path j does not depend on npaths.  A theta row the
 * transform rejects gives NaN for its curve (or path).  npaths == 0 or no times: a no-op.  Blocking; uses the
 * multi-series' scratch (one call per handle at a time).  Paths run in chunks of B whose scratch stays within 4 GiB:
 * peak scratch B * (8 round32(total) + 8 nsim_total (p + p(p+1)/2 + 4) + ncurves (sizeof constants + 4)) bytes plus
 * 20 nsim_total + 8 (ncurves + 1) for the sorted times, plus the theta rows and priors. */
int carma_multi_simulate(carma_multi_series_t m, int kind, int p, int q, const carma_prior_t* priors,
                         const double* theta, size_t theta_rows, unsigned flags, const int64_t* s_offsets,
                         const double* tsim, size_t npaths, uint64_t seed, uint32_t curve_offset, double* ysim);
/* Kalman smoother (Bryson-Frazier adjoint form, an extension: the reference has none) of every curve in one pass forward
 * and one backward, O(ny + nq) steps per curve.  theta, priors and flags as carma_multi_filter.  Per point, in the CSR
 * order of the multi-series (total entries each), means without mu:
 *   mean / var:         E[f(t_i) | y] and Var[f(t_i) | y] of the noise-free process given all of the curve's data;
 *   loo_mean / loo_var: the law of y_i given every other point of its curve (measurement noise included), so that
 *                       (y_i - mu - loo_mean) / sqrt(loo_var) is the standardised deleted residual.
 * loglik (ncurves): bitwise what carma_multi_loglik returns for the same arguments.  q_offsets / tq as carma_multi_predict
 * (absolute times, any order; qmean / qvar in the caller's order), or both NULL for no queries: the smoothed process at
 * each query time (a data time gives that point's smoothed value, a time past the last point the forecast).  Any output
 * pointer may be NULL.  A row the transform rejects gives NaN outputs for its curve and -inf loglik.  Blocking; uses the
 * multi-series' scratch (one call per handle at a time).  Curves run in chunks whose records stay within 4 GiB: peak
 * scratch 32 round32(total) + 32 round32(nq) + 8 round32(ncurves + 1) + 8 ncurves bytes for the outputs and sorted
 * queries, plus the records of
 * the largest chunk, 8 ((p + 2) ny + (p + 3) nq) bytes summed over its curves (one curve's records even when they
 * exceed the budget), plus the theta rows and priors. */
int carma_multi_smooth(carma_multi_series_t m, int kind, int p, int q, const carma_prior_t* priors, const double* theta,
                       unsigned flags, double* mean, double* var, double* loo_mean, double* loo_var, double* loglik,
                       const int64_t* q_offsets, const double* tq, double* qmean, double* qvar);
/* Curvature of every curve's log-density at its theta row (an extension: the reference's get_mle returns at most scipy's
 * approximate hess_inv), by central finite differences evaluated on the device.  The function is exactly the one
 * carma_multi_loglik evaluates for the row, with the same kind, p, q, priors (NULL: defaults) and flags, log-prior term
 * on measerr_scale included; with the survey fits' flags (0 for p == 1, else CARMA_IGNORE_BOUNDS) it is -fun of the fit.
 *   Steps: h_i = rel_step * s_i, s = (theta_0, theta_1, theta_0, 1, 1, ...): sigma_y and measerr_scale relative, mu in
 *   units of sigma_y, every coordinate from 3 on (log or logit) absolute.  rel_step <= 0 selects
 *   CARMA_HESS_DEFAULT_REL_STEP = 2^-13 (about eps^(1/4)); a power of two makes h_i exact.  NaN or inf is rejected.
 *   Stencil, d^2 + d + 1 points per curve: the centre f0, theta +- h_i e_i (f+i, f-i), and for i < j
 *   theta + h_i e_i + h_j e_j (f+ij) and theta - h_i e_i - h_j e_j (f-ij).
 *   Assembly: g_i = (f+i - f-i) / 2h_i;  H_ii = (f+i - 2 f0 + f-i) / h_i^2;
 *   H_ij = (f+ij - f+i - f+j + 2 f0 - f-i - f-j + f-ij) / (2 h_i h_j), formed for i < j and mirrored;
 *   cov = (-H)^-1 through a Cholesky factorisation of -H.
 * Outputs (any may be NULL): loglik (ncurves) = f0, bitwise carma_multi_loglik's; grad (ncurves x d); hess and cov
 * (ncurves x d x d, row-major); status (ncurves) one of CARMA_HESS_*:
 *   OK          every output valid;
 *   REJECTED    the centre row fails the transform or the prior bounds: loglik -inf, the rest NaN;
 *   NONFINITE   a stencil value or a step is not finite or zero (e.g. CAR(1) on its prior's frequency bound): loglik
 *               valid, grad / hess / cov NaN;
 *   NOT_NEGDEF  the Cholesky factorisation of -H fails: grad and hess valid, cov NaN.
 * There is no one-sided fallback at a bound: a fit on a bound has no interior curvature and the status says so.  An
 * output depends only on its curve's data, theta row and prior.  Blocking; uses the multi-series' scratch (one call per
 * handle at a time).  Curves run in chunks whose stencil values (8 (d^2 + d + 1) bytes per curve) stay within 4 GiB;
 * outputs take 8 ncurves (2 d^2 + d + 2) bytes more, plus the theta rows and priors. */
#define CARMA_HESS_DEFAULT_REL_STEP 1.220703125e-4   /* 2^-13 */
enum {
    CARMA_HESS_OK = 0,
    CARMA_HESS_REJECTED = 1,
    CARMA_HESS_NONFINITE = 2,
    CARMA_HESS_NOT_NEGDEF = 3
};
int carma_multi_hessian(carma_multi_series_t m, int kind, int p, int q, const carma_prior_t* priors,
                        const double* theta /* ncurves x d */, unsigned flags, double rel_step, double* loglik,
                        double* grad, double* hess, double* cov, int* status);
/* Importance sampling of every curve's posterior from its Laplace approximation N(theta_c, cov_c) (an extension: the
 * reference has only MCMC), with the Pareto k-hat reliability diagnostic and an equally weighted resample, so that a
 * survey can keep the Gaussian answer where it is good and run MCMC only where k-hat says it is not.  S = ndraws.
 *   Factor: the lower Cholesky factor L of cov_c, reading only its lower triangle (the upper one is never read), in
 *   the fixed loop order s = cov_jj - sum_{k<j} L_jk^2, L_jj = sqrt(s), L_ij = (cov_ij - sum_{k<j} L_ik L_jk) / L_jj
 *   (i > j, sums left to right, every product and difference rounded on its own); log|L| = sum_i log L_ii.
 *   Draw j: coordinate pair k takes (u0, u1) = uniforms2(seed, j, STREAM_LAPLACE = 6, k, curve_offset + c) (Philox
 *   counters laid out as carma_multi_simulate's (path, point, curve)); r = sqrt(-2 log u0), z_2k = r cos(2 pi u1),
 *   z_2k+1 = r sin(2 pi u1) (the second is dropped when d is odd).  Row: s_i = sum_{k<=i} L_ik z_k accumulated left to
 *   right from 0, theta_i = theta_c,i + s_i, each product and sum rounded on its own (no contraction).
 *   logq = -1/2 sum_k z_k^2 - log|L| - (d/2) log(2 pi), the proposal's log-density of the row.
 *   logpost is bitwise what carma_multi_loglik returns for the row with the same kind, p, q, priors (NULL: defaults)
 *   and flags, log-prior included.
 *   Weights: lw_j = logpost_j - logq_j where logpost_j is finite, else -inf; a_j = lw_j - max_j lw_j, e_j = exp(a_j).
 *   ess = (sum e)^2 / sum e^2, the weight ESS of the raw weights.
 *   khat, the generalised-Pareto shape of the largest weights (Vehtari et al., PSIS; ArviZ _psislw / _gpdfit, r_eff = 1):
 *     M = ceil(min(0.2 S, 3 sqrt(S))); cut = max(a_(S-M-1), log DBL_MIN), a_(.) ascending and 0-based (S < 2: +inf);
 *     the tail is {a_j > cut}, n members; n <= 4: khat = +inf;
 *     else x = ascending(exp(a_j) - exp(cut)) over the tail, m = 30 + floor(sqrt(n)), and for i = 1 .. m
 *       b_i = (1 - sqrt(m / (i - 1/2))) / (3 x[floor(n/4 + 1/2) - 1]) + 1 / x[n-1],
 *       k_i = mean_t log1p(-b_i x_t),  L_i = n (log(-b_i / k_i) - k_i - 1),  w_i = 1 / sum_l exp(L_l - L_i);
 *     the w_i < 10 DBL_EPSILON are dropped and the rest renormalised; bbar = sum_i w_i b_i, k = mean_t log1p(-bbar x_t);
 *     khat = (n k + 5) / (n + 10).  khat <= 0.7: the importance sample is reliable; above, it is not (run MCMC).
 *   resample (systematic, from the raw weights): u = the first uniform of uniforms2(seed, 0, STREAM_LAPLACE_RESAMPLE =
 *   7, 0, curve_offset + c), C_j = e_0 + ... + e_j, T = C_{S-1}; resample[c, i] = the first j with C_j > ((i + u) / S) T,
 *   capped at S - 1: draws[c, resample[c, i]] is an equally weighted sample of the posterior.
 * Every reduction runs in a fixed order, so every output is deterministic.  A draw depends only on (seed, j,
 * curve_offset + c, theta_c, cov_c): batch mates, ndraws (a call with fewer draws gives a prefix of draws / logpost /
 * logq), chunking and curve subsets with a matching curve_offset change no bit.
 * Outputs (any may be NULL): draws (ncurves x ndraws x d), logpost, logq, resample (ncurves x ndraws), ess, khat,
 * status (ncurves) one of CARMA_LAPLACE_*, each curve's independent of the others':
 *   OK         every output valid;
 *   BAD_COV    theta_c or the lower triangle of cov_c is not finite, or the factorisation fails (s <= 0): draws,
 *              logpost, logq and khat NaN, ess 0, resample -1;
 *   NO_WEIGHT  no draw has a finite logpost (e.g. the proposal lies outside the prior): draws and logq valid, logpost
 *              as evaluated, ess 0, khat NaN, resample -1.
 * CARMA_ERR_ARG before any CUDA call: m, theta or cov NULL, an invalid (kind, p, q), ndraws 0 or above
 * CARMA_LAPLACE_MAX_DRAWS, curve_offset + ncurves > 2^32.  Blocking; uses the multi-series' scratch (one call per handle
 * at a time).  Curves run in chunks whose scratch, 8 S (d + 3) + 4 S + 8 d^2 + 32 bytes per curve, stays within 4 GiB
 * (CARMA_MULTI_LAPLACE_BUDGET bytes, read at every call); theta, cov and the priors of all curves take 8 ncurves
 * (d^2 + d) bytes and the priors more. */
#define CARMA_LAPLACE_MAX_DRAWS (1u << 20)
enum { CARMA_LAPLACE_OK = 0, CARMA_LAPLACE_BAD_COV = 1, CARMA_LAPLACE_NO_WEIGHT = 2 };
int carma_multi_laplace(carma_multi_series_t m, int kind, int p, int q, const carma_prior_t* priors /* NULL: defaults */,
                        const double* theta /* ncurves x d: centres */, const double* cov /* ncurves x d x d */,
                        unsigned flags, size_t ndraws, uint64_t seed, uint32_t curve_offset,
                        double* draws /* ncurves x ndraws x d */, double* logpost /* ncurves x ndraws */,
                        double* logq /* ncurves x ndraws */, int32_t* resample /* ncurves x ndraws */,
                        double* ess /* ncurves */, double* khat /* ncurves */, int* status /* ncurves */);

/* ---- one very long light curve: temporally parallel (associative-scan) form of the same LogDensity ----
 * Replaces the strictly sequential Filter() loop (src/include/kfilter.hpp:126-132) when there is a single
 * series and few theta rows, i.e. no batch parallelism (BASELINE config 5, ny = 10^6).  Same value as
 * carma_loglik_batch up to floating-point re-association.  chunk: points per thread (0 = default 128). */
int carma_loglik_scan_dev(carma_series_t s, int kind, int p, int q, const carma_prior_t* prior, size_t n,
                          const double* d_theta, double* d_logpost, unsigned flags, int chunk, void* stream);
int carma_loglik_scan(carma_series_t s, int kind, int p, int q, const carma_prior_t* prior, size_t n,
                      const double* theta, double* logpost, unsigned flags, int chunk);

/* ---- explicit-parameter filter: KalmanFilterp / KalmanFilter1 ------------------------------
 * Replaces KalmanFilterp(t,y,yerr,sigsqr,omega,ma).Filter() + GetMean()/GetVar()
 * (src/include/kfilter.hpp:303-334, 116-117; src/kfilter.cpp:138-215).  omega_reim: p complex roots as
 * (re,im) pairs in any order; ma: p coefficients.  The stored series is used as  y - mu  with
 * yerr*sqrt(measerr_scale) (pass mu=0, measerr_scale=1 for the raw class semantics).  For p == 1
 * this is KalmanFilter1 with omega_reim = (-omega, 0).  Outputs are host arrays of length ny. */
int carma_filter(carma_series_t s, double sigsqr, const double* omega_reim, const double* ma, int p,
                 double measerr_scale, double mu, double* mean, double* var);
/* Replaces nq calls of KalmanFilterp::Predict(time) (src/kfilter.cpp:218-286 with
 * InitializeCoefs/UpdateCoefs 290-337): forecasting, backcasting and interpolation. */
int carma_predict(carma_series_t s, double sigsqr, const double* omega_reim, const double* ma, int p,
                  double measerr_scale, double mu, const double* tq, size_t nq, double* qmean, double* qvar);

/* Replaces KalmanFilter<>::Simulate (src/include/kfilter.hpp:135-184): draws of the process at the times tsim (any
 * order; may coincide with data times) GIVEN the data, for `npaths` independent paths in one call:
 * ysim[path * nsim + i].  The reference draws one point at a time, inserts it into the series and re-predicts
 * (O(nsim (ny + nsim)) filter steps); here every path is an unconditional draw on the merged time grid plus the
 * conditional mean of the residual data (Matheron's rule): same joint law, O(ny + nsim) work per path, no per-point
 * allocation or host round trip.  Random numbers: Philox4x32-10 addressed by (seed, path, merged index).  The AR roots
 * must be distinct and closed under complex conjugation. */
int carma_simulate(carma_series_t s, double sigsqr, const double* omega_reim, const double* ma, int p,
                   double measerr_scale, double mu, const double* tsim, size_t nsim, uint64_t seed, size_t npaths,
                   double* ysim);

/* ---- parallel-tempering MCMC, fully on device ---------------------------------------------
 * Replaces RunCarmaSampler / RunCar1Sampler (src/carmcmc.cpp:30-177): temperature ladder,
 * AdaptiveMetro (src/steps.cpp:24-107), CholUpdateR1 (111-131), ExchangeStep
 * (src/include/steps.hpp:318-362) and Sampler::Run (src/samplers.cpp:57-115), for n_ensembles
 * independent ensembles on one series.  Random numbers are Philox4x32-10 addressed by
 * (seed, stream, chain = (ensemble_offset+e)*ntemps + temperature, iteration, slot). */
typedef struct carma_pt_opts {
    int nsamples;            /* stored samples of the coolest chain */
    int burnin;              /* iterations before sampling; adaptation stops after burnin */
    int thin;
    int ntemps;              /* nwalkers of RunCarmaSampler */
    double tmax;             /* 100  (src/carmcmc.cpp:92) */
    int dof;                 /* 8    (src/carmcmc.cpp:139), must be even */
    double target_rate;      /* 0.25 (src/carmcmc.cpp:141) */
    double gamma;            /* 2/3  (src/steps.cpp:29) */
    uint64_t seed;
    uint32_t ensemble_offset; /* global index of the first ensemble (multi-GPU sharding) */
    int max_start_attempts;  /* cap of the redraw-until-finite loop (src/carpack.cpp:182-227) */
    int order_mode;          /* 0 = reference step order (src/carmcmc.cpp:147-157), evaluated as a
                                skewed pipeline that is exactly equivalent; 1 = all temperatures
                                propose concurrently, then sequential exchanges (valid PT, not
                                decision-identical to the reference) */
    int record_trace;        /* 0/1: fill the trace arrays of carma_pt_run (parity tests) */
} carma_pt_opts_t;

typedef struct carma_pt_trace_rec {
    double lp_prop;  /* LogDensity(proposal)            (exchange: log-posterior of the colder chain) */
    double lp_cur;   /* cached log-posterior before the step */
    double alpha;    /* acceptance probability (0 if non-finite, src/steps.cpp:41-46) */
    double u;        /* uniform used; NaN if none was drawn */
    int accepted;
    int pad;
} carma_pt_trace_rec_t;

void carma_pt_default_opts(carma_pt_opts_t* o);
/* init: d values (SetStartingValue, src/carpack.cpp:233-265) or NULL (StartingValue draws).
 * Host outputs: samples[n_ensembles][nsamples][d], logposts[n_ensembles][nsamples],
 * accept_rates[n_ensembles][ntemps] (may be NULL), exchange_rates[n_ensembles][ntemps] (may be NULL).
 * Trace outputs (NULL unless opts->record_trace): ram_trace/exch_trace[n_ensembles][iters][ntemps],
 * proposals[n_ensembles][iters][ntemps][d], iters = burnin + nsamples*thin. */
int carma_pt_run(carma_series_t s, int kind, int p, int q, const carma_prior_t* prior, const carma_pt_opts_t* opts,
                 size_t n_ensembles, const double* init, double* samples, double* logposts, double* accept_rates,
                 double* exchange_rates, carma_pt_trace_rec_t* ram_trace, carma_pt_trace_rec_t* exch_trace,
                 double* proposals);
/* Device-resident variant used by the benchmark: outputs stay in HBM, no sync. */
int carma_pt_run_dev(carma_series_t s, int kind, int p, int q, const carma_prior_t* prior,
                     const carma_pt_opts_t* opts, size_t n_ensembles, const double* d_init, double* d_samples,
                     double* d_logposts, double* d_accept_rates, double* d_exchange_rates, void* stream);

/* One PT-MCMC run per light curve of a ragged batch, n_ensembles independent ensembles per curve, in ONE
 * launch (every block stages its own curve).  The survey-scale form of RunCarmaSampler: the reference
 * would loop over objects in Python.  priors: ncurves entries or NULL (population-variance defaults).
 * Host outputs: samples[ncurves][n_ensembles][nsamples][d], logposts[ncurves][n_ensembles][nsamples],
 * accept_rates / exchange_rates[ncurves][n_ensembles][ntemps] (may be NULL).  Chain ids of the Philox
 * streams: ((ensemble_offset + curve*n_ensembles + e) * ntemps + temperature). */
int carma_multi_pt_run(carma_multi_series_t m, int kind, int p, int q, const carma_prior_t* priors,
                       const carma_pt_opts_t* opts, size_t n_ensembles, double* samples, double* logposts,
                       double* accept_rates, double* exchange_rates);

/* ---- starting values ------------------------------------------------------------------------
 * Replaces CAR1/CARp/CARMA/ZCARMA::StartingValue (src/carpack.cpp:38-83, 175-230, 416-477, 586-644): draws from the
 * starting-value law until LogDensity is finite (at most max_attempts times), on the device, with the Philox
 * stream (seed, chain) that carma_pt_run would use for that chain -- so a host-driven sampler built from the
 * step classes starts exactly where the on-device sampler would.  theta_out: d values; logpost_out: its
 * log-density.  Returns CARMA_ERR_START when no finite value was found. */
int carma_starting_value(carma_series_t s, int kind, int p, int q, const carma_prior_t* prior, uint64_t seed,
                         uint32_t chain, int max_attempts, double* theta_out, double* logpost_out);

/* ---- multi-GPU: gather of per-rank summaries (NCCL) -----------------------------------------
 * One process per GPU; units of work are partitioned with no data-path collective, and at the end every rank
 * contributes `count` doubles (per-model -loglik / AICc / theta-hat, or survey moments) and receives everybody's:
 * all[r * count + k] = local[k] of rank r.  Replaces the result return of the reference's process pool
 * (src/carmcmc/carma_pack.py:111-119).  nccl_comm is an ncclComm_t (passed as void*): either one the host already
 * has, or one made by carma_comm_init_rank from an id that rank 0 obtained with carma_comm_unique_id and sent to the
 * other ranks by any means (file, socket, MPI).  NCCL is loaded at first use; without it these return CARMA_ERR_CUDA. */
#define CARMA_COMM_ID_BYTES 128
int carma_comm_unique_id(char id[CARMA_COMM_ID_BYTES]);
int carma_comm_init_rank(int nranks, int rank, const char id[CARMA_COMM_ID_BYTES], int device, void** comm);
int carma_comm_destroy(void* comm);
int carma_gather_summaries(void* nccl_comm, const double* local, size_t count, double* all /* nranks x count */,
                           void* stream);
/* device-pointer variant: no copies, no synchronisation */
int carma_gather_summaries_dev(void* nccl_comm, const double* d_local, size_t count, double* d_all, void* stream);

/* ---- utilities ---------------------------------------------------------------------------- */
/* Saturating FP64 FMA micro-benchmark on `device`: returns sustained DFMA TFLOP/s (2 flops per
 * FMA).  Used by bench.py as the measured FP64 roofline denominator. */
int carma_fp64_peak_tflops(int device, double* tflops);
/* Philox4x32-10 block and the Student-t draw built on it, exported so tests can pin the device
 * RNG against the oracle bit for bit. */
int carma_philox_dev(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint64_t seed, uint32_t* out4);
int carma_tdist_dev(uint64_t seed, uint32_t chain, uint32_t iter, uint32_t j, int dof, double* out);

/* The branch-free transcendentals of the Kalman time loop (csrc/fast_math.cuh), evaluated element-wise on host
 * arrays so tests can bound their error against libm.  rate is in TABLE STEPS per unit time, as the loop holds it
 * (lambda * 64/ln2 for a decay, Im(omega) * 64/pi for a phase):
 *   out_exp      = exp(rate dt ln2/64)                        (rate <= 0)
 *   out_sin/cos  = sin, cos(rate dt pi/64)                    (NaN if the all-conjugate and generic variants differ)
 *   out_sh/ch    = (1 - rho)/2, (1 + rho)/2, rho = out_exp    (transition of a real root pair)
 *   out_rcp      = 1 / rate */
int carma_fastmath_dev(const double* rate, const double* dt, size_t n, double* out_exp, double* out_sin, double* out_cos,
                       double* out_sh, double* out_ch, double* out_rcp);

#ifdef __cplusplus
}
#endif
#endif /* CARMA_B200_H */
