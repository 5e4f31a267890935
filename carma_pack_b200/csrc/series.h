// series.h -- host-side objects behind the opaque handles of include/carma_b200.h
#pragma once
#include <cuda_runtime.h>

#include <string>
#include <mutex>
#include <vector>

#include "../../include/carma_b200.h"
#include "kalman_cplx.cuh"

namespace carma {

struct SeriesStats {
    double mean, var_sample, var_pop, median_dt, min_dt, tmin, tmax;
};

void set_error(const std::string& msg);
bool cuda_ok(cudaError_t e, const char* what);

// scratch device buffer that only grows
// cudaFuncSetAttribute waits for running instances of the function: set per launch, it made kernels launched from
// different host threads (concurrent model fits) run one after the other.  Attributes are per device and always get the
// same value here, so each launch site sets them once per device: `static OncePerDevice once;` inside the (templated)
// launch function, then once.run([] { return cudaFuncSetAttribute(...); }).
struct OncePerDevice {
    std::mutex mu;
    bool done[64] = {};
    cudaError_t err[64] = {};
    template <class F>
    cudaError_t run(F f) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return f();
        std::lock_guard<std::mutex> lk(mu);
        if (!done[dev]) { err[dev] = f(); done[dev] = true; }
        return err[dev];
    }
};

void* dev_alloc(size_t bytes, const char* what);   // stream-ordered pool allocation, ready on return (loglik.cu)
void dev_free(void* p);

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    bool reserve(size_t bytes);
    void release();
};

}  // namespace carma

struct carma_series {
    int device = 0;
    size_t ny = 0;
    int nyp = 0;
    double* d_pack = nullptr;  // [dt | y | e2n] (3 x nyp) followed by t (ny)
    double e2_0 = 0.0;
    double dt_max = 1.0;  // longest sampling gap
    std::vector<double> t, y, yerr;
    carma::SeriesStats st{};
    carma::DevBuf scratch_in, scratch_out, scratch_misc, scratch_state;
    // pipeline slots for the asynchronous host-buffer entry points (own stream + buffers each)
    carma::DevBuf slot_in[CARMA_N_SLOTS], slot_out[CARMA_N_SLOTS];
    cudaStream_t slot_stream[CARMA_N_SLOTS] = {};
    cudaStream_t blk_stream[4] = {};   // the blocking batch call splits large batches over these
    carma::SeriesView view() const {
        carma::SeriesView v;
        v.dt = d_pack;
        v.y = d_pack + nyp;
        v.e2n = d_pack + 2 * (size_t)nyp;
        v.t = d_pack + 3 * (size_t)nyp;
        v.e2_0 = e2_0;
        v.dt_max = dt_max;
        v.ny = (int)ny;
        v.nyp = nyp;
        return v;
    }
};

namespace carma {
// per-curve constants needed by the on-device samplers (prior + starting-value statistics)
struct CurveInfo {
    carma_prior_t prior;
    double y_mean, y_var_sample, y_var_pop, median_dt, tspan;
    double min_dt, dt_max;   // shortest and longest gap of the curve (the optimiser's box, its rate clamp)
};
}  // namespace carma

struct carma_multi_series {
    int device = 0;
    size_t ncurves = 0;
    size_t total = 0;
    // SoA device arrays of length total (+pad): dt (to next point of the same curve, 0 at the end),
    // y, e2 (yerr^2), and CSR offsets (ncurves+1)
    double* d_dt = nullptr;
    double* d_y = nullptr;
    double* d_e2 = nullptr;
    long long* d_off = nullptr;
    std::vector<long long> off;
    std::vector<carma_prior_t> priors_pop, priors_sample;
    std::vector<carma::CurveInfo> info;  // default (population-variance) priors + statistics
    std::vector<double> t0;  // first time of every curve: the device holds gaps only, each curve's axis starts at 0
    carma::DevBuf scratch_in, scratch_out, scratch_pr, scratch_misc;
    carma::DevBuf scratch_pts, scratch_q;  // per-point filter outputs and per-query records (survey.cu)
    int max_ny = 0;
    double dt_max = 1.0;  // longest sampling gap over all curves
};

namespace carma {
// Arrange p roots closed under conjugation into the slots of the real-half recursion (ExplicitModel).
// Returns false when the set is not conjugate-symmetric (then only the general complex kernels apply).
bool arrange_roots(const double* omega_reim, const double* ma, int p, double sigsqr, double scale, double mu, ExplicitModel* out);
// scan.cu: time-parallel Filter() of one explicit model with per-point outputs (device pointers, may be null)
int scan_explicit(carma_series* s, int p, const ExplicitModel& ex, double* d_mean, double* d_var, double* d_state,
                  double* d_loglik, cudaStream_t st, const double* d_y_override = nullptr);
SeriesStats compute_stats(const double* t, const double* y, size_t n);
void prior_from_stats(const SeriesStats& st, int population_var, carma_prior_t* out);
bool valid_model(int kind, int p, int q);   // (kind, p, q) names a model the library evaluates
}  // namespace carma
