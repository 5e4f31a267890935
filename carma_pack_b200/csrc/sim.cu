// sim.cu -- on-device synthetic light curves for the survey-scale configuration (BASELINE config 5: 10^6
// irregularly sampled CARMA light curves).  One thread = one curve.
//
// Same recipe as the reference's Python generator:
//   carma_process (src/carmcmc/carma_pack.py:1148-1259): run the rotated state-space filter WITHOUT
//   measurement noise and draw every value from its one-step predictive law (innovations form);
//   sampling times dt = dt_min + |Cauchy|, truncated (cpp_tests/generate_test_data.py:17);
//   y = mu + process + yerr * N(0,1).
// The filter recursion is the KalmanReal code of the log-likelihood kernels, so a curve simulated here at
// theta* is by construction a draw from the model whose likelihood K1/K4 evaluate.  Random numbers:
// Philox4x32-10 addressed by (seed, curve, point): curves do not depend on how they are sharded.
#include <algorithm>
#include <cmath>
#include <string>
#include <vector>

#include "kalman_real.cuh"
#include "series.h"

namespace carma {

enum { STREAM_SIMULATE = 4 };
constexpr int SIM_BLOCK = 64;

template <int P>
__global__ void __launch_bounds__(SIM_BLOCK)
simulate_kernel(size_t ncurves, int ny, int kind, int q, int d, const double* __restrict__ theta_true,
                carma_prior_t pr, double yerr, double dt_min, double dt_max, unsigned long long seed, unsigned curve_offset,
                double* __restrict__ dt_out, double* __restrict__ y_out, double* __restrict__ e2_out,
                CurveInfo* __restrict__ info, int* __restrict__ status) {
    MathTab tb;
    tb.load();
    const size_t c = (size_t)blockIdx.x * SIM_BLOCK + threadIdx.x;
    if (c >= ncurves) return;
    double th[MAX_D];
    for (int j = 0; j < MAX_D; j++) th[j] = (j < d) ? theta_true[j] : 0.0;
    RealParams<P> prm;
    if (transform_theta<P>(kind, q, CARMA_IGNORE_BOUNDS | CARMA_LOGLIK_ONLY, pr, th, dt_max, prm) != TT_OK) {
        atomicExch(status, 1);
        return;
    }
    prm.scale = 0.0;  // the process itself carries no measurement noise
    const double mu = prm.mu;
    KalmanReal<P> kf;
    kf.reset(prm, 0.0);
    const uint32_t chain = (uint32_t)(curve_offset + c);
    double* pdt = dt_out + c * (size_t)ny;
    double* py = y_out + c * (size_t)ny;
    double* pe = e2_out + c * (size_t)ny;
    const double e2 = yerr * yerr;
    double sum = 0.0, sumsq = 0.0, tspan = 0.0, dmin = 1e300, dmax = 0.0;
    for (int i = 0; i < ny; i++) {
        double u0, u1, u2, u3;
        uniforms2(seed, chain, STREAM_SIMULATE, (uint32_t)i, 0u, &u0, &u1);
        uniforms2(seed, chain, STREAM_SIMULATE, (uint32_t)i, 1u, &u2, &u3);
        const double rr = sqrt(-2.0 * log(u0));
        double sn, cs;
        sincos(6.283185307179586476925286766559 * u1, &sn, &cs);
        const double z_proc = rr * cs, z_noise = rr * sn;  // two independent normals from one Box-Muller pair
        const double innov = sqrt(fmax(kf.var, 0.0)) * z_proc;
        const double yi = mu + (kf.mean + innov) + yerr * z_noise;
        py[i] = yi;
        pe[i] = e2;
        sum += yi;
        sumsq += yi * yi;
        if (i + 1 < ny) {
            double dt = fmin(dt_min + fabs(tan(3.14159265358979323846 * (u2 - 0.5))), dt_max);
            pdt[i] = dt;
            tspan += dt;
            dmin = fmin(dmin, dt);
            dmax = fmax(dmax, dt);
            const double inv = kf.var > 0.0 ? 1.0 / kf.var : 0.0;
            kf.measurement_update(innov, inv);
            kf.template predict_observe<false>(prm, tb, dt, 0.0);
        } else {
            pdt[i] = 0.0;
        }
        (void)u3;
    }
    // exact median of the ny-1 gaps by bisection on the value (one-time cost, keeps everything on device).
    // Invariant: #(dt <= lo) < k+1 <= #(dt <= hi); afterwards the k-th order statistic is min{dt > lo}.
    const int n1 = ny - 1, k = (n1 - 1) / 2;
    double lo = 0.0, hi = dt_max;
    for (int it = 0; it < 64; it++) {
        const double mid = 0.5 * (lo + hi);
        int cnt = 0;
        for (int i = 0; i < n1; i++) cnt += (pdt[i] <= mid);
        if (cnt >= k + 1) hi = mid; else lo = mid;
    }
    double kth = 1e300;
    for (int i = 0; i < n1; i++) if (pdt[i] > lo) kth = fmin(kth, pdt[i]);
    double med_lo = kth;
    if ((n1 & 1) == 0) {  // even count: average the two central order statistics
        double nxt = 1e300;
        int cnt = 0;
        for (int i = 0; i < n1; i++) { cnt += (pdt[i] <= kth); if (pdt[i] > kth) nxt = fmin(nxt, pdt[i]); }
        med_lo = (cnt >= k + 2) ? kth : 0.5 * (kth + nxt);
    }
    CurveInfo ci;
    const double mean = sum / (double)ny;
    ci.y_mean = mean;
    ci.y_var_pop = sumsq / (double)ny - mean * mean;
    ci.y_var_sample = ny > 1 ? ci.y_var_pop * (double)ny / (double)(ny - 1) : 0.0;
    ci.median_dt = med_lo;
    ci.tspan = tspan;
    ci.min_dt = dmin;
    ci.dt_max = dmax;
    ci.prior.max_stdev = 10.0 * sqrt(fmax(ci.y_var_pop, 0.0));
    ci.prior.max_freq = 1.0 / dmin;
    ci.prior.min_freq = 1.0 / tspan;
    ci.prior.kappa_high = 1.0 / dmin;
    ci.prior.kappa_low = fmax(1.0 / tspan, 1.0 / (10.0 * med_lo));
    ci.prior.measerr_dof = 50.0;
    info[c] = ci;
}

}  // namespace carma

using namespace carma;

extern "C" int carma_multi_series_simulate(size_t ncurves, size_t ny, int kind, int p, int q, const double* theta_true,
                                           const carma_prior_t* prior, double yerr, double dt_min, double dt_max, uint64_t seed,
                                           uint32_t curve_offset, int device, carma_multi_series_t* out) {
    if (!theta_true || !out || ncurves == 0 || ny < 2 || !(dt_min > 0) || !(dt_max > dt_min) || !(yerr >= 0)) {
        set_error("carma_multi_series_simulate: bad argument");
        return CARMA_ERR_ARG;
    }
    if (kind < CARMA_KIND_CAR1 || kind > CARMA_KIND_ZCARMA || p < 1 || p > MAX_P || (kind == CARMA_KIND_CAR1 && p != 1) ||
        (kind == CARMA_KIND_CARMA && !(q >= 0 && q < p))) {
        set_error("carma_multi_series_simulate: invalid (kind,p,q)");
        return CARMA_ERR_ARG;
    }
    if (!cuda_ok(cudaSetDevice(device), "cudaSetDevice")) return CARMA_ERR_CUDA;
    carma_multi_series* m = new (std::nothrow) carma_multi_series();
    if (!m) return CARMA_ERR_ALLOC;
    m->device = device;
    m->ncurves = ncurves;
    m->total = ncurves * ny;
    m->max_ny = (int)ny;
    m->off.resize(ncurves + 1);
    for (size_t c = 0; c <= ncurves; c++) m->off[c] = (long long)(c * ny);
    m->t0.assign(ncurves, 0.0);
    const int d = model_dim(kind, p, q);
    carma_prior_t pr;
    if (prior) {
        pr = *prior;
    } else {  // wide-open bounds (only CAR1 and the kappa of ZCARMA look at them under IGNORE_BOUNDS)
        pr.max_stdev = 1e300; pr.max_freq = 1e300; pr.min_freq = 0.0;
        pr.kappa_low = 0.0; pr.kappa_high = 1.0 / dt_min; pr.measerr_dof = 50.0;
    }
    double* d_theta = nullptr;
    CurveInfo* d_info = nullptr;
    int* d_status = nullptr;
    bool ok = cuda_ok(cudaMalloc((void**)&m->d_dt, (m->total + 1) * sizeof(double)), "cudaMalloc(sim dt)") &&
              cuda_ok(cudaMalloc((void**)&m->d_y, (m->total + 1) * sizeof(double)), "cudaMalloc(sim y)") &&
              cuda_ok(cudaMalloc((void**)&m->d_e2, (m->total + 1) * sizeof(double)), "cudaMalloc(sim e2)") &&
              cuda_ok(cudaMalloc((void**)&m->d_off, (ncurves + 1) * sizeof(long long)), "cudaMalloc(sim off)") &&
              cuda_ok(cudaMalloc((void**)&d_theta, d * sizeof(double)), "cudaMalloc(sim theta)") &&
              cuda_ok(cudaMalloc((void**)&d_info, ncurves * sizeof(CurveInfo)), "cudaMalloc(sim info)") &&
              cuda_ok(cudaMalloc((void**)&d_status, sizeof(int)), "cudaMalloc(sim status)") &&
              cuda_ok(cudaMemset(d_status, 0, sizeof(int)), "memset") &&
              cuda_ok(cudaMemset(m->d_e2 + m->total, 0, sizeof(double)), "memset") &&
              cuda_ok(cudaMemcpy(m->d_off, m->off.data(), (ncurves + 1) * sizeof(long long), cudaMemcpyHostToDevice), "H2D off") &&
              cuda_ok(cudaMemcpy(d_theta, theta_true, d * sizeof(double), cudaMemcpyHostToDevice), "H2D theta");
    if (ok) {
        unsigned grid = (unsigned)((ncurves + SIM_BLOCK - 1) / SIM_BLOCK);
#define LAUNCH_SIM(PP)                                                                                             \
    simulate_kernel<PP><<<grid, SIM_BLOCK>>>(ncurves, (int)ny, kind, q, d, d_theta, pr, yerr, dt_min, dt_max, seed,     \
                                             curve_offset, m->d_dt, m->d_y, m->d_e2, d_info, d_status)
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
        ok = cuda_ok(cudaGetLastError(), "simulate_kernel launch") && cuda_ok(cudaDeviceSynchronize(), "simulate_kernel");
    }
    int status = 0;
    if (ok) ok = cuda_ok(cudaMemcpy(&status, d_status, sizeof(int), cudaMemcpyDeviceToHost), "D2H status");
    if (ok && status) { set_error("carma_multi_series_simulate: theta_true is not a valid model (singular roots)"); ok = false; }
    if (ok) {
        m->info.resize(ncurves);
        ok = cuda_ok(cudaMemcpy(m->info.data(), d_info, ncurves * sizeof(CurveInfo), cudaMemcpyDeviceToHost), "D2H info");
    }
    if (d_theta) cudaFree(d_theta);
    if (d_info) cudaFree(d_info);
    if (d_status) cudaFree(d_status);
    if (!ok) {
        carma_multi_series_destroy(m);
        return status ? CARMA_ERR_ARG : CARMA_ERR_CUDA;
    }
    m->dt_max = dt_max;  // every gap is truncated at dt_max
    m->priors_pop.resize(ncurves);
    m->priors_sample.resize(ncurves);
    for (size_t c = 0; c < ncurves; c++) {
        m->priors_pop[c] = m->info[c].prior;
        m->priors_sample[c] = m->info[c].prior;
        m->priors_sample[c].max_stdev = 10.0 * std::sqrt(std::max(m->info[c].y_var_sample, 0.0));
    }
    *out = m;
    return CARMA_OK;
}

// copy one curve of a (simulated or uploaded) batch back to the host: time (from t0 = 0), y, yerr
extern "C" int carma_multi_series_get_curve(carma_multi_series_t m, size_t curve, double* time, double* y, double* yerr,
                                            size_t capacity, size_t* ny_out) {
    if (!m || curve >= m->ncurves || !time || !y || !yerr) { set_error("carma_multi_series_get_curve: bad argument"); return CARMA_ERR_ARG; }
    const size_t o0 = (size_t)m->off[curve], n = (size_t)(m->off[curve + 1] - m->off[curve]);
    if (ny_out) *ny_out = n;
    if (capacity < n) { set_error("carma_multi_series_get_curve: capacity too small"); return CARMA_ERR_ARG; }
    if (!cuda_ok(cudaSetDevice(m->device), "cudaSetDevice")) return CARMA_ERR_CUDA;
    std::vector<double> dt(n), e2(n);
    bool ok = cuda_ok(cudaMemcpy(dt.data(), m->d_dt + o0, n * sizeof(double), cudaMemcpyDeviceToHost), "D2H dt") &&
              cuda_ok(cudaMemcpy(y, m->d_y + o0, n * sizeof(double), cudaMemcpyDeviceToHost), "D2H y") &&
              cuda_ok(cudaMemcpy(e2.data(), m->d_e2 + o0, n * sizeof(double), cudaMemcpyDeviceToHost), "D2H e2");
    if (!ok) return CARMA_ERR_CUDA;
    double t = 0.0;
    for (size_t i = 0; i < n; i++) {
        time[i] = t;
        t += dt[i];
        yerr[i] = std::sqrt(e2[i]);
    }
    return CARMA_OK;
}
