// loglik.cu -- batched CARMA log-density kernels (K1/K2/K4) and the explicit-parameter
// filter / predict kernels, plus their C-ABI entry points.
//
// K1  loglik_batch_kernel<P>:  one thread = one theta = one complete LogDensity
//     (carpack.hpp:131-176 -> kfilter.cpp:138-215).  The light curve (dt, y, yerr^2) is staged once
//     per block in shared memory by the TMA engine (cp.async.bulk + mbarrier, double buffered for
//     long series) and read by every thread with broadcast LDS; the filter state lives in registers.
// K4  multi_loglik_kernel<P>:  one thread = one light curve with its own theta.
#include <cmath>
#include <cstdio>
#include <cstring>
#include <algorithm>
#include <cstdlib>
#include <limits>
#include <type_traits>
#include <utility>
#include <vector>

#include "kalman_real.cuh"
#include "series.h"

namespace carma {

// ---------------------------------------------------------------------------------------------
// K1
// ---------------------------------------------------------------------------------------------
constexpr int K1_BLOCK = 64;
constexpr int K1_CHUNK = 512;  // points per staged chunk: compile-time strides, so the loop's three LDS share one address register

// resident blocks per SM wanted for each P (bounds the register allocation so that the
// BASELINE batch of 65,536 thetas fits in one wave of 148 SMs: 7 x 64 x 148 = 66,304 at P = 5)
__host__ __device__ constexpr int k1_min_blocks(int P) { return P <= 4 ? 8 : (P == 5 ? 7 : (P == 6 ? 5 : 4)); }

template <int P>
__global__ void __launch_bounds__(K1_BLOCK, k1_min_blocks(P))
loglik_batch_kernel(SeriesView sv, int kind, int q, int d, unsigned flags, carma_prior_t prior,
                    const double* __restrict__ theta, double* __restrict__ out, size_t n) {
    // series chunk buffers, aliased with the LU scratch of the prologue (the math tables are static shared arrays)
    extern __shared__ __align__(16) double smem[];
    __shared__ __align__(8) uint64_t bars[2];

    const int tid = threadIdx.x;
    const size_t row = (size_t)blockIdx.x * K1_BLOCK + tid;
    const int ny = sv.ny;
    const int nchunks = (ny + K1_CHUNK - 1) / K1_CHUNK;
    double* work = smem;

    if (tid == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        fence_mbar_init();
    }
    MathTab tb;
    tb.load();  // ends with __syncthreads()

    auto issue = [&](int k) {
        // chunk k -> buffer k&1 : three bulk copies (dt, y, e2n), byte counts multiples of 16
        const int start = k * K1_CHUNK;
        const int len = min(K1_CHUNK, sv.nyp - start);
        const uint32_t bytes = (uint32_t)len * 8u;
        double* dst = work + (size_t)(k & 1) * 3 * K1_CHUNK;
        mbar_expect_tx(&bars[k & 1], 3u * bytes);
        bulk_g2s(dst, sv.dt + start, bytes, &bars[k & 1]);
        bulk_g2s(dst + K1_CHUNK, sv.y + start, bytes, &bars[k & 1]);
        bulk_g2s(dst + 2 * K1_CHUNK, sv.e2n + start, bytes, &bars[k & 1]);
    };

    // ---- per-theta prologue.  The P x P complex LU of the Vandermonde solve works in shared memory
    // ([element][thread], conflict-free), in the space the series buffers take over afterwards.
    RealParams<P> prm;
    KalmanReal<P> kf;
    LogLikAcc acc;
    bool active = row < n;
    int status = TT_OK;
    if (active) {
        // theta is read straight from global memory (the transform touches only its first d entries)
        status = transform_theta<P, false, true>(kind, q, flags, prior, theta + row * (size_t)d, sv.dt_max, prm, nullptr,
                                                 work + tid, K1_BLOCK);
        if (status != TT_OK) active = false;
    }
    if (active) kf.reset(prm, sv.e2_0);
    acc.init();
    // the generic-proxy accesses above must be ordered before the bulk (async-proxy) writes into the same bytes
    fence_proxy_async();
    __syncthreads();
    if (tid == 0) {
        issue(0);
        if (nchunks > 1) issue(1);
    }

    // ---- time loop
    const uint32_t work_addr = smem_u32(work);
    for (int k = 0; k < nchunks; k++) {
        const int buf = k & 1;
        mbar_wait(&bars[buf], (uint32_t)((k >> 1) & 1));
        if (active) {
            const SeriesSmem src{work_addr + (uint32_t)buf * 3u * K1_CHUNK * 8u, K1_CHUNK * 8u, 2u * K1_CHUNK * 8u};
            const int start = k * K1_CHUNK;
            const int len = min(K1_CHUNK, ny - start);
            const int nadv = (start + len == ny) ? len - 1 : len;  // no advance after the last point
            filter_span_any<P, false>(kf, acc, prm, tb, src, len, nadv);
        }
        if (k + 2 < nchunks) {
            __syncthreads();  // every thread is done with this buffer
            if (tid == 0) issue(k + 2);
        }
    }

    if (row < n) {
        double r;
        if (status != TT_OK) r = -INFINITY;
        else if (acc.bad()) r = loglik_exact_slow<P>(prm, tb, SeriesPtr{sv.dt, sv.y, sv.e2n}, ny, sv.e2_0) + prm.logprior;
        else r = acc.value() + prm.logprior;
        out[row] = r;
    }
}

static size_t k1_smem_bytes(int P, int ny) {
    const int nchunks = (ny + K1_CHUNK - 1) / K1_CHUNK;
    size_t series = (size_t)(nchunks > 1 ? 2 : 1) * 3 * K1_CHUNK * sizeof(double);
    size_t lu = (size_t)2 * P * P * K1_BLOCK * sizeof(double);  // LU scratch of the prologue (aliased)
    return std::max(series, lu);
}

// the > 48 KiB opt-in for every order at once, once per device (cudaFuncSetAttribute waits for running kernels: see
// OncePerDevice in series.h)
template <int P>
static cudaError_t k1_attr_from() {
    cudaError_t e = cudaFuncSetAttribute(loglik_batch_kernel<P>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
    if (e != cudaSuccess) return e;
    if constexpr (P < MAX_P) return k1_attr_from<P + 1>();
    else return cudaSuccess;
}
static cudaError_t k1_attrs() {
    static OncePerDevice once;
    return once.run([] { return k1_attr_from<1>(); });
}

template <int P>
static cudaError_t launch_k1(const SeriesView& sv, int kind, int q, int d, unsigned flags, const carma_prior_t& prior,
                             const double* d_theta, double* d_out, size_t n, cudaStream_t stream) {
    const size_t smem = k1_smem_bytes(P, sv.ny);
    unsigned grid = (unsigned)((n + K1_BLOCK - 1) / K1_BLOCK);
    if (smem > 48 * 1024) {
        // > 48 KiB of dynamic shared memory needs the opt-in (P = 7: 54,528 B).  Per device and always the same
        // value, so concurrent callers cannot disagree.
        cudaError_t e = k1_attrs();
        if (e != cudaSuccess) return e;
    }
    loglik_batch_kernel<P><<<grid, K1_BLOCK, smem, stream>>>(sv, kind, q, d, flags, prior, d_theta, d_out, n);
    return cudaGetLastError();
}

cudaError_t launch_loglik_batch(const SeriesView& sv, int kind, int p, int q, unsigned flags,
                                const carma_prior_t& prior, const double* d_theta, double* d_out, size_t n,
                                cudaStream_t stream) {
    int d = model_dim(kind, p, q);
    switch (p) {
        case 1: return launch_k1<1>(sv, kind, q, d, flags, prior, d_theta, d_out, n, stream);
        case 2: return launch_k1<2>(sv, kind, q, d, flags, prior, d_theta, d_out, n, stream);
        case 3: return launch_k1<3>(sv, kind, q, d, flags, prior, d_theta, d_out, n, stream);
        case 4: return launch_k1<4>(sv, kind, q, d, flags, prior, d_theta, d_out, n, stream);
        case 5: return launch_k1<5>(sv, kind, q, d, flags, prior, d_theta, d_out, n, stream);
        case 6: return launch_k1<6>(sv, kind, q, d, flags, prior, d_theta, d_out, n, stream);
        case 7: return launch_k1<7>(sv, kind, q, d, flags, prior, d_theta, d_out, n, stream);
        default: return cudaErrorInvalidValue;
    }
}

// ---------------------------------------------------------------------------------------------
// K4: one light curve per thread (ragged, CSR offsets); per-curve theta and prior
// ---------------------------------------------------------------------------------------------
constexpr int K4_BLOCK = 64;

// GTAB: math tables read from global memory (default, see MathTabGlobal) instead of static shared memory
// BLK4: the curve is fetched four steps per access with the next block in flight (filter_span_blocks); false: one
// step per access, one step ahead (CARMA_K4_LOADS=scalar, kept for comparison)
template <int P, bool GTAB, bool BLK4>
__global__ void __launch_bounds__(K4_BLOCK, P <= 3 ? 8 : 1)   // P <= 3: 128 registers, 8 blocks (4 warps per scheduler); measured at P = 3
multi_loglik_kernel(const double* __restrict__ dt, const double* __restrict__ y, const double* __restrict__ e2,
                    const long long* __restrict__ off, size_t ncurves, double dt_max, int kind, int q, int d, unsigned flags,
                    const carma_prior_t* __restrict__ priors, const double* __restrict__ theta,
                    double* __restrict__ out) {
    typename std::conditional<GTAB, MathTabGlobal, MathTab>::type tb;
    tb.load();
    const size_t c = (size_t)blockIdx.x * K4_BLOCK + threadIdx.x;
    if (c >= ncurves) return;
    const long long o0 = off[c], o1 = off[c + 1];
    const int ny = (int)(o1 - o0);
    double th[MAX_D];
#pragma unroll
    for (int j = 0; j < MAX_D; j++) th[j] = (j < d) ? theta[c * (size_t)d + j] : 0.0;
    RealParams<P> prm;
    carma_prior_t pr = priors[c];
    int status = transform_theta<P>(kind, q, flags, pr, th, dt_max, prm);
    if (status != TT_OK || ny <= 0) {
        out[c] = (ny <= 0) ? 0.0 : -INFINITY;
        return;
    }
    KalmanReal<P> kf;
    LogLikAcc acc;
    kf.reset(prm, e2[o0]);
    acc.init();
    // e2 of the NEXT point is needed at step i: pass the array shifted by one
    const SeriesPtr src{dt + o0, y + o0, e2 + o0 + 1};
    if (BLK4) filter_span_blocks_any<P>(kf, acc, prm, tb, dt + o0, y + o0, e2 + o0, ny);
    else filter_span_any<P, true>(kf, acc, prm, tb, src, ny, ny - 1);
    out[c] = (acc.bad() ? loglik_exact_slow<P>(prm, tb, src, ny, e2[o0]) : acc.value()) + prm.logprior;
}

cudaError_t launch_multi_loglik(const carma_multi_series* m, int kind, int p, int q, unsigned flags,
                                const carma_prior_t* d_priors, const double* d_theta, double* d_out,
                                cudaStream_t stream) {
    int d = model_dim(kind, p, q);
    unsigned grid = (unsigned)((m->ncurves + K4_BLOCK - 1) / K4_BLOCK);
    static const bool scalar_loads = [] { const char* e = getenv("CARMA_K4_LOADS"); return e && !strcmp(e, "scalar"); }();
    // math tables: static shared arrays with the block loads (the curve no longer lives in L1 between steps, so the
    // 4.6 kB per block are free: survey 1.27 -> 1.41e8 curves/s); global memory with the scalar loads, where shared
    // tables cost the survey 10 % of L1 hits.  CARMA_K4_TABLES=smem|global overrides.
    static const bool smem_tab = [] {
        const char* e = getenv("CARMA_K4_TABLES");
        if (e && !strcmp(e, "smem")) return true;
        if (e && !strcmp(e, "global")) return false;
        return !scalar_loads;
    }();
#define LAUNCH_K4_AS(PP, GT, B4)                                                                                      \
    multi_loglik_kernel<PP, GT, B4><<<grid, K4_BLOCK, 0, stream>>>(m->d_dt, m->d_y, m->d_e2, m->d_off, m->ncurves,    \
                                                                   m->dt_max, kind, q, d, flags, d_priors, d_theta, d_out)
    // the block loads need the three arrays to sit alike within a 32-byte sector (separate allocations: they do)
    const bool alike = ((((size_t)m->d_dt ^ (size_t)m->d_y) | ((size_t)m->d_dt ^ (size_t)m->d_e2)) & 31u) == 0;
    const bool scalar_now = scalar_loads || !alike;
#define LAUNCH_K4(PP)                                                                                                 \
    if (smem_tab) { if (scalar_now) LAUNCH_K4_AS(PP, false, false); else LAUNCH_K4_AS(PP, false, true); }             \
    else { if (scalar_now) LAUNCH_K4_AS(PP, true, false); else LAUNCH_K4_AS(PP, true, true); }
    switch (p) {
        case 1: LAUNCH_K4(1); break;
        case 2: LAUNCH_K4(2); break;
        case 3: LAUNCH_K4(3); break;
        case 4: LAUNCH_K4(4); break;
        case 5: LAUNCH_K4(5); break;
        case 6: LAUNCH_K4(6); break;
        case 7: LAUNCH_K4(7); break;
        default: return cudaErrorInvalidValue;
    }
#undef LAUNCH_K4
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// explicit-parameter filter / predict (KalmanFilterp class API)
// ---------------------------------------------------------------------------------------------
struct FilterArgs {
    double sigsqr, scale, mu;
    double omega[2 * MAX_P];
    double ma[MAX_P];
    int p;
};

__global__ void filter_kernel(SeriesView sv, FilterArgs a, double* __restrict__ mean, double* __restrict__ var,
                              int* __restrict__ status) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    KalmanCplx kf;
    kf.scale = a.scale;
    kf.mu = a.mu;
    if (!kf.reset(a.sigsqr, a.omega, a.ma, a.p, sv.e2_0, sv.y[0])) {
        *status = 1;
        return;
    }
    *status = 0;
    mean[0] = kf.mean;
    var[0] = kf.var;
    for (int i = 1; i < sv.ny; i++) {
        kf.update(sv.dt[i - 1], sv.y[i], sv.e2n[i - 1]);
        mean[i] = kf.mean;
        var[i] = kf.var;
    }
}

// one thread per query time (kfilter.cpp:218-286)
__global__ void predict_kernel(SeriesView sv, FilterArgs a, const double* __restrict__ tq, size_t nq,
                               double* __restrict__ qmean, double* __restrict__ qvar, int* __restrict__ status) {
    size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= nq) return;
    const double time = tq[k];
    const int ny = sv.ny;
    int ipredict = 0;
    while (time > sv.t[ipredict]) {
        ipredict++;
        if (ipredict == ny) break;
    }
    KalmanCplx kf;
    kf.scale = a.scale;
    kf.mu = a.mu;
    if (!kf.reset(a.sigsqr, a.omega, a.ma, a.p, sv.e2_0, sv.y[0])) {
        *status = 1;
        qmean[k] = NAN;
        qvar[k] = NAN;
        return;
    }
    for (int i = 1; i < ipredict; i++) kf.update(sv.dt[i - 1], sv.y[i], sv.e2n[i - 1]);
    double pmean, pvar;
    if (ipredict == 0) {
        pmean = 0.0;
        pvar = kf.var - a.scale * sv.e2_0;  // Re(b V b^H): kf.g still holds V b^H
    } else {
        kf.gain_and_advance(kf.var, fabs(time - sv.t[ipredict - 1]));
        double m = 0.0;
        for (int i = 0; i < kf.p; i++) m += kf.b[i].re * kf.x[i].re - kf.b[i].im * kf.x[i].im;
        pmean = m;
        pvar = kf.quad_form();
    }
    if (ipredict == ny) {
        qmean[k] = pmean;
        qvar[k] = pvar;
        return;
    }
    double prec = 1.0 / pvar;
    pmean *= prec;
    auto e2_at = [&](int i) { return i == 0 ? sv.e2_0 : sv.e2n[i - 1]; };
    kf.initialize_coefs(fabs(sv.t[ipredict] - time), pmean / prec, pvar, e2_at(ipredict));
    prec += kf.yslope * kf.yslope / kf.var;
    pmean += kf.yslope * ((sv.y[ipredict] - a.mu) - kf.yconst) / kf.var;
    for (int i = ipredict + 1; i < ny; i++) {
        kf.update_coefs(sv.dt[i - 1], sv.y[i - 1], e2_at(i));
        prec += kf.yslope * kf.yslope / kf.var;
        pmean += kf.yslope * ((sv.y[i] - a.mu) - kf.yconst) / kf.var;
    }
    pvar = 1.0 / prec;
    pmean *= pvar;
    qmean[k] = pmean;
    qvar[k] = pvar;
}

// ---------------------------------------------------------------------------------------------
// Predict in the real-half recursion, resuming from stored forward states (explicit models whose roots are closed
// under conjugation -- every model the theta parameterisation can produce).  The forward filter runs ONCE (time-parallel,
// scan.cu) and leaves the state predicted at every data point; a query thread loads the state in front of its
// insertion point and runs only the linear-coefficient pass over the points behind it (kfilter.cpp:252-281).
// ---------------------------------------------------------------------------------------------
template <int P>
__global__ void __launch_bounds__(64)
predict_real_kernel(SeriesView sv, ExplicitModel ex, const double* __restrict__ state, const double* __restrict__ tq, size_t nq,
                    double* __restrict__ qmean, double* __restrict__ qvar /* may be null */) {
    constexpr int SD = P + P * (P + 1) / 2;
    MathTab tb;
    tb.load();
    const size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= nq) return;
    RealParams<P> prm;
    if (explicit_constants<P>(ex, sv.dt_max, prm) != TT_OK) { qmean[k] = NAN; if (qvar) qvar[k] = NAN; return; }
    const double time = tq[k];
    const int ny = sv.ny;
    int lo = 0, hi = ny;  // ip = number of data times strictly before `time` (kfilter.cpp:223-229)
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (sv.t[mid] < time) lo = mid + 1; else hi = mid;
    }
    const int ip = lo;
    const double* st = state + (size_t)(ip > 0 ? ip - 1 : 0) * SD;
    const double gap_before = ip > 0 ? fabs(time - sv.t[ip - 1]) : 0.0;
    const double gap_after = ip < ny ? fabs(sv.t[ip] - time) : 0.0;
    double pmean, pvar;
    predict_resume<P>(prm, tb, st, st + P, ip, ny, gap_before, gap_after, [&](int i) { return sv.y[i]; },
                      [&](int i) { return sv.dt[i]; }, [&](int i) { return i == 0 ? sv.e2_0 : sv.e2n[i - 1]; },
                      &pmean, &pvar);
    qmean[k] = pmean;
    if (qvar) qvar[k] = pvar;
}

// ---------------------------------------------------------------------------------------------
// Conditional simulation (KalmanFilter<>::Simulate, kfilter.hpp:135-184) by Matheron's rule: a draw of the process at
// the requested times GIVEN the data is   f_prior(t*) + E[f(t*) | data'],   data' = (y - mu) - f_prior(T) - eps,
// with f_prior an unconditional draw of the process on the merged grid (data times T and requested times t*) and eps
// fresh measurement noise.  O(ny + nsim) work per path instead of the reference's insert-and-re-predict loop
// (O(nsim (ny + nsim))), and every path of a call is independent: one thread draws one prior path (innovations form
// of the noise-free filter, as simulate_kernel), the conditional mean comes from the fast Predict above.
// ---------------------------------------------------------------------------------------------
template <int P>
__global__ void __launch_bounds__(64)
sim_prior_kernel(ExplicitModel ex, double dt_max, int nm, const double* __restrict__ dtm /* nm: gap to next merged point */,
                 const int* __restrict__ idx /* nm: >= 0 data index, < 0: -(sim index) - 1 */, const double* __restrict__ y,
                 const double* __restrict__ yerr, int ny, int nsim, unsigned long long seed, int npaths,
                 double* __restrict__ yres /* [npaths][nyp] residual data */, int nyp, double* __restrict__ fsim /* [npaths][nsim] */) {
    MathTab tb;
    tb.load();
    const int path = blockIdx.x * blockDim.x + threadIdx.x;
    if (path >= npaths) return;
    RealParams<P> prm;
    if (explicit_constants<P>(ex, dt_max, prm) != TT_OK) {
        for (int i = 0; i < nsim; i++) fsim[(size_t)path * nsim + i] = NAN;
        return;
    }
    const double mu = prm.mu, sscale = sqrt(prm.scale);
    prm.scale = 0.0;   // the process itself carries no measurement noise
    KalmanReal<P> kf;
    kf.reset(prm, 0.0);
    for (int k = 0; k < nm; k++) {
        double innov, rr, sn;
        const double f = condsim_draw(kf, seed, (uint32_t)path, (uint32_t)k, 0u, &innov, &rr, &sn);
        const int id = idx[k];
        if (id >= 0) yres[(size_t)path * nyp + id] = (y[id] - mu) - f - sscale * yerr[id] * rr * sn;   // second normal: eps
        else fsim[(size_t)path * nsim + (-id - 1)] = f;
        if (k + 1 < nm) condsim_next(kf, prm, tb, innov, dtm[k]);
    }
}

__global__ void add_prior_kernel(const double* __restrict__ fsim, double mu, size_t n, double* __restrict__ out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = out[i] + fsim[i] + mu;
}

bool arrange_roots(const double* om, const double* ma, int p, double sigsqr, double scale, double mu, ExplicitModel* out) {
    if (p < 1 || p > MAX_P) return false;
    std::vector<int> reals, used(p, 0);
    std::vector<std::pair<int, int> > pairs;
    for (int i = 0; i < p; i++) {
        if (used[i]) continue;
        const double re = om[2 * i], im = om[2 * i + 1];
        if (!std::isfinite(re) || !std::isfinite(im)) return false;
        if (im == 0.0) { reals.push_back(i); used[i] = 1; continue; }
        int partner = -1;
        const double mag = std::hypot(re, im);
        for (int j = i + 1; j < p; j++) {
            if (used[j]) continue;
            if (std::fabs(om[2 * j] - re) <= 1e-13 * mag && std::fabs(om[2 * j + 1] + im) <= 1e-13 * mag) { partner = j; break; }
        }
        if (partner < 0) return false;
        used[i] = used[partner] = 1;
        pairs.push_back(im < 0 ? std::make_pair(i, partner) : std::make_pair(partner, i));  // first root: Im <= 0
    }
    if ((reals.size() & 1u) != (size_t)(p & 1)) return false;
    std::sort(reals.begin(), reals.end(), [&](int a, int b) { return om[2 * a] < om[2 * b]; });
    ExplicitModel ex{};
    ex.sigsqr = sigsqr; ex.scale = scale; ex.mu = mu; ex.cmask = 0;
    int slot = 0;
    for (auto& pr : pairs) {
        ex.w_re[2 * slot] = om[2 * pr.first]; ex.w_im[2 * slot] = om[2 * pr.first + 1];
        ex.w_re[2 * slot + 1] = om[2 * pr.first]; ex.w_im[2 * slot + 1] = -om[2 * pr.first + 1];   // the exact conjugate
        ex.cmask |= 1u << slot;
        slot++;
    }
    size_t r = 0;
    for (; r + 1 < reals.size(); r += 2, slot++) {   // two real roots per slot, the more negative one first
        ex.w_re[2 * slot] = om[2 * reals[r]]; ex.w_im[2 * slot] = 0.0;
        ex.w_re[2 * slot + 1] = om[2 * reals[r + 1]]; ex.w_im[2 * slot + 1] = 0.0;
        if (ex.w_re[2 * slot] == ex.w_re[2 * slot + 1]) return false;  // repeated root: singular Vandermonde
    }
    if (p & 1) { ex.w_re[p - 1] = om[2 * reals[r]]; ex.w_im[p - 1] = 0.0; }
    for (int i = 0; i < MAX_P; i++) ex.ma[i] = i < p ? ma[i] : 0.0;
    *out = ex;
    return true;
}

// ---------------------------------------------------------------------------------------------
// Posterior post-processing (SURVEY 8f-2; src/carmcmc/carma_pack.py:439-546): one thread per stored sample turns the
// theta row into the derived quantities CarmaSample exposes -- AR roots, AR polynomial, normalised MA coefficients,
// sigma of the driving noise, PSD widths and centroids -- with the formulas of CarmaSample._ar_roots / _ar_coefs /
// _ma_coefs / _sigma_noise (IEEE division throughout; the same root, MA and variance code paths as transform_theta).
// Row layout of `out` (width 6P + 2): [ roots (re, im) x P | ar_coefs P+1 (highest power first) | ma_coefs P (beta_0 = 1,
// zero beyond q) | sigma | psd_width P | psd_centroid P ].
// ---------------------------------------------------------------------------------------------
template <int P>
__global__ void __launch_bounds__(128) derived_params_kernel(int kind, int q, carma_prior_t pr, const double* __restrict__ theta,
                                                             size_t n, double* __restrict__ out) {
    constexpr double PI = 3.14159265358979323846;
    const size_t r = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    const int d = model_dim(kind, P, q);
    const double* th = theta + r * (size_t)d;
    double* o = out + r * (size_t)(6 * P + 2);
    cxd w[P], ac[P + 1];
    double ma[P];
    const double sigsqr = derive_row<P, true>(kind, q, pr, th, w, ma, ac);
#pragma unroll
    for (int k = 0; k < P; k++) {
        o[2 * k] = w[k].re;
        o[2 * k + 1] = w[k].im;
        o[2 * P + (P + 1) + k] = ma[k];
        o[4 * P + 2 + k] = -w[k].re / (2.0 * PI);
        o[5 * P + 2 + k] = fabs(w[k].im) / (2.0 * PI);
    }
#pragma unroll
    for (int k = 0; k <= P; k++) o[2 * P + k] = ac[k].re;
    o[4 * P + 1] = sqrt(sigsqr);
}

template <int P>
static cudaError_t launch_derived(int kind, int q, const carma_prior_t& pr, const double* d_theta, size_t n, double* d_out,
                                  cudaStream_t st) {
    derived_params_kernel<P><<<(unsigned)((n + 127) / 128), 128, 0, st>>>(kind, q, pr, d_theta, n, d_out);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// FP64 FMA saturation micro-benchmark (roofline denominator measured on the same GPU)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) dfma_peak_kernel(double* out, int iters, double a, double b) {
    double x0 = threadIdx.x * 1e-3, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6,
           x7 = x0 + 7;
    for (int i = 0; i < iters; i++) {
        x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
        x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
    }
    double s = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
    if (s == 12345.678) out[0] = s;
}

__global__ void fastmath_kernel(const double* __restrict__ l, const double* __restrict__ dt, size_t n, double* __restrict__ e,
                                double* __restrict__ sn, double* __restrict__ cs, double* __restrict__ sr, double* __restrict__ cr,
                                double* __restrict__ rc) {
    MathTab tb;
    tb.load();
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    e[i] = exp_scaled(l[i], dt[i], tb);
    double s, c, s1, c1;
    rot_scaled<true>(l[i], dt[i], true, tb, &s, &c);
    rot_scaled<false>(l[i], dt[i], true, tb, &s1, &c1);
    if (s1 != s || c1 != c) s = NAN;  // the all-conjugate and the generic variant must agree bit for bit
    sn[i] = s;
    cs[i] = c;
    rot_scaled<false>(l[i], dt[i], false, tb, &s, &c);
    sr[i] = s;
    cr[i] = c;
    rc[i] = rcp_fast(l[i]);
}

__global__ void philox_kernel(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint64_t seed, uint32_t* out) {
    philox4x32_10(c0, c1, c2, c3, seed, out);
}
__global__ void tdist_kernel(uint64_t seed, uint32_t chain, uint32_t iter, uint32_t j, int dof, double* out) {
    *out = tdist_draw(seed, chain, STREAM_PROPOSAL, iter, j, dof);
}

// ---------------------------------------------------------------------------------------------
// host helpers
// ---------------------------------------------------------------------------------------------
static thread_local std::string g_last_error;
void set_error(const std::string& msg) { g_last_error = msg; }
bool cuda_ok(cudaError_t e, const char* what) {
    if (e == cudaSuccess) return true;
    set_error(std::string(what) + ": " + cudaGetErrorString(e));
    (void)cudaGetLastError();  // a reported (non-sticky) error must not resurface in a later, unrelated launch check
    return false;
}
// Device memory comes from the device's stream-ordered pool.  cudaMalloc / cudaFree synchronise with the work in flight
// on the device: a series handle that allocated its scratch buffers for the first time while OTHER host threads had long
// kernels running (concurrent model fits of choose_order) stalled behind them, and the fits ended up one after the
// other (measured: 4.2 s cold against 1.2 s with pre-allocated buffers).  A first allocation now waits for nothing; a
// buffer that has to GROW still waits for the device before the old block goes back to the pool, because asynchronous
// entry points (carma_*_dev) may have work queued on it in streams this library does not own.
static cudaStream_t alloc_stream() {
    static std::mutex mu;
    static cudaStream_t st[64] = {};
    static bool pool_set[64] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    std::lock_guard<std::mutex> lk(mu);
    if (!st[dev] && cudaStreamCreateWithFlags(&st[dev], cudaStreamNonBlocking) != cudaSuccess) st[dev] = nullptr;
    if (!pool_set[dev]) {
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
            unsigned long long keep = ~0ull;   // freed blocks stay in the pool: no trip to the OS, no implicit synchronisation
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
        pool_set[dev] = true;
    }
    return st[dev];
}
void* dev_alloc(size_t bytes, const char* what) {
    void* q = nullptr;
    cudaStream_t as = alloc_stream();
    if (!as) return cuda_ok(cudaMalloc(&q, bytes), what) ? q : nullptr;
    if (!cuda_ok(cudaMallocAsync(&q, bytes, as), what) || !cuda_ok(cudaStreamSynchronize(as), what)) return nullptr;
    return q;
}
void dev_free(void* q) {
    if (!q) return;
    cudaStream_t as = alloc_stream();
    cudaDeviceSynchronize();   // see above: what cudaFree did implicitly
    if (!as || cudaFreeAsync(q, as) != cudaSuccess) cudaFree(q);
}
bool DevBuf::reserve(size_t bytes) {
    if (bytes <= cap) return true;
    if (p) dev_free(p);
    cap = 0;
    p = dev_alloc(bytes, "device allocation (scratch)");
    if (!p) return false;
    cap = bytes;
    return true;
}
void DevBuf::release() {
    if (p) dev_free(p);
    p = nullptr;
    cap = 0;
}

SeriesStats compute_stats(const double* t, const double* y, size_t n) {
    SeriesStats s{};
    double sum = 0, sq = 0;
    for (size_t i = 0; i < n; i++) { sum += y[i]; sq += y[i] * y[i]; }
    s.mean = sum / (double)n;
    s.var_pop = sq / (double)n - s.mean * s.mean;  // carmcmc.cpp:85-88
    double ss = 0;
    for (size_t i = 0; i < n; i++) ss += (y[i] - s.mean) * (y[i] - s.mean);
    s.var_sample = n > 1 ? ss / (double)(n - 1) : 0.0;  // arma::var
    s.tmin = t[0];
    s.tmax = t[n - 1];
    if (n > 1) {
        std::vector<double> dt(n - 1);
        for (size_t i = 0; i + 1 < n; i++) dt[i] = t[i + 1] - t[i];
        std::sort(dt.begin(), dt.end());
        size_t m = dt.size();
        s.median_dt = (m % 2) ? dt[m / 2] : 0.5 * (dt[m / 2 - 1] + dt[m / 2]);
        s.min_dt = dt[0];
    } else {
        s.median_dt = s.min_dt = 1.0;
    }
    return s;
}

void prior_from_stats(const SeriesStats& st, int population_var, carma_prior_t* out) {
    out->max_stdev = 10.0 * std::sqrt(population_var ? st.var_pop : st.var_sample);
    out->max_freq = 1.0 / st.min_dt;
    out->min_freq = 1.0 / (st.tmax - st.tmin);
    out->kappa_high = 1.0 / st.min_dt;
    out->kappa_low = std::max(1.0 / (st.tmax - st.tmin), 1.0 / (10.0 * st.median_dt));
    out->measerr_dof = 50.0;
}

bool valid_model(int kind, int p, int q) {
    if (kind < CARMA_KIND_CAR1 || kind > CARMA_KIND_ZCARMA) return false;
    if (kind == CARMA_KIND_CAR1) return p == 1;
    if (p < 1 || p > MAX_P) return false;
    if (kind == CARMA_KIND_CARMA) return q >= 0 && q < p;
    return true;
}

}  // namespace carma

using namespace carma;

// =============================================================================================
// C ABI
// =============================================================================================
extern "C" {

const char* carma_last_error(void) { return g_last_error.c_str(); }
int carma_abi_version(void) { return CARMA_B200_ABI_VERSION; }

int carma_device_count(int* count) {
    if (!count) return CARMA_ERR_ARG;
    if (!cuda_ok(cudaGetDeviceCount(count), "cudaGetDeviceCount")) { *count = 0; return CARMA_ERR_CUDA; }
    return CARMA_OK;
}

int carma_series_create(const double* time, const double* y, const double* yerr, size_t ny, int device,
                        carma_series_t* out) {
    if (!time || !y || !yerr || !out || ny < 2) { set_error("carma_series_create: null pointer or ny < 2"); return CARMA_ERR_ARG; }
    for (size_t i = 0; i + 1 < ny; i++)
        if (!(time[i + 1] > time[i])) { set_error("carma_series_create: times must be strictly increasing"); return CARMA_ERR_ARG; }
    if (!cuda_ok(cudaSetDevice(device), "cudaSetDevice")) return CARMA_ERR_CUDA;
    carma_series* s = new (std::nothrow) carma_series();
    if (!s) return CARMA_ERR_ALLOC;
    s->device = device;
    s->ny = ny;
    s->nyp = (int)((ny + 1) & ~(size_t)1);
    s->t.assign(time, time + ny);
    s->y.assign(y, y + ny);
    s->yerr.assign(yerr, yerr + ny);
    s->st = compute_stats(time, y, ny);
    s->e2_0 = yerr[0] * yerr[0];
    s->dt_max = 0.0;
    for (size_t i = 0; i + 1 < ny; i++) s->dt_max = std::max(s->dt_max, time[i + 1] - time[i]);
    std::vector<double> pack(3 * (size_t)s->nyp + ny, 0.0);
    for (size_t i = 0; i < ny; i++) {
        pack[i] = (i + 1 < ny) ? time[i + 1] - time[i] : 0.0;
        pack[s->nyp + i] = y[i];
        pack[2 * (size_t)s->nyp + i] = (i + 1 < ny) ? yerr[i + 1] * yerr[i + 1] : 0.0;
        pack[3 * (size_t)s->nyp + i] = time[i];
    }
    s->d_pack = (double*)dev_alloc(pack.size() * sizeof(double), "device allocation (series)");
    if (!s->d_pack) { delete s; return CARMA_ERR_CUDA; }
    if (!cuda_ok(cudaMemcpy(s->d_pack, pack.data(), pack.size() * sizeof(double), cudaMemcpyHostToDevice), "cudaMemcpy(series)")) {
        dev_free(s->d_pack); delete s; return CARMA_ERR_CUDA;
    }
    *out = s;
    return CARMA_OK;
}

int carma_series_destroy(carma_series_t s) {
    if (!s) return CARMA_OK;
    cudaSetDevice(s->device);
    if (s->d_pack) dev_free(s->d_pack);
    s->scratch_in.release(); s->scratch_out.release(); s->scratch_misc.release(); s->scratch_state.release();
    for (int k = 0; k < CARMA_N_SLOTS; k++) {
        s->slot_in[k].release(); s->slot_out[k].release();
        if (s->slot_stream[k]) cudaStreamDestroy(s->slot_stream[k]);
    }
    for (int k = 0; k < 4; k++)
        if (s->blk_stream[k]) cudaStreamDestroy(s->blk_stream[k]);
    delete s;
    return CARMA_OK;
}

int carma_series_length(carma_series_t s, size_t* ny) {
    if (!s || !ny) return CARMA_ERR_ARG;
    *ny = s->ny;
    return CARMA_OK;
}

int carma_series_default_prior(carma_series_t s, int population_var, carma_prior_t* out) {
    if (!s || !out) return CARMA_ERR_ARG;
    prior_from_stats(s->st, population_var, out);
    return CARMA_OK;
}

int carma_loglik_batch_dev(carma_series_t s, int kind, int p, int q, const carma_prior_t* prior, size_t n,
                           const double* d_theta, double* d_logpost, unsigned flags, void* stream) {
    if (!s || !prior || (!d_theta && n) || (!d_logpost && n)) { set_error("carma_loglik_batch_dev: null argument"); return CARMA_ERR_ARG; }
    if (!valid_model(kind, p, q)) { set_error("carma_loglik_batch_dev: invalid (kind,p,q)"); return CARMA_ERR_ARG; }
    if (n == 0) return CARMA_OK;
    if (!cuda_ok(launch_loglik_batch(s->view(), kind, p, q, flags, *prior, d_theta, d_logpost, n, (cudaStream_t)stream),
                 "loglik_batch_kernel launch"))
        return CARMA_ERR_CUDA;
    return CARMA_OK;
}

int carma_loglik_batch(carma_series_t s, int kind, int p, int q, const carma_prior_t* prior, size_t n,
                       const double* theta, double* logpost, unsigned flags) {
    if (!s || !prior || (!theta && n) || (!logpost && n)) { set_error("carma_loglik_batch: null argument"); return CARMA_ERR_ARG; }
    if (!valid_model(kind, p, q)) { set_error("carma_loglik_batch: invalid (kind,p,q)"); return CARMA_ERR_ARG; }
    if (n == 0) return CARMA_OK;
    if (!cuda_ok(cudaSetDevice(s->device), "cudaSetDevice")) return CARMA_ERR_CUDA;
    size_t d = (size_t)model_dim(kind, p, q);
    if (!s->scratch_in.reserve(n * d * sizeof(double)) || !s->scratch_out.reserve(n * sizeof(double))) return CARMA_ERR_CUDA;
    // Large batches go as four pieces on four streams, so that the copy of a piece overlaps the kernels of the pieces
    // before it and the four kernels share the SMs like one launch (pinned host memory; with pageable memory the copies
    // are staged and nothing is lost).  Rows are independent and a row's arithmetic does not depend on its batch mates:
    // same bits as one launch.
    const size_t npieces = n >= 16384 ? 4 : 1;
    if (npieces > 1)
        for (int k = 0; k < 4; k++)
            if (!s->blk_stream[k] && !cuda_ok(cudaStreamCreateWithFlags(&s->blk_stream[k], cudaStreamNonBlocking), "cudaStreamCreate")) return CARMA_ERR_CUDA;
    const size_t per = ((n + npieces - 1) / npieces + 63) & ~(size_t)63;
    for (size_t k = 0, r0 = 0; k < npieces && r0 < n; k++, r0 += per) {
        const size_t nr = std::min(per, n - r0);
        cudaStream_t st = npieces > 1 ? s->blk_stream[k & 3] : (cudaStream_t)0;
        double* din = (double*)s->scratch_in.p + r0 * d;
        double* dout = (double*)s->scratch_out.p + r0;
        if (!cuda_ok(cudaMemcpyAsync(din, theta + r0 * d, nr * d * sizeof(double), cudaMemcpyHostToDevice, st), "H2D theta")) return CARMA_ERR_CUDA;
        int rc = carma_loglik_batch_dev(s, kind, p, q, prior, nr, din, dout, flags, st);
        if (rc) return rc;
        if (!cuda_ok(cudaMemcpyAsync(logpost + r0, dout, nr * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H logpost")) return CARMA_ERR_CUDA;
    }
    if (npieces > 1) {
        for (int k = 0; k < 4; k++)
            if (!cuda_ok(cudaStreamSynchronize(s->blk_stream[k]), "loglik_batch sync")) return CARMA_ERR_CUDA;
    } else if (!cuda_ok(cudaStreamSynchronize(0), "loglik_batch sync")) {
        return CARMA_ERR_CUDA;
    }
    return CARMA_OK;
}

int carma_loglik_batch_async(carma_series_t s, int kind, int p, int q, const carma_prior_t* prior, size_t n,
                             const double* theta, double* logpost, unsigned flags, int slot) {
    if (!s || !prior || (!theta && n) || (!logpost && n) || slot < 0 || slot >= CARMA_N_SLOTS) { set_error("carma_loglik_batch_async: bad argument"); return CARMA_ERR_ARG; }
    if (!valid_model(kind, p, q)) { set_error("carma_loglik_batch_async: invalid (kind,p,q)"); return CARMA_ERR_ARG; }
    if (n == 0) return CARMA_OK;
    if (!cuda_ok(cudaSetDevice(s->device), "cudaSetDevice")) return CARMA_ERR_CUDA;
    if (!s->slot_stream[slot] && !cuda_ok(cudaStreamCreateWithFlags(&s->slot_stream[slot], cudaStreamNonBlocking), "cudaStreamCreate")) return CARMA_ERR_CUDA;
    cudaStream_t st = s->slot_stream[slot];
    size_t d = (size_t)model_dim(kind, p, q);
    // growing a slot buffer must not race with work still queued on that slot
    if (n * d * sizeof(double) > s->slot_in[slot].cap || n * sizeof(double) > s->slot_out[slot].cap) {
        if (!cuda_ok(cudaStreamSynchronize(st), "slot sync")) return CARMA_ERR_CUDA;
        if (!s->slot_in[slot].reserve(n * d * sizeof(double)) || !s->slot_out[slot].reserve(n * sizeof(double))) return CARMA_ERR_CUDA;
    }
    if (!cuda_ok(cudaMemcpyAsync(s->slot_in[slot].p, theta, n * d * sizeof(double), cudaMemcpyHostToDevice, st), "H2D theta")) return CARMA_ERR_CUDA;
    int rc = carma_loglik_batch_dev(s, kind, p, q, prior, n, (const double*)s->slot_in[slot].p, (double*)s->slot_out[slot].p, flags, st);
    if (rc) return rc;
    if (!cuda_ok(cudaMemcpyAsync(logpost, s->slot_out[slot].p, n * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H logpost")) return CARMA_ERR_CUDA;
    return CARMA_OK;
}

int carma_loglik_batch_wait(carma_series_t s, int slot) {
    if (!s || slot < 0 || slot >= CARMA_N_SLOTS) { set_error("carma_loglik_batch_wait: bad argument"); return CARMA_ERR_ARG; }
    if (!s->slot_stream[slot]) return CARMA_OK;
    if (!cuda_ok(cudaSetDevice(s->device), "cudaSetDevice")) return CARMA_ERR_CUDA;
    if (!cuda_ok(cudaStreamSynchronize(s->slot_stream[slot]), "loglik_batch_wait")) return CARMA_ERR_CUDA;
    return CARMA_OK;
}

int carma_derived_params_dev(int kind, int p, int q, const carma_prior_t* prior, size_t n, const double* d_theta,
                             double* d_out, void* stream) {
    if ((!d_theta || !d_out) && n) { set_error("carma_derived_params_dev: null argument"); return CARMA_ERR_ARG; }
    if (!valid_model(kind, p, q)) { set_error("carma_derived_params_dev: invalid (kind,p,q)"); return CARMA_ERR_ARG; }
    if (kind == CARMA_KIND_ZCARMA && !prior) { set_error("carma_derived_params_dev: ZCARMA needs the prior (kappa bounds)"); return CARMA_ERR_ARG; }
    if (n == 0) return CARMA_OK;
    carma_prior_t pr{};
    if (prior) pr = *prior;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e;
    switch (p) {
        case 1: e = launch_derived<1>(kind, q, pr, d_theta, n, d_out, st); break;
        case 2: e = launch_derived<2>(kind, q, pr, d_theta, n, d_out, st); break;
        case 3: e = launch_derived<3>(kind, q, pr, d_theta, n, d_out, st); break;
        case 4: e = launch_derived<4>(kind, q, pr, d_theta, n, d_out, st); break;
        case 5: e = launch_derived<5>(kind, q, pr, d_theta, n, d_out, st); break;
        case 6: e = launch_derived<6>(kind, q, pr, d_theta, n, d_out, st); break;
        case 7: e = launch_derived<7>(kind, q, pr, d_theta, n, d_out, st); break;
        default: e = cudaErrorInvalidValue;
    }
    if (!cuda_ok(e, "derived_params_kernel launch")) return CARMA_ERR_CUDA;
    return CARMA_OK;
}

int carma_derived_params(int kind, int p, int q, const carma_prior_t* prior, size_t n, const double* theta, double* out,
                         int device) {
    if ((!theta || !out) && n) { set_error("carma_derived_params: null argument"); return CARMA_ERR_ARG; }
    if (!valid_model(kind, p, q)) { set_error("carma_derived_params: invalid (kind,p,q)"); return CARMA_ERR_ARG; }
    if (n == 0) return CARMA_OK;
    if (!cuda_ok(cudaSetDevice(device), "cudaSetDevice")) return CARMA_ERR_CUDA;
    const size_t d = (size_t)model_dim(kind, p, q), w = (size_t)(6 * p + 2);
    double *d_th = nullptr, *d_o = nullptr;
    if (!cuda_ok(cudaMalloc(&d_th, n * d * sizeof(double)), "cudaMalloc") || !cuda_ok(cudaMalloc(&d_o, n * w * sizeof(double)), "cudaMalloc")) {
        cudaFree(d_th);
        return CARMA_ERR_CUDA;
    }
    int rc = CARMA_ERR_CUDA;
    if (cuda_ok(cudaMemcpy(d_th, theta, n * d * sizeof(double), cudaMemcpyHostToDevice), "H2D theta")) {
        rc = carma_derived_params_dev(kind, p, q, prior, n, d_th, d_o, nullptr);
        if (rc == CARMA_OK && !cuda_ok(cudaMemcpy(out, d_o, n * w * sizeof(double), cudaMemcpyDeviceToHost), "D2H derived")) rc = CARMA_ERR_CUDA;
    }
    cudaFree(d_th);
    cudaFree(d_o);
    return rc;
}

int carma_log_prior(int kind, int p, const double* theta, const carma_prior_t* prior, double* out) {
    if (!theta || !prior || !out) return CARMA_ERR_ARG;
    double scale = theta[1];
    double lp = -0.5 * prior->measerr_dof / scale - (1.0 + prior->measerr_dof / 2.0) * std::log(scale);
    if (kind == CARMA_KIND_ZCARMA) {
        double x = theta[3 + p];
        lp += -x - 2.0 * std::log(1.0 + std::exp(-x));
    }
    *out = lp;
    return CARMA_OK;
}

// ---- multi-series ---------------------------------------------------------------------------
int carma_multi_series_create(const double* time, const double* y, const double* yerr, const int64_t* offsets,
                              size_t ncurves, int device, carma_multi_series_t* out) {
    if (!time || !y || !yerr || !offsets || !out || ncurves == 0) { set_error("carma_multi_series_create: null argument"); return CARMA_ERR_ARG; }
    if (!cuda_ok(cudaSetDevice(device), "cudaSetDevice")) return CARMA_ERR_CUDA;
    size_t total = (size_t)offsets[ncurves];
    carma_multi_series* m = new (std::nothrow) carma_multi_series();
    if (!m) return CARMA_ERR_ALLOC;
    m->device = device; m->ncurves = ncurves; m->total = total; m->dt_max = 0.0;
    m->off.assign(offsets, offsets + ncurves + 1);
    m->priors_pop.resize(ncurves); m->priors_sample.resize(ncurves);
    m->t0.resize(ncurves);
    std::vector<double> dt(total + 1, 0.0), e2(total + 1, 0.0);
    for (size_t c = 0; c < ncurves; c++) {
        size_t o0 = (size_t)offsets[c], o1 = (size_t)offsets[c + 1];
        if (o1 < o0 + 2) { set_error("carma_multi_series_create: every curve needs >= 2 points"); delete m; return CARMA_ERR_ARG; }
        m->max_ny = std::max(m->max_ny, (int)(o1 - o0));
        m->t0[c] = time[o0];
        double curve_dt_max = 0.0;
        for (size_t i = o0; i < o1; i++) {
            if (i + 1 < o1) {
                dt[i] = time[i + 1] - time[i];
                m->dt_max = std::max(m->dt_max, dt[i]);
                curve_dt_max = std::max(curve_dt_max, dt[i]);
                if (!(dt[i] > 0)) { set_error("carma_multi_series_create: times must be strictly increasing within a curve"); delete m; return CARMA_ERR_ARG; }
            }
            e2[i] = yerr[i] * yerr[i];
        }
        SeriesStats st = compute_stats(time + o0, y + o0, o1 - o0);
        prior_from_stats(st, 1, &m->priors_pop[c]);
        prior_from_stats(st, 0, &m->priors_sample[c]);
        CurveInfo ci;
        ci.prior = m->priors_pop[c];
        ci.y_mean = st.mean; ci.y_var_sample = st.var_sample; ci.y_var_pop = st.var_pop;
        ci.median_dt = st.median_dt; ci.tspan = st.tmax - st.tmin;
        ci.min_dt = st.min_dt; ci.dt_max = curve_dt_max;
        m->info.push_back(ci);
    }
    bool ok = cuda_ok(cudaMalloc((void**)&m->d_dt, (total + 1) * sizeof(double)), "cudaMalloc(multi dt)") &&
              cuda_ok(cudaMalloc((void**)&m->d_y, (total + 1) * sizeof(double)), "cudaMalloc(multi y)") &&
              cuda_ok(cudaMalloc((void**)&m->d_e2, (total + 1) * sizeof(double)), "cudaMalloc(multi e2)") &&
              cuda_ok(cudaMalloc((void**)&m->d_off, (ncurves + 1) * sizeof(long long)), "cudaMalloc(multi off)") &&
              cuda_ok(cudaMemcpy(m->d_dt, dt.data(), total * sizeof(double), cudaMemcpyHostToDevice), "H2D dt") &&
              cuda_ok(cudaMemcpy(m->d_y, y, total * sizeof(double), cudaMemcpyHostToDevice), "H2D y") &&
              cuda_ok(cudaMemcpy(m->d_e2, e2.data(), total * sizeof(double), cudaMemcpyHostToDevice), "H2D e2") &&
              cuda_ok(cudaMemcpy(m->d_off, m->off.data(), (ncurves + 1) * sizeof(long long), cudaMemcpyHostToDevice), "H2D off");
    if (!ok) { carma_multi_series_destroy(m); return CARMA_ERR_CUDA; }
    *out = m;
    return CARMA_OK;
}

int carma_multi_series_destroy(carma_multi_series_t m) {
    if (!m) return CARMA_OK;
    cudaSetDevice(m->device);
    if (m->d_dt) cudaFree(m->d_dt);
    if (m->d_y) cudaFree(m->d_y);
    if (m->d_e2) cudaFree(m->d_e2);
    if (m->d_off) cudaFree(m->d_off);
    m->scratch_in.release(); m->scratch_out.release(); m->scratch_pr.release(); m->scratch_misc.release();
    m->scratch_pts.release(); m->scratch_q.release();
    delete m;
    return CARMA_OK;
}

int carma_multi_series_default_priors(carma_multi_series_t m, int population_var, carma_prior_t* out) {
    if (!m || !out) return CARMA_ERR_ARG;
    const std::vector<carma_prior_t>& src = population_var ? m->priors_pop : m->priors_sample;
    std::memcpy(out, src.data(), src.size() * sizeof(carma_prior_t));
    return CARMA_OK;
}

int carma_multi_series_curve_stats(carma_multi_series_t m, carma_curve_stats_t* out) {
    if (!m || !out) { set_error("carma_multi_series_curve_stats: null argument"); return CARMA_ERR_ARG; }
    for (size_t c = 0; c < m->ncurves; c++) {
        const CurveInfo& ci = m->info[c];
        carma_curve_stats_t& o = out[c];
        o.y_mean = ci.y_mean; o.y_var_pop = ci.y_var_pop; o.y_var_sample = ci.y_var_sample;
        o.min_dt = ci.min_dt; o.median_dt = ci.median_dt; o.tspan = ci.tspan; o.dt_max = ci.dt_max;
        o.ny = m->off[c + 1] - m->off[c];
    }
    return CARMA_OK;
}

int carma_multi_loglik_dev(carma_multi_series_t m, int kind, int p, int q, const carma_prior_t* d_priors,
                           const double* d_theta, double* d_logpost, unsigned flags, void* stream) {
    if (!m || !d_priors || !d_theta || !d_logpost) { set_error("carma_multi_loglik_dev: null argument"); return CARMA_ERR_ARG; }
    if (!valid_model(kind, p, q)) { set_error("carma_multi_loglik_dev: invalid (kind,p,q)"); return CARMA_ERR_ARG; }
    if (!cuda_ok(launch_multi_loglik(m, kind, p, q, flags, d_priors, d_theta, d_logpost, (cudaStream_t)stream), "multi_loglik_kernel launch"))
        return CARMA_ERR_CUDA;
    return CARMA_OK;
}

int carma_multi_loglik(carma_multi_series_t m, int kind, int p, int q, const carma_prior_t* priors,
                       const double* theta, double* logpost, unsigned flags) {
    if (!m || !theta || !logpost) { set_error("carma_multi_loglik: null argument"); return CARMA_ERR_ARG; }
    if (!valid_model(kind, p, q)) { set_error("carma_multi_loglik: invalid (kind,p,q)"); return CARMA_ERR_ARG; }
    if (!cuda_ok(cudaSetDevice(m->device), "cudaSetDevice")) return CARMA_ERR_CUDA;
    size_t d = (size_t)model_dim(kind, p, q), n = m->ncurves;
    if (!m->scratch_in.reserve(n * d * sizeof(double)) || !m->scratch_out.reserve(n * sizeof(double)) ||
        !m->scratch_pr.reserve(n * sizeof(carma_prior_t)))
        return CARMA_ERR_CUDA;
    const carma_prior_t* hp = priors ? priors : m->priors_pop.data();
    cudaStream_t st = 0;
    if (!cuda_ok(cudaMemcpyAsync(m->scratch_pr.p, hp, n * sizeof(carma_prior_t), cudaMemcpyHostToDevice, st), "H2D priors")) return CARMA_ERR_CUDA;
    if (!cuda_ok(cudaMemcpyAsync(m->scratch_in.p, theta, n * d * sizeof(double), cudaMemcpyHostToDevice, st), "H2D theta")) return CARMA_ERR_CUDA;
    int rc = carma_multi_loglik_dev(m, kind, p, q, (const carma_prior_t*)m->scratch_pr.p, (const double*)m->scratch_in.p,
                                    (double*)m->scratch_out.p, flags, st);
    if (rc) return rc;
    if (!cuda_ok(cudaMemcpyAsync(logpost, m->scratch_out.p, n * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H logpost")) return CARMA_ERR_CUDA;
    if (!cuda_ok(cudaStreamSynchronize(st), "multi_loglik sync")) return CARMA_ERR_CUDA;
    return CARMA_OK;
}

// ---- explicit-parameter filter / predict ------------------------------------------------------
static int fill_filter_args(FilterArgs& a, double sigsqr, const double* omega_reim, const double* ma, int p,
                            double measerr_scale, double mu) {
    if (!omega_reim || !ma || p < 1 || p > MAX_P) { set_error("filter: invalid omega/ma/p"); return CARMA_ERR_ARG; }
    a.sigsqr = sigsqr; a.scale = measerr_scale; a.mu = mu; a.p = p;
    for (int i = 0; i < 2 * MAX_P; i++) a.omega[i] = i < 2 * p ? omega_reim[i] : 0.0;
    for (int i = 0; i < MAX_P; i++) a.ma[i] = i < p ? ma[i] : 0.0;
    return CARMA_OK;
}

int carma_filter(carma_series_t s, double sigsqr, const double* omega_reim, const double* ma, int p,
                 double measerr_scale, double mu, double* mean, double* var) {
    if (!s || !mean || !var) { set_error("carma_filter: null argument"); return CARMA_ERR_ARG; }
    FilterArgs a;
    int rc = fill_filter_args(a, sigsqr, omega_reim, ma, p, measerr_scale, mu);
    if (rc) return rc;
    if (!cuda_ok(cudaSetDevice(s->device), "cudaSetDevice")) return CARMA_ERR_CUDA;
    size_t ny = s->ny;
    if (!s->scratch_out.reserve((2 * ny + 2) * sizeof(double))) return CARMA_ERR_CUDA;
    double* d_mean = (double*)s->scratch_out.p;
    double* d_var = d_mean + ny;
    int* d_status = (int*)(d_var + ny);
    // roots closed under conjugation (every physical model): the time-parallel real-half filter (scan.cu) writes
    // mean / var of all points; otherwise the general complex recursion on one thread
    ExplicitModel ex;
    const char* env_general = getenv("CARMA_PREDICT_GENERAL");
    if (!(env_general && env_general[0] == '1') && arrange_roots(omega_reim, ma, p, sigsqr, measerr_scale, mu, &ex)) {
        double* d_ll = (double*)d_status;
        int rc2 = scan_explicit(s, p, ex, d_mean, d_var, nullptr, d_ll, 0);
        if (rc2) return rc2;
        double ll = 0.0;
        if (!cuda_ok(cudaMemcpy(&ll, d_ll, sizeof(double), cudaMemcpyDeviceToHost), "D2H loglik")) return CARMA_ERR_CUDA;
        if (std::isfinite(ll) || std::isnan(ll)) {   // -inf = the constants could not be formed: let the complex path report it
            if (!cuda_ok(cudaMemcpy(mean, d_mean, ny * sizeof(double), cudaMemcpyDeviceToHost), "D2H mean")) return CARMA_ERR_CUDA;
            if (!cuda_ok(cudaMemcpy(var, d_var, ny * sizeof(double), cudaMemcpyDeviceToHost), "D2H var")) return CARMA_ERR_CUDA;
            return CARMA_OK;
        }
    }
    filter_kernel<<<1, 32>>>(s->view(), a, d_mean, d_var, d_status);
    if (!cuda_ok(cudaGetLastError(), "filter_kernel launch")) return CARMA_ERR_CUDA;
    int status = 0;
    if (!cuda_ok(cudaMemcpy(&status, d_status, sizeof(int), cudaMemcpyDeviceToHost), "D2H status")) return CARMA_ERR_CUDA;
    if (status) {
        // singular Vandermonde system: the reference throws from arma::solve (kfilter.cpp:158)
        for (size_t i = 0; i < ny; i++) { mean[i] = std::numeric_limits<double>::quiet_NaN(); var[i] = mean[i]; }
        return CARMA_OK;
    }
    if (!cuda_ok(cudaMemcpy(mean, d_mean, ny * sizeof(double), cudaMemcpyDeviceToHost), "D2H mean")) return CARMA_ERR_CUDA;
    if (!cuda_ok(cudaMemcpy(var, d_var, ny * sizeof(double), cudaMemcpyDeviceToHost), "D2H var")) return CARMA_ERR_CUDA;
    return CARMA_OK;
}

int carma_predict(carma_series_t s, double sigsqr, const double* omega_reim, const double* ma, int p,
                  double measerr_scale, double mu, const double* tq, size_t nq, double* qmean, double* qvar) {
    if (!s || !tq || !qmean || !qvar) { set_error("carma_predict: null argument"); return CARMA_ERR_ARG; }
    if (nq == 0) return CARMA_OK;
    FilterArgs a;
    int rc = fill_filter_args(a, sigsqr, omega_reim, ma, p, measerr_scale, mu);
    if (rc) return rc;
    if (!cuda_ok(cudaSetDevice(s->device), "cudaSetDevice")) return CARMA_ERR_CUDA;
    if (!s->scratch_in.reserve(nq * sizeof(double)) || !s->scratch_out.reserve((2 * nq + 2) * sizeof(double))) return CARMA_ERR_CUDA;
    double* d_tq = (double*)s->scratch_in.p;
    double* d_m = (double*)s->scratch_out.p;
    double* d_v = d_m + nq;
    int* d_status = (int*)(d_v + nq);
    if (!cuda_ok(cudaMemset(d_status, 0, sizeof(int)), "memset status")) return CARMA_ERR_CUDA;
    if (!cuda_ok(cudaMemcpy(d_tq, tq, nq * sizeof(double), cudaMemcpyHostToDevice), "H2D tq")) return CARMA_ERR_CUDA;
    // fast path: one time-parallel forward filter leaves the predicted state at every data point; every query resumes
    // from the state in front of it (real-half recursion).  Needs conjugate-symmetric roots and room for the states.
    ExplicitModel ex;
    const size_t state_doubles = (size_t)s->ny * (size_t)(p + p * (p + 1) / 2);
    const char* env_general = getenv("CARMA_PREDICT_GENERAL");   // "1": force the general complex kernel (tests, timing)
    const bool force_general = env_general && env_general[0] == '1';
    if (!force_general && state_doubles * sizeof(double) <= ((size_t)1 << 30) &&
        arrange_roots(omega_reim, ma, p, sigsqr, measerr_scale, mu, &ex)) {
        if (!s->scratch_state.reserve((state_doubles + 2) * sizeof(double))) return CARMA_ERR_CUDA;
        double* d_state = (double*)s->scratch_state.p;
        double* d_ll = d_state + state_doubles;
        int rc2 = scan_explicit(s, p, ex, nullptr, nullptr, d_state, d_ll, 0);
        if (rc2) return rc2;
        double ll = 0.0;
        if (!cuda_ok(cudaMemcpy(&ll, d_ll, sizeof(double), cudaMemcpyDeviceToHost), "D2H loglik")) return CARMA_ERR_CUDA;
        if (std::isfinite(ll) || std::isnan(ll)) {
            const unsigned g64 = (unsigned)((nq + 63) / 64);
            SeriesView sv = s->view();
#define LAUNCH_PR(PP) predict_real_kernel<PP><<<g64, 64>>>(sv, ex, d_state, d_tq, nq, d_m, d_v)
            switch (p) {
                case 1: LAUNCH_PR(1); break;
                case 2: LAUNCH_PR(2); break;
                case 3: LAUNCH_PR(3); break;
                case 4: LAUNCH_PR(4); break;
                case 5: LAUNCH_PR(5); break;
                case 6: LAUNCH_PR(6); break;
                default: LAUNCH_PR(7); break;
            }
#undef LAUNCH_PR
            if (!cuda_ok(cudaGetLastError(), "predict_real_kernel launch")) return CARMA_ERR_CUDA;
            if (!cuda_ok(cudaMemcpy(qmean, d_m, nq * sizeof(double), cudaMemcpyDeviceToHost), "D2H qmean")) return CARMA_ERR_CUDA;
            if (!cuda_ok(cudaMemcpy(qvar, d_v, nq * sizeof(double), cudaMemcpyDeviceToHost), "D2H qvar")) return CARMA_ERR_CUDA;
            return CARMA_OK;
        }
    }
    unsigned grid = (unsigned)((nq + 31) / 32);
    predict_kernel<<<grid, 32>>>(s->view(), a, d_tq, nq, d_m, d_v, d_status);
    if (!cuda_ok(cudaGetLastError(), "predict_kernel launch")) return CARMA_ERR_CUDA;
    if (!cuda_ok(cudaMemcpy(qmean, d_m, nq * sizeof(double), cudaMemcpyDeviceToHost), "D2H qmean")) return CARMA_ERR_CUDA;
    if (!cuda_ok(cudaMemcpy(qvar, d_v, nq * sizeof(double), cudaMemcpyDeviceToHost), "D2H qvar")) return CARMA_ERR_CUDA;
    return CARMA_OK;
}

// ---- conditional simulation -------------------------------------------------------------------
int carma_simulate(carma_series_t s, double sigsqr, const double* omega_reim, const double* ma, int p, double measerr_scale,
                   double mu, const double* tsim, size_t nsim, uint64_t seed, size_t npaths, double* ysim) {
    if (!s || !omega_reim || !ma || !tsim || !ysim) { set_error("carma_simulate: null argument"); return CARMA_ERR_ARG; }
    if (nsim == 0 || npaths == 0) return CARMA_OK;
    ExplicitModel ex;
    if (!arrange_roots(omega_reim, ma, p, sigsqr, measerr_scale, mu, &ex)) {
        set_error("carma_simulate: the AR roots must be distinct and closed under complex conjugation (1 <= p <= 7)");
        return CARMA_ERR_ARG;
    }
    for (size_t i = 0; i < nsim; i++)
        if (!std::isfinite(tsim[i])) { set_error("carma_simulate: non-finite time"); return CARMA_ERR_ARG; }
    if (!cuda_ok(cudaSetDevice(s->device), "cudaSetDevice")) return CARMA_ERR_CUDA;
    const size_t ny = s->ny, nm = ny + nsim;
    // merged grid: data points and requested points in time order (a requested time equal to a data time follows it)
    std::vector<size_t> order(nsim);
    for (size_t i = 0; i < nsim; i++) order[i] = i;
    std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) { return tsim[a] < tsim[b]; });
    std::vector<double> tm(nm), dtm(nm, 0.0);
    std::vector<int> idx(nm);
    size_t a = 0, b = 0;
    for (size_t k = 0; k < nm; k++) {
        if (b >= nsim || (a < ny && s->t[a] <= tsim[order[b]])) { tm[k] = s->t[a]; idx[k] = (int)a; a++; }
        else { tm[k] = tsim[order[b]]; idx[k] = -(int)order[b] - 1; b++; }
    }
    double dt_max = s->dt_max;
    for (size_t k = 0; k + 1 < nm; k++) { dtm[k] = tm[k + 1] - tm[k]; dt_max = std::max(dt_max, dtm[k]); }
    const size_t state_doubles = ny * (size_t)(p + p * (p + 1) / 2);
    char* base = nullptr;
    auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const size_t b_dtm = al(nm * 8), b_idx = al(nm * 4), b_yerr = al(ny * 8), b_yres = al(npaths * ny * 8), b_fsim = al(npaths * nsim * 8),
                 b_tq = al(nsim * 8), b_state = al((state_doubles + 2) * 8), b_out = al(npaths * nsim * 8);
    if (!cuda_ok(cudaMalloc((void**)&base, b_dtm + b_idx + b_yerr + b_yres + b_fsim + b_tq + b_state + b_out), "cudaMalloc(simulate)"))
        return CARMA_ERR_CUDA;
    double* d_dtm = (double*)base;
    int* d_idx = (int*)(base + b_dtm);
    double* d_yerr = (double*)(base + b_dtm + b_idx);
    double* d_yres = (double*)((char*)d_yerr + b_yerr);
    double* d_fsim = (double*)((char*)d_yres + b_yres);
    double* d_tq = (double*)((char*)d_fsim + b_fsim);
    double* d_state = (double*)((char*)d_tq + b_tq);
    double* d_ll = d_state + state_doubles;
    double* d_out = (double*)((char*)d_state + b_state);
    SeriesView sv = s->view();
    bool ok = cuda_ok(cudaMemcpy(d_dtm, dtm.data(), nm * 8, cudaMemcpyHostToDevice), "H2D dtm") &&
              cuda_ok(cudaMemcpy(d_idx, idx.data(), nm * 4, cudaMemcpyHostToDevice), "H2D idx") &&
              cuda_ok(cudaMemcpy(d_yerr, s->yerr.data(), ny * 8, cudaMemcpyHostToDevice), "H2D yerr") &&
              cuda_ok(cudaMemcpy(d_tq, tsim, nsim * 8, cudaMemcpyHostToDevice), "H2D tsim");
    int rc = CARMA_OK;
    if (ok) {
        const unsigned g = (unsigned)((npaths + 63) / 64);
#define LAUNCH_SP(PP) sim_prior_kernel<PP><<<g, 64>>>(ex, dt_max, (int)nm, d_dtm, d_idx, sv.y, d_yerr, (int)ny, (int)nsim, seed, (int)npaths, d_yres, (int)ny, d_fsim)
        switch (p) {
            case 1: LAUNCH_SP(1); break;
            case 2: LAUNCH_SP(2); break;
            case 3: LAUNCH_SP(3); break;
            case 4: LAUNCH_SP(4); break;
            case 5: LAUNCH_SP(5); break;
            case 6: LAUNCH_SP(6); break;
            default: LAUNCH_SP(7); break;
        }
#undef LAUNCH_SP
        ok = cuda_ok(cudaGetLastError(), "sim_prior_kernel launch");
    }
    ExplicitModel ex0 = ex;
    ex0.mu = 0.0;   // the residual data are already centred
    for (size_t path = 0; ok && path < npaths; path++) {
        const double* d_y = d_yres + path * ny;
        rc = scan_explicit(s, p, ex0, nullptr, nullptr, d_state, d_ll, 0, d_y);
        if (rc) { ok = false; break; }
        SeriesView svp = sv;
        svp.y = d_y;
        const unsigned g64 = (unsigned)((nsim + 63) / 64);
#define LAUNCH_PR(PP) predict_real_kernel<PP><<<g64, 64>>>(svp, ex0, d_state, d_tq, nsim, d_out + path * nsim, nullptr)
        switch (p) {
            case 1: LAUNCH_PR(1); break;
            case 2: LAUNCH_PR(2); break;
            case 3: LAUNCH_PR(3); break;
            case 4: LAUNCH_PR(4); break;
            case 5: LAUNCH_PR(5); break;
            case 6: LAUNCH_PR(6); break;
            default: LAUNCH_PR(7); break;
        }
#undef LAUNCH_PR
        ok = cuda_ok(cudaGetLastError(), "predict_real_kernel launch");
    }
    if (ok) {
        const size_t n = npaths * nsim;
        add_prior_kernel<<<(unsigned)((n + 255) / 256), 256>>>(d_fsim, mu, n, d_out);
        ok = cuda_ok(cudaGetLastError(), "add_prior_kernel launch") &&
             cuda_ok(cudaMemcpy(ysim, d_out, n * 8, cudaMemcpyDeviceToHost), "D2H ysim");
    }
    cudaFree(base);
    if (rc) return rc;
    return ok ? CARMA_OK : CARMA_ERR_CUDA;
}

// ---- utilities --------------------------------------------------------------------------------
int carma_fp64_peak_tflops(int device, double* tflops) {
    if (!tflops) return CARMA_ERR_ARG;
    if (!cuda_ok(cudaSetDevice(device), "cudaSetDevice")) return CARMA_ERR_CUDA;
    cudaDeviceProp prop;
    if (!cuda_ok(cudaGetDeviceProperties(&prop, device), "cudaGetDeviceProperties")) return CARMA_ERR_CUDA;
    double* d_out = nullptr;
    if (!cuda_ok(cudaMalloc((void**)&d_out, sizeof(double)), "cudaMalloc")) return CARMA_ERR_CUDA;
    int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 1 << 16;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    dfma_peak_kernel<<<blocks, threads>>>(d_out, 1 << 12, 1.0000001, 1e-9);  // warm-up
    double best = 0.0;
    for (int rep = 0; rep < 3; rep++) {
        cudaEventRecord(e0);
        dfma_peak_kernel<<<blocks, threads>>>(d_out, iters, 1.0000001, 1e-9);
        cudaEventRecord(e1);
        if (!cuda_ok(cudaEventSynchronize(e1), "dfma_peak sync")) { cudaFree(d_out); return CARMA_ERR_CUDA; }
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        double fl = 2.0 * 8.0 * (double)iters * (double)blocks * (double)threads;
        best = std::max(best, fl / (ms * 1e-3) / 1e12);
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(d_out);
    *tflops = best;
    return CARMA_OK;
}

int carma_fastmath_dev(const double* rate, const double* dt, size_t n, double* out_exp, double* out_sin, double* out_cos,
                       double* out_sh, double* out_ch, double* out_rcp) {
    if (!rate || !dt || !out_exp || !out_sin || !out_cos || !out_sh || !out_ch || !out_rcp) return CARMA_ERR_ARG;
    if (n == 0) return CARMA_OK;
    double* d = nullptr;
    if (!cuda_ok(cudaMalloc((void**)&d, 8 * n * sizeof(double)), "cudaMalloc")) return CARMA_ERR_CUDA;
    bool ok = cuda_ok(cudaMemcpy(d, rate, n * sizeof(double), cudaMemcpyHostToDevice), "H2D rate") &&
              cuda_ok(cudaMemcpy(d + n, dt, n * sizeof(double), cudaMemcpyHostToDevice), "H2D dt");
    if (ok) {
        fastmath_kernel<<<(unsigned)((n + 127) / 128), 128>>>(d, d + n, n, d + 2 * n, d + 3 * n, d + 4 * n, d + 5 * n, d + 6 * n, d + 7 * n);
        double* outs[6] = {out_exp, out_sin, out_cos, out_sh, out_ch, out_rcp};
        ok = cuda_ok(cudaGetLastError(), "fastmath_kernel launch");
        for (int k = 0; k < 6 && ok; k++)
            ok = cuda_ok(cudaMemcpy(outs[k], d + (2 + k) * n, n * sizeof(double), cudaMemcpyDeviceToHost), "D2H");
    }
    cudaFree(d);
    return ok ? CARMA_OK : CARMA_ERR_CUDA;
}

int carma_philox_dev(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint64_t seed, uint32_t* out4) {
    if (!out4) return CARMA_ERR_ARG;
    uint32_t* d = nullptr;
    if (!cuda_ok(cudaMalloc((void**)&d, 4 * sizeof(uint32_t)), "cudaMalloc")) return CARMA_ERR_CUDA;
    philox_kernel<<<1, 1>>>(c0, c1, c2, c3, seed, d);
    bool ok = cuda_ok(cudaMemcpy(out4, d, 4 * sizeof(uint32_t), cudaMemcpyDeviceToHost), "philox D2H");
    cudaFree(d);
    return ok ? CARMA_OK : CARMA_ERR_CUDA;
}

int carma_tdist_dev(uint64_t seed, uint32_t chain, uint32_t iter, uint32_t j, int dof, double* out) {
    if (!out) return CARMA_ERR_ARG;
    double* d = nullptr;
    if (!cuda_ok(cudaMalloc((void**)&d, sizeof(double)), "cudaMalloc")) return CARMA_ERR_CUDA;
    tdist_kernel<<<1, 1>>>(seed, chain, iter, j, dof, d);
    bool ok = cuda_ok(cudaMemcpy(out, d, sizeof(double), cudaMemcpyDeviceToHost), "tdist D2H");
    cudaFree(d);
    return ok ? CARMA_OK : CARMA_ERR_CUDA;
}

}  // extern "C"
