// posterior.cu -- survey-scale summaries of MCMC samples: what CarmaSample / MCMCSample compute from one curve's trace,
// for the traces of many curves at once, without the per-sample arrays crossing PCIe.
//   psd_rows_kernel<P>          one thread = one theta row: derive_row (shared with derived_params_kernel) -> the row of
//                               the PSD kernels, [ sigma^2 | roots (re, im) x P | beta x P ];
//   psd_band_shared_kernel<P>   one block = FT frequencies of one curve: the PSD of every sample at those frequencies into
//                               shared memory, a bitonic sort per column, then the percentiles;
//   psd_eval_kernel<P>          the global-memory path for columns too long for shared memory: the PSD of every sample
//   psd_select_global_kernel    into a (curve, frequency, sample) scratch array, then one block per column selects the
//                               order statistics by a radix select on the order-preserving 64-bit key of the double;
//   effective_samples_kernel    one warp = one column of one series: MCMCSample.effective_samples.
// The percentiles are np.percentile(psd, pct, axis=0) (method "linear") of the kernel's own PSD values, bit for bit:
// the same two order statistics and the same interpolation (numpy's _lerp), written without FMA contraction.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <string>

#include "select.cuh"
#include "theta_transform.cuh"
#include "series.h"

namespace carma {

constexpr int PSD_THREADS = 256;
constexpr int PSD_TILE_KEYS = 8192;   // keys a shared-path block aims for: several frequencies of a short column
constexpr double TWO_PI = 6.283185307179586;   // 2.0 * np.pi

template <int P>
__host__ __device__ constexpr int psd_row_width() { return 1 + 3 * P; }

// numpy's _lerp(a, b, t): a + (b - a) t, or b - (b - a)(1 - t) where t >= 0.5, each operation rounded on its own
__device__ __forceinline__ double np_lerp(double a, double b, double t) {
    const double d = __dsub_rn(b, a);
    return t >= 0.5 ? __dsub_rn(b, __dmul_rn(d, __dsub_rn(1.0, t))) : __dadd_rn(a, __dmul_rn(d, t));
}

// np.percentile's index arithmetic for n values: g = pct / 100, v = (n - 1) g, k = floor(v), t = v - k.  false for a
// percentile outside [0, 100] (the _dev entry point cannot check them on the host).
__device__ __forceinline__ bool pct_index(double pct, size_t n, size_t* k, double* t) {
    const double g = __ddiv_rn(pct, 100.0);
    if (!(g >= 0.0 && g <= 1.0)) return false;
    const double v = __dmul_rn((double)(n - 1), g);
    const double fl = floor(v);
    *k = (size_t)fl;
    *t = __dsub_rn(v, fl);
    return true;
}

template <int P>
__global__ void __launch_bounds__(128) psd_rows_kernel(int kind, int q, const carma_prior_t* __restrict__ priors,
                                                       const double* __restrict__ theta, size_t nrows, size_t nsamples,
                                                       double* __restrict__ rows) {
    const size_t r = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nrows) return;
    const int d = model_dim(kind, P, q);
    carma_prior_t pr{};
    if (priors) pr = priors[r / nsamples];
    cxd w[P];
    double ma[P];
    const double sigma = sqrt(derive_row<P>(kind, q, pr, theta + r * (size_t)d, w, ma));   // CarmaSample's sigma
    double* o = rows + r * psd_row_width<P>();
    o[0] = sigma * sigma;
#pragma unroll
    for (int k = 0; k < P; k++) {
        o[1 + 2 * k] = w[k].re;
        o[2 + 2 * k] = w[k].im;
        o[1 + 2 * P + k] = ma[k];
    }
}

// PSD(f) = sigma^2 |sum_{k<=nb} beta_k (2 pi i f)^k|^2 / prod_k |2 pi i f - w_k|^2, the numerator by Horner; every operation
// rounded on its own so that a host evaluation in the same order reproduces it.  Non-finite values become NaN.
template <int P>
__device__ __forceinline__ double psd_value(const double* __restrict__ row, int nb, double f) {
    const double om = __dmul_rn(TWO_PI, f);
    double nr = row[1 + 2 * P + nb], ni = 0.0;
    for (int k = nb - 1; k >= 0; k--) {
        const double r = __dsub_rn(row[1 + 2 * P + k], __dmul_rn(ni, om));
        ni = __dmul_rn(nr, om);
        nr = r;
    }
    const double num = __dadd_rn(__dmul_rn(nr, nr), __dmul_rn(ni, ni));
    double den = 1.0;
#pragma unroll
    for (int k = 0; k < P; k++) {
        const double dr = -row[1 + 2 * k], di = __dsub_rn(om, row[2 + 2 * k]);
        den = __dmul_rn(den, __dadd_rn(__dmul_rn(dr, dr), __dmul_rn(di, di)));
    }
    const double v = __ddiv_rn(__dmul_rn(row[0], num), den);
    return isfinite(v) ? v : (double)NAN;
}

struct BandArgs {
    const double* rows;      // ncurves * ns rows of psd_row_width<P>()
    int nb;                  // degree of the MA polynomial
    size_t nc, ns, nf;
    const double* freq;      // freq_stride = 0 (one row) or nf (one row per curve)
    size_t freq_stride;
    const double* pct;
    size_t npct;
    double* out;             // (c * npct + j) * nf + f
    double* psd_out;         // (c * ns + s) * nf + f, or null
};

constexpr int PSD_MAX_FT = 256;   // frequencies per shared-path block

// Shared path: block = (curve, tile of FT frequencies); keys[ft * n2 + s], n2 = 2^lg the power of two >= ns, the padding
// holding the largest key so that it sorts last; a bitonic sort orders every column of the tile at once.  FT * n2 <=
// 16384, so the indices are 32-bit and every division by a power of two is a shift or a mask.  (A radix
// select on the shared column instead of the sort took 2.5x as long at 10^4 curves x 1000 samples x 200 frequencies:
// DESIGN.md.)
template <int P>
__global__ void __launch_bounds__(PSD_THREADS) psd_band_shared_kernel(BandArgs a, int FT, int lg) {
    extern __shared__ unsigned long long keys[];
    __shared__ int has_nan[PSD_MAX_FT];
    const size_t ntiles = (a.nf + FT - 1) / FT;
    const size_t c = blockIdx.x / ntiles, f0 = (blockIdx.x % ntiles) * FT;
    const int nft = (int)(FT < a.nf - f0 ? FT : a.nf - f0);
    const double* fr = a.freq + c * a.freq_stride + f0;
    const double* rows = a.rows + c * a.ns * psd_row_width<P>();
    for (int i = threadIdx.x; i < nft; i += blockDim.x) has_nan[i] = 0;
    __syncthreads();
    const unsigned n2 = 1u << lg;
    for (unsigned i = threadIdx.x; i < ((unsigned)nft << lg); i += blockDim.x) {
        const int ft = (int)(i >> lg);
        const unsigned s = i & (n2 - 1);
        unsigned long long k = ~0ull;
        if (s < a.ns) {
            const double v = psd_value<P>(rows + s * psd_row_width<P>(), a.nb, fr[ft]);
            if (a.psd_out) a.psd_out[(c * a.ns + s) * a.nf + f0 + ft] = v;
            if (isnan(v)) has_nan[ft] = 1;
            k = order_key(v);
        }
        keys[i] = k;
    }
    __syncthreads();
    const unsigned pairs = lg > 0 ? (unsigned)nft << (lg - 1) : 0u;
    for (int lsz = 1; lsz <= lg; lsz++) {            // merge size 2^lsz
        for (int lst = lsz - 1; lst >= 0; lst--) {   // stride 2^lst
            for (unsigned i = threadIdx.x; i < pairs; i += blockDim.x) {
                const unsigned col = i >> (lg - 1), j = i & ((n2 >> 1) - 1);
                const unsigned lo = ((j >> lst) << (lst + 1)) | (j & ((1u << lst) - 1)), hi = lo + (1u << lst);
                unsigned long long* kc = keys + (col << lg);
                const unsigned long long x = kc[lo], y = kc[hi];
                if ((x > y) == (((lo >> lsz) & 1u) == 0)) { kc[lo] = y; kc[hi] = x; }
            }
            __syncthreads();
        }
    }
    for (size_t i = threadIdx.x; i < (size_t)nft * a.npct; i += blockDim.x) {
        const int ft = (int)(i / a.npct);
        const size_t j = i % a.npct;
        size_t k;
        double t, r = NAN;
        if (!has_nan[ft] && pct_index(a.pct[j], a.ns, &k, &t))
            r = np_lerp(key_value(keys[ft * n2 + k]), key_value(keys[ft * n2 + (k + 1 < a.ns ? k + 1 : k)]), t);
        a.out[(c * a.npct + j) * a.nf + f0 + ft] = r;
    }
}

// Global path, step 1: one thread = one (curve, sample) row, all frequencies; scratch[(c * nf + f) * ns + s].
template <int P>
__global__ void __launch_bounds__(128) psd_eval_kernel(BandArgs a, double* __restrict__ scratch) {
    const size_t r = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= a.nc * a.ns) return;
    const size_t c = r / a.ns, s = r % a.ns;
    const double* row = a.rows + r * psd_row_width<P>();
    const double* fr = a.freq + c * a.freq_stride;
    for (size_t f = 0; f < a.nf; f++) {
        const double v = psd_value<P>(row, a.nb, fr[f]);
        scratch[(c * a.nf + f) * a.ns + s] = v;
        if (a.psd_out) a.psd_out[r * a.nf + f] = v;
    }
}

// Global path, step 2: one block = one (curve, frequency) column.
__global__ void __launch_bounds__(PSD_THREADS) psd_select_global_kernel(BandArgs a, const double* __restrict__ scratch) {
    __shared__ SelectSmem sm;
    __shared__ int has_nan;
    const size_t col = blockIdx.x, c = col / a.nf, f = col % a.nf;
    const double* x = scratch + col * a.ns;
    if (threadIdx.x == 0) has_nan = 0;
    __syncthreads();
    for (size_t i = threadIdx.x; i < a.ns; i += blockDim.x)
        if (isnan(x[i])) has_nan = 1;
    __syncthreads();
    for (size_t j = 0; j < a.npct; j++) {
        size_t k;
        double t, r = NAN;
        if (!has_nan && pct_index(a.pct[j], a.ns, &k, &t)) {
            unsigned long long ka, kb;
            block_select_pair(x, a.ns, k, sm, &ka, &kb);
            r = np_lerp(key_value(ka), key_value(kb), t);
        }
        if (threadIdx.x == 0) a.out[(c * a.npct + j) * a.nf + f] = r;
    }
}

template <int P>
static cudaError_t launch_band(int kind, int q, const carma_prior_t* d_priors, const double* d_theta, BandArgs a,
                               bool global, cudaStream_t st) {
    const size_t nrows = a.nc * a.ns;
    double* d_rows = nullptr;
    double* d_scr = nullptr;
    cudaError_t e = cudaMallocAsync((void**)&d_rows, nrows * psd_row_width<P>() * sizeof(double), st);
    if (e != cudaSuccess) return e;
    a.rows = d_rows;
    psd_rows_kernel<P><<<(unsigned)((nrows + 127) / 128), 128, 0, st>>>(kind, q, d_priors, d_theta, nrows, a.ns, d_rows);
    e = cudaGetLastError();
    int lg = 0;
    while (((size_t)1 << lg) < a.ns) lg++;
    const size_t n2 = (size_t)1 << lg;
    int dev = 0, optin = 0;
    if (e == cudaSuccess) e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    const size_t static_smem = sizeof(int) * PSD_MAX_FT;
    if (!global && n2 * sizeof(unsigned long long) + static_smem > (size_t)optin) global = true;
    if (e == cudaSuccess && !global) {
        const int FT = (int)std::max<size_t>(1, std::min<size_t>(std::min<size_t>(a.nf, PSD_MAX_FT), PSD_TILE_KEYS / n2));
        const size_t smem = (size_t)FT * n2 * sizeof(unsigned long long);
        const size_t blocks = a.nc * ((a.nf + FT - 1) / FT);
        e = cudaFuncSetAttribute(psd_band_shared_kernel<P>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess) {
            psd_band_shared_kernel<P><<<(unsigned)blocks, PSD_THREADS, smem, st>>>(a, FT, lg);
            e = cudaGetLastError();
        }
    } else if (e == cudaSuccess) {
        e = cudaMallocAsync((void**)&d_scr, nrows * a.nf * sizeof(double), st);
        if (e == cudaSuccess) {
            psd_eval_kernel<P><<<(unsigned)((nrows + 127) / 128), 128, 0, st>>>(a, d_scr);
            e = cudaGetLastError();
        }
        if (e == cudaSuccess) {
            psd_select_global_kernel<<<(unsigned)(a.nc * a.nf), PSD_THREADS, 0, st>>>(a, d_scr);
            e = cudaGetLastError();
        }
    }
    if (d_scr) cudaFreeAsync(d_scr, st);
    cudaFreeAsync(d_rows, st);
    return e;
}

__device__ __forceinline__ double warp_sum(double v) {   // butterfly: every lane ends with the same, order-fixed sum
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// MCMCSample.effective_samples of column `col` of series s: r = x - mean, ac[j] = sum r_i r_{i+j} / max(sum r^2, 1e-300),
// tau = 1 + 2 sum ac[j] while ac[j] > 0.05, ess = n / tau.  Lags one at a time until the cutoff: O(n * lags used).
// Lane l sums the terms i = l, l + 32, ... in order, then a butterfly: the result depends on n only.  A column whose
// values are all equal gets ess = n: the residuals are zero (numpy's answer whenever its mean of the column is exact; when
// that mean rounds, numpy's residuals are a constant offset, ac[j] ~ 1 - j/n and its ess collapses towards 1).
__global__ void __launch_bounds__(256) effective_samples_kernel(size_t nseries, size_t n, size_t k, const double* __restrict__ x,
                                                                double* __restrict__ ess) {
    const size_t g = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) / 32;
    const unsigned lane = threadIdx.x & 31u;
    if (g >= nseries * k) return;
    const double* xs = x + (g / k) * n * k + (g % k);
    double sum = 0.0, lo = xs[0], hi = xs[0];
    for (size_t i = lane; i < n; i += 32) {
        const double v = xs[i * k];
        sum += v;
        lo = fmin(lo, v);
        hi = fmax(hi, v);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lo = fmin(lo, __shfl_xor_sync(0xffffffffu, lo, o));
        hi = fmax(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
    if (lo == hi) {
        if (lane == 0) ess[g] = (double)n;
        return;
    }
    const double mean = warp_sum(sum) / (double)n;
    double ss = 0.0;
    for (size_t i = lane; i < n; i += 32) {
        const double r = xs[i * k] - mean;
        ss += r * r;
    }
    const double norm = fmax(warp_sum(ss), 1e-300);
    double tau = 1.0;
    for (size_t j = 1; j < n; j++) {
        double acc = 0.0;
        for (size_t i = lane; i + j < n; i += 32) acc += (xs[i * k] - mean) * (xs[(i + j) * k] - mean);
        const double ac = warp_sum(acc) / norm;
        if (!(ac > 0.05)) break;
        tau += 2.0 * ac;
    }
    if (lane == 0) ess[g] = (double)n / tau;
}

static int psd_args_ok(const char* fn, int kind, int p, int q, const void* priors, size_t ncurves, size_t nsamples,
                       const void* theta, const void* freq, size_t freq_rows, size_t nfreq, const void* pct, size_t npct,
                       const void* out) {
    if (!valid_model(kind, p, q)) { set_error(std::string(fn) + ": invalid (kind,p,q)"); return CARMA_ERR_ARG; }
    if (ncurves && freq_rows != 1 && freq_rows != ncurves) {
        set_error(std::string(fn) + ": freq_rows must be 1 or ncurves");
        return CARMA_ERR_ARG;
    }
    const bool work = ncurves && nsamples && nfreq && npct;
    if (work && (!theta || !freq || !pct || !out)) { set_error(std::string(fn) + ": null argument"); return CARMA_ERR_ARG; }
    if (work && kind == CARMA_KIND_ZCARMA && !priors) {
        set_error(std::string(fn) + ": ZCARMA needs the priors (kappa bounds)");
        return CARMA_ERR_ARG;
    }
    return CARMA_OK;
}

static int nb_of(int kind, int p, int q) { return kind == CARMA_KIND_CARMA ? q : kind == CARMA_KIND_ZCARMA ? p - 1 : 0; }

static bool psd_force_global() {
    const char* env = getenv("CARMA_PSD_GLOBAL_SELECT");   // "1": always the global-memory path (tests, timing)
    return env && env[0] == '1';
}

static cudaError_t launch_band_p(int kind, int p, int q, const carma_prior_t* d_priors, const double* d_theta,
                                 const BandArgs& a, cudaStream_t st) {
    const bool global = psd_force_global();
    switch (p) {
        case 1: return launch_band<1>(kind, q, d_priors, d_theta, a, global, st);
        case 2: return launch_band<2>(kind, q, d_priors, d_theta, a, global, st);
        case 3: return launch_band<3>(kind, q, d_priors, d_theta, a, global, st);
        case 4: return launch_band<4>(kind, q, d_priors, d_theta, a, global, st);
        case 5: return launch_band<5>(kind, q, d_priors, d_theta, a, global, st);
        case 6: return launch_band<6>(kind, q, d_priors, d_theta, a, global, st);
        default: return launch_band<7>(kind, q, d_priors, d_theta, a, global, st);
    }
}

}  // namespace carma

using namespace carma;

extern "C" {

int carma_psd_quantiles_dev(int kind, int p, int q, const carma_prior_t* d_priors, size_t ncurves, size_t nsamples,
                            const double* d_theta, const double* d_freq, size_t freq_rows, size_t nfreq,
                            const double* d_pct, size_t npct, double* d_out, double* d_psd_out, void* stream) {
    int rc = psd_args_ok("carma_psd_quantiles_dev", kind, p, q, d_priors, ncurves, nsamples, d_theta, d_freq, freq_rows,
                         nfreq, d_pct, npct, d_out);
    if (rc) return rc;
    if (!ncurves || !nsamples || !nfreq || !npct) return CARMA_OK;
    BandArgs a{};
    a.nb = nb_of(kind, p, q);
    a.nc = ncurves; a.ns = nsamples; a.nf = nfreq;
    a.freq = d_freq; a.freq_stride = freq_rows > 1 ? nfreq : 0;
    a.pct = d_pct; a.npct = npct; a.out = d_out; a.psd_out = d_psd_out;
    if (!cuda_ok(launch_band_p(kind, p, q, d_priors, d_theta, a, (cudaStream_t)stream), "psd_quantiles launch"))
        return CARMA_ERR_CUDA;
    return CARMA_OK;
}

int carma_psd_quantiles(int kind, int p, int q, const carma_prior_t* priors, size_t ncurves, size_t nsamples,
                        const double* theta, const double* freq, size_t freq_rows, size_t nfreq, const double* pct,
                        size_t npct, double* out, double* psd_out, int device) {
    int rc = psd_args_ok("carma_psd_quantiles", kind, p, q, priors, ncurves, nsamples, theta, freq, freq_rows, nfreq, pct,
                         npct, out);
    if (rc) return rc;
    if (!ncurves || !nsamples || !nfreq || !npct) return CARMA_OK;
    for (size_t j = 0; j < npct; j++)
        if (!(pct[j] >= 0.0 && pct[j] <= 100.0)) { set_error("carma_psd_quantiles: percentiles must lie in [0, 100]"); return CARMA_ERR_ARG; }
    if (!cuda_ok(cudaSetDevice(device), "cudaSetDevice")) return CARMA_ERR_CUDA;
    // Curves go in chunks of B whose device footprint stays within the budget (CARMA_PSD_BUDGET bytes, read at every
    // call so that a test can force several chunks).  An output depends only on its curve: chunking changes no bit.
    const size_t d = (size_t)model_dim(kind, p, q);
    const size_t per_curve = nsamples * (d + psd_row_width<MAX_P>() + nfreq * (psd_out ? 2 : 1)) + npct * nfreq +
                             (freq_rows > 1 ? nfreq : 0) + 1;
    size_t budget = (size_t)4 << 30;
    if (const char* env = getenv("CARMA_PSD_BUDGET")) budget = (size_t)std::strtoull(env, nullptr, 10);
    const size_t B = std::max<size_t>(1, std::min(ncurves, budget / (per_curve * sizeof(double))));
    cudaStream_t st = 0;
    const size_t fr_b = (freq_rows > 1 ? B : 1) * nfreq;
    double *d_th = nullptr, *d_fr = nullptr, *d_pct = nullptr, *d_out = nullptr, *d_psd = nullptr;
    carma_prior_t* d_pr = nullptr;
    bool ok = cuda_ok(cudaMalloc((void**)&d_th, B * nsamples * d * sizeof(double)), "cudaMalloc theta") &&
              cuda_ok(cudaMalloc((void**)&d_fr, fr_b * sizeof(double)), "cudaMalloc freq") &&
              cuda_ok(cudaMalloc((void**)&d_pct, npct * sizeof(double)), "cudaMalloc pct") &&
              cuda_ok(cudaMalloc((void**)&d_out, B * npct * nfreq * sizeof(double)), "cudaMalloc out") &&
              (!psd_out || cuda_ok(cudaMalloc((void**)&d_psd, B * nsamples * nfreq * sizeof(double)), "cudaMalloc psd")) &&
              (!priors || cuda_ok(cudaMalloc((void**)&d_pr, B * sizeof(carma_prior_t)), "cudaMalloc priors")) &&
              cuda_ok(cudaMemcpyAsync(d_pct, pct, npct * sizeof(double), cudaMemcpyHostToDevice, st), "H2D pct");
    if (ok && freq_rows == 1) ok = cuda_ok(cudaMemcpyAsync(d_fr, freq, nfreq * sizeof(double), cudaMemcpyHostToDevice, st), "H2D freq");
    for (size_t c0 = 0; ok && c0 < ncurves; c0 += B) {
        const size_t nb = std::min(B, ncurves - c0);
        ok = cuda_ok(cudaMemcpyAsync(d_th, theta + c0 * nsamples * d, nb * nsamples * d * sizeof(double), cudaMemcpyHostToDevice, st), "H2D theta") &&
             (freq_rows == 1 || cuda_ok(cudaMemcpyAsync(d_fr, freq + c0 * nfreq, nb * nfreq * sizeof(double), cudaMemcpyHostToDevice, st), "H2D freq")) &&
             (!priors || cuda_ok(cudaMemcpyAsync(d_pr, priors + c0, nb * sizeof(carma_prior_t), cudaMemcpyHostToDevice, st), "H2D priors"));
        if (!ok) break;
        rc = carma_psd_quantiles_dev(kind, p, q, d_pr, nb, nsamples, d_th, d_fr, freq_rows == 1 ? 1 : nb, nfreq, d_pct, npct,
                                     d_out, d_psd, st);
        if (rc) break;
        ok = cuda_ok(cudaMemcpyAsync(out + c0 * npct * nfreq, d_out, nb * npct * nfreq * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H out") &&
             (!psd_out || cuda_ok(cudaMemcpyAsync(psd_out + c0 * nsamples * nfreq, d_psd, nb * nsamples * nfreq * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H psd"));
    }
    if (ok && !rc) ok = cuda_ok(cudaStreamSynchronize(st), "psd_quantiles sync");
    cudaFree(d_th); cudaFree(d_fr); cudaFree(d_pct); cudaFree(d_out); cudaFree(d_psd); cudaFree(d_pr);
    if (rc) return rc;
    return ok ? CARMA_OK : CARMA_ERR_CUDA;
}

int carma_effective_samples_dev(size_t nseries, size_t n, size_t k, const double* d_x, double* d_ess, void* stream) {
    if (!nseries || !n || !k) return CARMA_OK;
    if (!d_x || !d_ess) { set_error("carma_effective_samples_dev: null argument"); return CARMA_ERR_ARG; }
    const size_t warps = nseries * k;
    effective_samples_kernel<<<(unsigned)((warps + 7) / 8), 256, 0, (cudaStream_t)stream>>>(nseries, n, k, d_x, d_ess);
    if (!cuda_ok(cudaGetLastError(), "effective_samples_kernel launch")) return CARMA_ERR_CUDA;
    return CARMA_OK;
}

int carma_effective_samples(size_t nseries, size_t n, size_t k, const double* x, double* ess, int device) {
    if (!nseries || !n || !k) return CARMA_OK;
    if (!x || !ess) { set_error("carma_effective_samples: null argument"); return CARMA_ERR_ARG; }
    if (!cuda_ok(cudaSetDevice(device), "cudaSetDevice")) return CARMA_ERR_CUDA;
    double *d_x = nullptr, *d_e = nullptr;
    int rc = CARMA_ERR_CUDA;
    if (cuda_ok(cudaMalloc((void**)&d_x, nseries * n * k * sizeof(double)), "cudaMalloc x") &&
        cuda_ok(cudaMalloc((void**)&d_e, nseries * k * sizeof(double)), "cudaMalloc ess") &&
        cuda_ok(cudaMemcpy(d_x, x, nseries * n * k * sizeof(double), cudaMemcpyHostToDevice), "H2D x")) {
        rc = carma_effective_samples_dev(nseries, n, k, d_x, d_e, nullptr);
        if (rc == CARMA_OK && !cuda_ok(cudaMemcpy(ess, d_e, nseries * k * sizeof(double), cudaMemcpyDeviceToHost), "D2H ess"))
            rc = CARMA_ERR_CUDA;
    }
    cudaFree(d_x);
    cudaFree(d_e);
    return rc;
}

}  // extern "C"
