// laplacecheck.cu -- TEST INFRASTRUCTURE (never part of the product library).
// The HOST side of carma_multi_laplace's per-curve arithmetic (laplace.cuh): the Cholesky factor, and the weight
// summaries multi_laplace_summary_kernel computes (weight ESS, Pareto k-hat, systematic resampling), composed here in
// plain sequential loops behind a tiny C ABI: tests/test_survey_laplace_host.py checks them against numpy without a GPU.
// Build:  nvcc -O2 -std=c++17 -Xcompiler -fPIC -shared -o liblaplacecheck.so laplacecheck.cu   (host code only)
#include <algorithm>
#include <vector>

#include "../../carma_pack_b200/csrc/laplace.cuh"

using namespace carma;

extern "C" int lap_chol_host(int d, const double* centre, const double* cov, double* L, double* logdet) {
    if (d < 1 || d > MAX_D) return -1;
    return lap_cholesky(d, centre, cov, L, logdet);
}

// weight ESS, k-hat and the resample of S log weights lw (-inf allowed, at least one finite), u the resampling uniform
extern "C" int lap_summary_host(const double* lw, size_t S, double u, double* ess, double* khat, int* resample) {
    double mx = -INFINITY;
    for (size_t i = 0; i < S; i++) mx = std::max(mx, lw[i]);
    if (mx == -INFINITY) return CARMA_LAPLACE_NO_WEIGHT;
    std::vector<double> e(S), C(S);
    double s1 = 0.0, s2 = 0.0;
    for (size_t i = 0; i < S; i++) {
        e[i] = exp(lw[i] - mx);
        s1 += e[i];
        s2 += e[i] * e[i];
    }
    *ess = s1 * s1 / s2;
    *khat = INFINITY;
    if (S >= 2) {
        std::vector<double> srt(lw, lw + S);
        std::sort(srt.begin(), srt.end());
        const double cut = std::max(srt[S - psis_tail_len(S) - 1] - mx, LAP_LOG_DBL_MIN), ecut = exp(cut);
        std::vector<double> x;
        for (size_t i = 0; i < S; i++)
            if (lw[i] - mx > cut) x.push_back(exp(lw[i] - mx) - ecut);
        const int n = (int)x.size();
        if (n > 4) {
            std::sort(x.begin(), x.end());
            const int m = gpd_m(n);
            std::vector<double> b(m), Lp(m), w(m);
            for (int i = 0; i < m; i++) {
                b[i] = gpd_b(i + 1, m, x.data(), n);
                double k = 0.0;
                for (int t = 0; t < n; t++) k += log1p(-b[i] * x[t]);
                Lp[i] = gpd_profile(n, b[i], k / n);
            }
            for (int i = 0; i < m; i++) w[i] = gpd_weight(i, m, Lp.data());
            const double bbar = gpd_bbar(m, b.data(), w.data());
            double k = 0.0;
            for (int t = 0; t < n; t++) k += log1p(-bbar * x[t]);
            *khat = gpd_khat(n, k / n);
        }
    }
    double run = 0.0;
    for (size_t i = 0; i < S; i++) C[i] = run += e[i];
    for (size_t i = 0; i < S; i++) resample[i] = (int)resample_find(C.data(), S, resample_target(i, u, S, C[S - 1]));
    return CARMA_LAPLACE_OK;
}
