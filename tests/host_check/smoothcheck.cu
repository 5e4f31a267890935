// smoothcheck.cu -- TEST INFRASTRUCTURE (never part of the product library).
// The HOST side of the smoother's per-curve passes (smooth_forward / smooth_backward, kalman_real.cuh), which
// multi_smooth_kernel runs one thread per curve, behind a tiny C ABI: tests/test_survey_smooth_host.py checks the
// recursion against the dense Gaussian-process conditional without a GPU.
// Build:  nvcc -O2 -std=c++17 -Xcompiler -fPIC -shared -o libsmoothcheck.so smoothcheck.cu   (host code only)
#include <algorithm>
#include <cmath>
#include <cstddef>
#include <numeric>
#include <vector>

#include "../../carma_pack_b200/csrc/kalman_real.cuh"

using namespace carma;

template <int P>
static void one(int kind, int q, unsigned flags, const carma_prior_t& pr, const double* th, const double* dt,
                const double* y, const double* e2, int ny, double dt_max, const double* qtq, const long long* perm,
                long long nq, double* out, double* qm, double* qv) {
    RealParams<P> prm;
    if (transform_theta<P>(kind, q, flags, pr, th, dt_max, prm) != TT_OK) {
        for (int i = 0; i < 4 * ny; i++) out[i] = NAN;
        out[4 * ny] = -INFINITY;
        return;
    }
    MathTab tb;
    tb.load();
    std::vector<double> rp((size_t)(P + 2) * ny), rq((size_t)(P + 3) * std::max(nq, 1ll));
    KalmanReal<P> kf;
    LogLikAcc acc;
    kf.reset(prm, e2[0]);
    acc.init();
    smooth_forward<P, false>(kf, acc, prm, tb, dt, y, e2, ny, rp.data(), (size_t)ny, 0, nq, qtq, rq.data(), (size_t)nq,
                             perm, qm, qv);
    out[4 * ny] = acc.value() + prm.logprior;
    smooth_backward<P>(prm, tb, dt, y, ny, rp.data(), (size_t)ny, 0, nq, rq.data(), (size_t)nq, perm, out, out + ny,
                       out + 2 * ny, out + 3 * ny, qm, qv);
}

// One curve: t (strictly increasing), y, yerr; queries tq (absolute, any order).  out (4 ny + 1): mean | var | loo_mean |
// loo_var | loglik; qm / qv in the order of tq.  All means without mu.
extern "C" int smoothcheck(int kind, int p, int q, unsigned flags, const carma_prior_t* prior, const double* t,
                           const double* y, const double* yerr, size_t ny, const double* theta, const double* tq, size_t nq,
                           double* out, double* qm, double* qv) {
    if (p < 1 || p > MAX_P || ny < 2) return 1;
    std::vector<double> dt(ny, 0.0), e2(ny);
    double dt_max = 0.0;
    for (size_t i = 0; i < ny; i++) {
        if (i + 1 < ny) dt[i] = t[i + 1] - t[i];
        e2[i] = yerr[i] * yerr[i];
        dt_max = std::max(dt_max, dt[i]);
    }
    std::vector<long long> perm(nq);
    std::iota(perm.begin(), perm.end(), 0ll);
    std::stable_sort(perm.begin(), perm.end(), [&](long long a, long long b) { return tq[a] < tq[b]; });
    std::vector<double> qtq(nq);
    for (size_t k = 0; k < nq; k++) {
        qtq[k] = tq[perm[k]] - t[0];
        dt_max = std::max(dt_max, std::max(qtq[k] - (t[ny - 1] - t[0]), -qtq[k]));
    }
    double th[MAX_D] = {0};
    for (int j = 0; j < model_dim(kind, p, q); j++) th[j] = theta[j];
#define ONE(PP) one<PP>(kind, q, flags, *prior, th, dt.data(), y, e2.data(), (int)ny, dt_max, qtq.data(), perm.data(), \
                        (long long)nq, out, qm, qv)
    switch (p) {
        case 1: ONE(1); break;
        case 2: ONE(2); break;
        case 3: ONE(3); break;
        case 4: ONE(4); break;
        case 5: ONE(5); break;
        case 6: ONE(6); break;
        default: ONE(7); break;
    }
#undef ONE
    return 0;
}
