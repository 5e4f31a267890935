// hesscheck.cu -- TEST INFRASTRUCTURE (never part of the product library).
// The HOST side of carma_multi_hessian's stencil and assembly (hess_point_dirs / hess_scale / hess_assemble,
// hessian.cuh), which multi_hessian_eval_kernel and multi_hessian_assemble_kernel run on the device, behind a tiny
// C ABI: tests/test_survey_hessian_host.py checks them against numpy without a GPU.
// Build:  nvcc -O2 -std=c++17 -Xcompiler -fPIC -shared -o libhesscheck.so hesscheck.cu   (host code only)
#include "../../carma_pack_b200/csrc/hessian.cuh"

using namespace carma;

// The d^2 + d + 1 stencil rows of theta (d entries) with relative step rel_step, row-major into rows.
extern "C" int hess_rows(int d, const double* theta, double rel_step, double* rows) {
    if (d < 1 || d > MAX_D) return 1;
    for (int k = 0; k < hess_points(d); k++) {
        int a, b;
        double sa, sb;
        hess_point_dirs(k, d, &a, &sa, &b, &sb);
        for (int j = 0; j < d; j++) {
            const double h = rel_step * hess_scale(theta[0], theta[1], j);
            const double s = (j == a) ? sa : (j == b) ? sb : 0.0;
            rows[k * d + j] = (s > 0.0) ? theta[j] + h : (s < 0.0) ? theta[j] - h : theta[j];
        }
    }
    return 0;
}

// One curve's assembly: f (d^2 + d + 1 stencil values), h (d steps) -> g, H, cov; returns the CARMA_HESS_* status.
extern "C" int hess_assemble_host(int d, const double* f, const double* h, double* g, double* H, double* cov) {
    if (d < 1 || d > MAX_D) return -1;
    return hess_assemble(d, f, h, g, H, cov);
}
