// Host build of fit_covariance (dfk_lm_core.cuh), for the CPU-side uncertainty tests.
#include <vector>

#include "../../deepfmkit_b200/csrc/dfk_lm_core.cuh"

extern "C" {

// cov[nfit][8] of rows[nfit][row_stride] on qi[nfit][2N]
void hh_fit_covariance(int N, long long nfit, const double* qi, const double* rows, int row_stride, double* cov) {
    std::vector<double> bes(N + 2);
    for (long long f = 0; f < nfit; ++f)
        dfk::fit_covariance(N, qi + f * 2 * N, 1, bes.data(), 1, rows + f * row_stride, cov + f * dfk::kCovStride);
}

}  // extern "C"
