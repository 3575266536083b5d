// Host build of the stability core (dfk_stability.cuh: the double-double running sums, the rounded differences and
// the finish), for the CPU-side tests.  The running sums are sequential double-double sums (the device's tiled scan
// adds in another order, which changes nothing where the sums are exact); the squared terms are accumulated in the
// device's order: per slice of kStabSlice terms, thread t's terms t + 256 r in order, a fixed tree over the threads,
// then the slices in order.
#include <algorithm>
#include <cstdint>
#include <vector>

#include "../../deepfmkit_b200/csrc/dfk_stability.cuh"

using namespace dfk;

namespace {

// out[0] = 0, out[k] = sum_{i<k} in[i], k <= L
std::vector<DDval> running_sum(const std::vector<DDval>& in) {
    std::vector<DDval> out(in.size() + 1);
    out[0] = {0.0, 0.0};
    for (size_t i = 0; i < in.size(); ++i) out[i + 1] = i ? dd_add(out[i], in[i]) : in[i];
    return out;
}

}  // namespace

extern "C" {

// One series of N samples (data_type 0 phase, 1 freq) at the n_m averaging factors m.  dev[4][n_m], n[4][n_m] in
// the order oadev, mdev, tdev, ohdev (all four are computed whatever is requested).
void sh_stability(const double* v, int64_t N, int data_type, const int64_t* m_list, int n_m, double fs, double* dev,
                  int64_t* n) {
    std::vector<DDval> in(N);
    for (int64_t i = 0; i < N; ++i) in[i] = {v[i], 0.0};
    std::vector<DDval> X = data_type == 1 ? running_sum(in) : in;
    const long long Nx = static_cast<long long>(X.size());
    const std::vector<DDval> S = running_sum(X);
    for (int t = 0; t < n_m; ++t) {
        const long long m = m_list[t];
        const long long na = stab_n_oadev(Nx, m), nm = stab_n_mdev(Nx, m), nh = stab_n_ohdev(Nx, m);
        const long long nmax = std::max(na, std::max(nm, nh));
        double sums[kStabSums] = {0.0, 0.0, 0.0};
        for (long long first = 0; first < nmax; first += kStabSlice) {
            double acc[kStabSums][kStabTermThreads] = {};
            for (int th = 0; th < kStabTermThreads; ++th) {
                for (int r = 0; r < kStabTermsPerThread; ++r) {
                    const long long j = first + static_cast<long long>(r) * kStabTermThreads + th;
                    if (j < na) {
                        const double d = stab_second_diff(X[j], X[j + m], X[j + 2 * m]);
                        acc[0][th] = fma(d, d, acc[0][th]);
                    }
                    if (j < nm) {
                        const double d = stab_third_diff(S[j], S[j + m], S[j + 2 * m], S[j + 3 * m]);
                        acc[1][th] = fma(d, d, acc[1][th]);
                    }
                    if (j < nh) {
                        const double d = stab_third_diff(X[j], X[j + m], X[j + 2 * m], X[j + 3 * m]);
                        acc[2][th] = fma(d, d, acc[2][th]);
                    }
                }
            }
            for (int w = kStabTermThreads / 2; w > 0; w >>= 1)
                for (int th = 0; th < w; ++th)
                    for (int k = 0; k < kStabSums; ++k) acc[k][th] = dd_plus(acc[k][th], acc[k][th + w]);
            for (int k = 0; k < kStabSums; ++k) sums[k] = dd_plus(sums[k], acc[k][0]);
        }
        double d4[4];
        stab_finish_one(sums, m, Nx, fs, data_type == 1 ? 1.0 : fs, d4);
        const long long ns[4] = {na, nm, nm, nh};
        for (int k = 0; k < 4; ++k) {
            dev[k * n_m + t] = d4[k];
            n[k * n_m + t] = ns[k] > 0 ? ns[k] : 0;
        }
    }
}

}  // extern "C"
