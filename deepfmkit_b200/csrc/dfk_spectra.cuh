// Post-fit step of the readout (SURVEY 8f-4): block means of a raw-rate series at the fit rate
// (dsp.py:3-56 vectorized_downsample) and the log-frequency spectral density of a fitted series
// (core.py:590-609 / data.py:239-244 -> spectools.lpsd, restated from Troebs & Heinzel 2006 and the LTPDA scheduler;
// see oracle/post_oracle.py for the sources), and the cross-spectral density of two sets of series on the same plan.
#pragma once
#include "dfk_common.cuh"

namespace dfk {

// ---------------------------------------------------------------------------------------------------------------
// Block means.  HBM-bound: 8 B read per sample, 8 B written per R samples.  A block of R samples is summed by a
// warp (R < kDsCtaMin) or by a whole CTA (R >= kDsCtaMin) with 128-bit loads, four in flight per lane.
// ---------------------------------------------------------------------------------------------------------------
constexpr int kDsThreads = 256;
constexpr int kDsCtaMin = 4096;

DFK_D double ds_partial(const double* __restrict__ p, long long R, int lane, int width) {
    // sum of p[0..R) over `width` cooperating lanes; p 16-byte aligned is the fast path
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
    long long i = 0;
    if ((reinterpret_cast<uintptr_t>(p) & 15u) == 0) {
        const double2* q = reinterpret_cast<const double2*>(p);
        const long long n2 = R >> 1;
        long long k = lane;
        for (; k + 3ll * width < n2; k += 4ll * width) {
            const double2 v0 = __ldcs(q + k), v1 = __ldcs(q + k + width), v2 = __ldcs(q + k + 2 * width),
                          v3 = __ldcs(q + k + 3 * width);
            a0 += v0.x + v0.y;
            a1 += v1.x + v1.y;
            a2 += v2.x + v2.y;
            a3 += v3.x + v3.y;
        }
        for (; k < n2; k += width) {
            const double2 v = __ldcs(q + k);
            a0 += v.x + v.y;
        }
        i = n2 << 1;
        if (lane == 0 && i < R) a1 += p[i];
    } else {
        for (long long k = lane; k < R; k += width) a0 += p[k];
    }
    return (a0 + a1) + (a2 + a3);
}

__global__ void __launch_bounds__(kDsThreads) downsample_kernel(const double* __restrict__ x, long long nblk, long long R,
                                                               double* __restrict__ out) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const double inv = 1.0 / static_cast<double>(R);
    if (R >= kDsCtaMin) {
        __shared__ double part[kDsThreads / 32];
        for (long long b = blockIdx.x; b < nblk; b += gridDim.x) {
            double s = warp_sum(ds_partial(x + b * R, R, threadIdx.x, kDsThreads));
            if (lane == 0) part[warp] = s;
            __syncthreads();
            if (threadIdx.x == 0) {
                double t = 0.0;
#pragma unroll
                for (int w = 0; w < kDsThreads / 32; ++w) t += part[w];
                out[b] = t * inv;
            }
            __syncthreads();
        }
    } else {
        const long long nw = static_cast<long long>(gridDim.x) * (kDsThreads / 32);
        for (long long b = blockIdx.x * (kDsThreads / 32ll) + warp; b < nblk; b += nw) {
            const double s = warp_sum(ds_partial(x + b * R, R, lane, 32));
            if (lane == 0) out[b] = s * inv;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// LPSD.  For frequency j the record is cut into K_j overlapping segments of L_j samples; each is detrended
// (polynomial of degree `order`), windowed and projected on exp(2 pi i m_j n / L_j) with a fractional bin m_j; the
// spectrum is the mean of |.|^2 over the segments.  Window and twiddle depend on (j, n) only, so a group of up to
// kLpsdGroup consecutive segments shares every evaluation of them: a warp (L < kLpsdCtaMin) or a CTA takes a group,
// lanes stride n.  Group sums land in a scratch table in a fixed order, so results do not depend on scheduling.
// ---------------------------------------------------------------------------------------------------------------
constexpr int kLpsdThreads = 256;
constexpr int kLpsdGroup = 8;
constexpr int kLpsdCtaMin = 2048;

struct LpsdFreq {        // one row of the plan, device copy
    long long L, K;      // segment length, number of segments
    double p;            // 2 pi m / L  (angle per sample)
    double shift;        // samples between segment starts
    long long tile0;     // first tile of this frequency
    long long group0;    // first slot of this frequency in the group-sum table
};

struct LpsdParams {
    const double* x;        // sample i of series c at x[c * ld_c + i * stride]
    long long N, stride, ld_c;
    const LpsdFreq* plan;
    int nf;
    long long ntiles;       // per series
    long long ngroups;      // per series
    int order;              // -1 none, 0 mean, 1 linear, 2 quadratic
    int window;             // 0 Kaiser, 1 Hann
    double beta;            // Kaiser: pi * alpha
    double inv_i0_beta;
    double* group_sum;      // [C][ngroups]
};

// 1 / k^2, k = 1..64: the series below spends its time in this factor (a division per term was ~90 % of the LPSD
// kernel: the window is evaluated once per sample and group of segments, 40-50 terms each at 200 dB side lobes)
__device__ __constant__ double kInvSquare[64] = {1.0 / 1.0, 1.0 / 4.0, 1.0 / 9.0, 1.0 / 16.0, 1.0 / 25.0, 1.0 / 36.0, 1.0 / 49.0, 1.0 / 64.0, 1.0 / 81.0, 1.0 / 100.0, 1.0 / 121.0, 1.0 / 144.0, 1.0 / 169.0, 1.0 / 196.0, 1.0 / 225.0, 1.0 / 256.0, 1.0 / 289.0, 1.0 / 324.0, 1.0 / 361.0, 1.0 / 400.0, 1.0 / 441.0, 1.0 / 484.0, 1.0 / 529.0, 1.0 / 576.0, 1.0 / 625.0, 1.0 / 676.0, 1.0 / 729.0, 1.0 / 784.0, 1.0 / 841.0, 1.0 / 900.0, 1.0 / 961.0, 1.0 / 1024.0, 1.0 / 1089.0, 1.0 / 1156.0, 1.0 / 1225.0, 1.0 / 1296.0, 1.0 / 1369.0, 1.0 / 1444.0, 1.0 / 1521.0, 1.0 / 1600.0, 1.0 / 1681.0, 1.0 / 1764.0, 1.0 / 1849.0, 1.0 / 1936.0, 1.0 / 2025.0, 1.0 / 2116.0, 1.0 / 2209.0, 1.0 / 2304.0, 1.0 / 2401.0, 1.0 / 2500.0, 1.0 / 2601.0, 1.0 / 2704.0, 1.0 / 2809.0, 1.0 / 2916.0, 1.0 / 3025.0, 1.0 / 3136.0, 1.0 / 3249.0, 1.0 / 3364.0, 1.0 / 3481.0, 1.0 / 3600.0, 1.0 / 3721.0, 1.0 / 3844.0, 1.0 / 3969.0, 1.0 / 4096.0};

DFK_D double bessel_i0(double x) {
    // power series sum (x^2/4)^k / (k!)^2: all terms positive, converges in < 60 terms for x <= 40
    const double q = 0.25 * x * x;
    double term = 1.0, sum = 1.0;
    for (int k = 1; k < 200; ++k) {
        term *= k <= 64 ? q * kInvSquare[k - 1] : q / (static_cast<double>(k) * static_cast<double>(k));
        sum += term;
        if (term < 1e-17 * sum) break;
    }
    return sum;
}

DFK_D double lpsd_window(const LpsdParams& P, long long n, double half_len) {
    if (P.window == 0) {
        const double z = (static_cast<double>(n) - half_len) / half_len;  // np.kaiser(L + 1, beta)[n]
        const double a = fmax(1.0 - z * z, 0.0);
        return bessel_i0(P.beta * sqrt(a)) * P.inv_i0_beta;
    }
    return 0.5 * (1.0 - cospi(static_cast<double>(n) / half_len));
}

DFK_D long long lpsd_start(double shift, long long k) { return static_cast<long long>(floor(static_cast<double>(k) * shift + 0.5)); }

// One group: segments k0 .. k0+ns-1 of frequency row F, by `width` lanes (lane = this thread's index among them).
// On return re[s], im[s] (s < ns) hold, on every lane, the segment's projection A_s = sum_n w_n v_n e^{+i p n}
// (v detrended), its lane partials reduced by the caller-supplied functor `reduce` (warp or CTA wide).
template <class Reduce>
DFK_D void lpsd_group_dft(const LpsdParams& P, const LpsdFreq& F, const double* __restrict__ xc, long long k0, int ns,
                          int lane, int width, Reduce reduce, double (&re)[kLpsdGroup], double (&im)[kLpsdGroup]) {
    const long long L = F.L;
    long long start[kLpsdGroup];
#pragma unroll
    for (int s = 0; s < kLpsdGroup; ++s) start[s] = lpsd_start(F.shift, k0 + (s < ns ? s : 0));
    // detrend coefficients on the orthogonal basis 1, u, u^2 - (L^2 - 1)/12 with u = n - (L - 1)/2
    double c0[kLpsdGroup], c1[kLpsdGroup], c2[kLpsdGroup];
    const double mid = 0.5 * static_cast<double>(L - 1);
    const double Ld = static_cast<double>(L);
    const double q2 = (Ld * Ld - 1.0) / 12.0;
#pragma unroll
    for (int s = 0; s < kLpsdGroup; ++s) c0[s] = c1[s] = c2[s] = 0.0;
    if (P.order >= 0) {
        for (long long n = lane; n < L; n += width) {
            const double u = static_cast<double>(n) - mid;
            const double p2 = u * u - q2;
#pragma unroll
            for (int s = 0; s < kLpsdGroup; ++s) {
                if (s < ns) {
                    const double v = xc[(start[s] + n) * P.stride];
                    c0[s] += v;
                    if (P.order >= 1) c1[s] = fma(v, u, c1[s]);
                    if (P.order >= 2) c2[s] = fma(v, p2, c2[s]);
                }
            }
        }
        const double n0 = Ld, n1 = Ld * q2, n2 = Ld * (Ld * Ld - 1.0) * (Ld * Ld - 4.0) / 180.0;
#pragma unroll
        for (int s = 0; s < kLpsdGroup; ++s) {
            if (s < ns) {
                c0[s] = reduce(c0[s]) / n0;
                c1[s] = (P.order >= 1 && L > 1) ? reduce(c1[s]) / n1 : 0.0;
                c2[s] = (P.order >= 2 && L > 2) ? reduce(c2[s]) / n2 : 0.0;
            }
        }
    }
#pragma unroll
    for (int s = 0; s < kLpsdGroup; ++s) re[s] = im[s] = 0.0;
    const double half_len = 0.5 * Ld;
    for (long long n = lane; n < L; n += width) {
        const double w = lpsd_window(P, n, half_len);
        double sn, cs;
        sincos(F.p * static_cast<double>(n), &sn, &cs);
        const double wc = w * cs, ws = w * sn;
        const double u = static_cast<double>(n) - mid;
        const double p2 = u * u - q2;
#pragma unroll
        for (int s = 0; s < kLpsdGroup; ++s) {
            if (s < ns) {
                double v = xc[(start[s] + n) * P.stride];
                v -= c0[s] + c1[s] * u + c2[s] * p2;
                re[s] = fma(v, wc, re[s]);
                im[s] = fma(v, ws, im[s]);
            }
        }
    }
    // the reduced values, in the order the lanes reach them: re[0], im[0], re[1], ...
#pragma unroll
    for (int s = 0; s < kLpsdGroup; ++s) {
        if (s < ns) {
            const double r = reduce(re[s]), i = reduce(im[s]);
            re[s] = r;
            im[s] = i;
        }
    }
}

// The group(s) of segments that tile `tile` of one series covers (a CTA per group when L >= kLpsdCtaMin, else a warp
// per group): emit(F, g, ns, re, im, lead) receives, on every lane of the group, frequency row F, the group's index g
// within the row, its segment count and the reduced projections; `lead` is true on one lane per group.
template <class Emit>
DFK_D void lpsd_tile(const LpsdParams& P, const double* __restrict__ xc, long long tile, double* red, Emit emit) {
    // frequency row of this tile: last row with tile0 <= tile
    int lo = 0, hi = P.nf - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (P.plan[mid].tile0 <= tile) lo = mid; else hi = mid - 1;
    }
    const LpsdFreq F = P.plan[lo];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long t = tile - F.tile0;
    double re[kLpsdGroup], im[kLpsdGroup];
    if (F.L >= kLpsdCtaMin) {
        // one group per tile, all lanes of the CTA
        const long long k0 = t * kLpsdGroup;
        const int ns = static_cast<int>(min(static_cast<long long>(kLpsdGroup), F.K - k0));
        auto reduce = [&](double v) {
            v = warp_sum(v);
            __syncthreads();
            if (lane == 0) red[warp] = v;
            __syncthreads();
            double s = 0.0;
#pragma unroll
            for (int w = 0; w < kLpsdThreads / 32; ++w) s += red[w];
            return s;
        };
        lpsd_group_dft(P, F, xc, k0, ns, threadIdx.x, kLpsdThreads, reduce, re, im);
        emit(F, t, ns, re, im, threadIdx.x == 0);
    } else {
        // a group per warp
        const long long g = t * (kLpsdThreads / 32) + warp;
        const long long k0 = g * kLpsdGroup;
        if (k0 >= F.K) return;
        const int ns = static_cast<int>(min(static_cast<long long>(kLpsdGroup), F.K - k0));
        auto reduce = [&](double v) { return warp_sum(v); };
        lpsd_group_dft(P, F, xc, k0, ns, lane, 32, reduce, re, im);
        emit(F, g, ns, re, im, lane == 0);
    }
}

__global__ void __launch_bounds__(kLpsdThreads) lpsd_segment_kernel(const LpsdParams P) {
    __shared__ double red[kLpsdThreads / 32];
    const long long c = blockIdx.y;
    double* out = P.group_sum + c * P.ngroups;
    lpsd_tile(P, P.x + c * P.ld_c, blockIdx.x, red,
              [&](const LpsdFreq& F, long long g, int ns, const double (&re)[kLpsdGroup], const double (&im)[kLpsdGroup],
                  bool lead) {
                  double total = 0.0;
#pragma unroll
                  for (int s = 0; s < kLpsdGroup; ++s)
                      if (s < ns) total += re[s] * re[s] + im[s] * im[s];
                  if (lead) out[F.group0 + g] = total;
              });
}

// Window sums S1 = sum w_n and S2 = sum w_n^2 of row F by a CTA of kThreads lanes (lane partials in n order, warp
// sums, then a fixed pairwise tree over the warps); red1, red2 hold kThreads / 32 doubles each.
template <int kThreads>
DFK_D void lpsd_window_sums(const LpsdParams& P, const LpsdFreq& F, double* red1, double* red2, double& s1, double& s2) {
    static_assert(kThreads == 128 || kThreads == 256, "fixed reduction tree for 4 or 8 warps");
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    s1 = s2 = 0.0;
    const double half_len = 0.5 * static_cast<double>(F.L);
    for (long long n = threadIdx.x; n < F.L; n += kThreads) {
        const double w = lpsd_window(P, n, half_len);
        s1 += w;
        s2 = fma(w, w, s2);
    }
    s1 = warp_sum(s1);
    s2 = warp_sum(s2);
    if (lane == 0) {
        red1[warp] = s1;
        red2[warp] = s2;
    }
    __syncthreads();
    s1 = (red1[0] + red1[1]) + (red1[2] + red1[3]);
    s2 = (red2[0] + red2[1]) + (red2[2] + red2[3]);
    if constexpr (kThreads == 256) {
        s1 += (red1[4] + red1[5]) + (red1[6] + red1[7]);
        s2 += (red2[4] + red2[5]) + (red2[6] + red2[7]);
    }
}

// Per (series, frequency): mean over the groups in order, window sums S1, S2, scaling to PS / PSD / ENBW.
__global__ void __launch_bounds__(128) lpsd_finish_kernel(const LpsdParams P, long long C, double fs, double* __restrict__ ps,
                                                         double* __restrict__ psd, double* __restrict__ enbw) {
    __shared__ double r1[4], r2[4];
    const int j = blockIdx.x;
    const LpsdFreq F = P.plan[j];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double s1, s2;
    lpsd_window_sums<128>(P, F, r1, r2, s1, s2);
    const long long ng = (F.K + kLpsdGroup - 1) / kLpsdGroup;
    for (long long c = 0; c < C; ++c) {
        const double* g = P.group_sum + c * P.ngroups + F.group0;
        double total = 0.0;
        for (long long i = threadIdx.x; i < ng; i += 128) total += g[i];
        total = warp_sum(total);
        __syncthreads();
        if (lane == 0) r1[warp] = total;
        __syncthreads();
        if (threadIdx.x == 0) {
            const double avg = ((r1[0] + r1[1]) + (r1[2] + r1[3])) / static_cast<double>(F.K);
            ps[c * P.nf + j] = 2.0 * avg / (s1 * s1);
            psd[c * P.nf + j] = 2.0 * avg / (fs * s2);
        }
    }
    if (threadIdx.x == 0) enbw[j] = fs * s2 / (s1 * s1);
}

// ---------------------------------------------------------------------------------------------------------------
// Cross-spectral density on the LPSD plan (the LTPDA log-frequency CSD).  For frequency row j, segment s of series u
// has the projection A_{u,s} = sum_n w_n v_n e^{+i p_j n} that lpsd_group_dft forms (v detrended): the complex
// conjugate of the usual DFT X.  Then
//   Sxy[a,b,j] = 2 / (fs S2_j) * (1 / K_j) * sum_s A_{x_a,s} conj(A_{y_b,s})
// is the one-sided CSD in the E[conj(X) Y] convention, and Sxx, Syy are the same sum on one series: lpsd's psd.
// Stage 1 stores every segment's A in a table [series][group0 * kLpsdGroup + k] (at most kLpsdGroup - 1 unused slots
// per row); the finish kernel takes a frequency row per CTA and sums each auto and cross term over the K_j segments in
// a fixed order (lane partials in segment order, warp sums, a fixed tree over the warps), so the result does not
// depend on scheduling.  Each product is rounded on its own (no contraction), so a series against itself gives a
// real Sxy bit-equal to its Sxx.
// ---------------------------------------------------------------------------------------------------------------
constexpr int kLcsdFinishThreads = 256;

struct LcsdParams {
    LpsdParams P;        // the plan and the series x (P.x, P.ld_c); P.group_sum is not used
    const double* y;     // sample i of y series b at y[b * ld_y + i * P.stride]
    long long ld_y;
    long long cx, cy;
    double2* seg;        // [cx + cy][nslots]: x series first, then y
    long long nslots;    // P.ngroups * kLpsdGroup
};

__global__ void __launch_bounds__(kLpsdThreads) lcsd_segment_kernel(const LcsdParams Q) {
    __shared__ double red[kLpsdThreads / 32];
    const long long u = blockIdx.y;
    const double* xc = u < Q.cx ? Q.P.x + u * Q.P.ld_c : Q.y + (u - Q.cx) * Q.ld_y;
    double2* out = Q.seg + u * Q.nslots;
    lpsd_tile(Q.P, xc, blockIdx.x, red,
              [&](const LpsdFreq& F, long long g, int ns, const double (&re)[kLpsdGroup], const double (&im)[kLpsdGroup],
                  bool lead) {
                  if (!lead) return;
                  double2* o = out + (F.group0 + g) * kLpsdGroup;
#pragma unroll
                  for (int s = 0; s < kLpsdGroup; ++s)
                      if (s < ns) o[s] = make_double2(re[s], im[s]);
              });
}

// Per frequency row: S1, S2, then every auto term (series 0 .. cx+cy-1: psd[u][j]) and every pair (a, b)
// (sxy[(a * cy + b) * nf + j] as re, im), then ENBW.
__global__ void __launch_bounds__(kLcsdFinishThreads) lcsd_finish_kernel(const LcsdParams Q, double fs,
                                                                        double* __restrict__ psd,
                                                                        double* __restrict__ sxy,
                                                                        double* __restrict__ enbw) {
    constexpr int kWarps = kLcsdFinishThreads / 32;
    __shared__ double r1[kWarps], r2[kWarps];
    const int j = blockIdx.x;
    const int nf = Q.P.nf;
    const LpsdFreq F = Q.P.plan[j];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double s1, s2;
    lpsd_window_sums<kLcsdFinishThreads>(Q.P, F, r1, r2, s1, s2);
    const long long nauto = Q.cx + Q.cy, nterms = nauto + Q.cx * Q.cy;
    const double2* row = Q.seg + F.group0 * kLpsdGroup;
    for (long long term = 0; term < nterms; ++term) {
        const bool cross = term >= nauto;
        const long long pair = term - nauto;
        const long long a = cross ? pair / Q.cy : term, b = cross ? Q.cx + pair % Q.cy : term;
        const double2* A = row + a * Q.nslots;
        const double2* B = row + b * Q.nslots;
        double re = 0.0, im = 0.0;
        for (long long s = threadIdx.x; s < F.K; s += kLcsdFinishThreads) {
            const double2 p = A[s], q = B[s];
            // A conj(B) = (p.x q.x + p.y q.y) + i (p.y q.x - p.x q.y)
            re = __dadd_rn(re, __dadd_rn(__dmul_rn(p.x, q.x), __dmul_rn(p.y, q.y)));
            im = __dadd_rn(im, __dsub_rn(__dmul_rn(p.y, q.x), __dmul_rn(p.x, q.y)));
        }
        re = warp_sum(re);
        im = warp_sum(im);
        __syncthreads();  // the previous term's (or the window sums') reads of r1, r2 are done
        if (lane == 0) {
            r1[warp] = re;
            r2[warp] = im;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            re = ((r1[0] + r1[1]) + (r1[2] + r1[3])) + ((r1[4] + r1[5]) + (r1[6] + r1[7]));
            im = ((r2[0] + r2[1]) + (r2[2] + r2[3])) + ((r2[4] + r2[5]) + (r2[6] + r2[7]));
            const double K = static_cast<double>(F.K);
            if (cross) {
                sxy[2 * (pair * nf + j)] = 2.0 * (re / K) / (fs * s2);
                sxy[2 * (pair * nf + j) + 1] = 2.0 * (im / K) / (fs * s2);
            } else {
                psd[term * nf + j] = 2.0 * (re / K) / (fs * s2);
            }
        }
    }
    if (threadIdx.x == 0) enbw[j] = fs * s2 / (s1 * s1);
}

}  // namespace dfk
