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

// ---------------------------------------------------------------------------------------------------------------
// Conditioned spectra on the LPSD plan (multiple-input / single-output analysis, Bendat & Piersol, Random Data, ch. 7).
// Witnesses x_1..x_Cx, targets y_1..y_Cy; for frequency row j with c_j = 2 / (fs S2_j K_j) and the segment table of
// lcsd_segment_kernel (x series first, then y):
//   Sxx[a,b,j] = c_j sum_s A_{x_a,s} conj(A_{x_b,s})   the Cx x Cx Hermitian witness matrix (diagonal: lpsd's psd)
//   Sxy[a,t,j] = c_j sum_s A_{x_a,s} conj(A_{y_t,s})   lcsd's convention, E[conj(X) Y]
//   Syy[t,j]   = lpsd's psd of target t
//   H[:,t,j]   = Sxx^-1 Sxy[:,t]                      joint (MISO) transfer functions; for Cx = 1, lcsd's tf
//   Sres[t,j]  = Syy - Sxy[:,t]^H Sxx^-1 Sxy[:,t]     conditioned PSD: y_t after the best linear subtraction of all x
//   mcoh[t,j]  = 1 - Sres / Syy                       multiple coherence (NaN where Syy = 0)
// H, Sres and mcoh are NaN on a row where K_j < Cx (the estimated Sxx has rank <= K_j) or where the Cholesky
// factorisation of Sxx meets a pivot that is not above kCondPivotTol times its diagonal entry (a witness that the
// earlier ones explain to within that fraction: a duplicated or linearly dependent witness).
//
// lcsd_gram_kernel forms the raw sums (before c_j) as a complex product of the segment table per row: output pairs
// (witness a, series b) in tiles of kGramRows x kGramCols, over the Sxx upper triangle and all of Sxy, plus tiles of
// kGramCols target diagonals (Syy); the Cy x Cy target block is never formed.  A CTA stages kGramChunk segments of its
// rows and columns in shared memory; warp w sums the segments w, w + 8, ... of each chunk in a register tile of 2 x 4
// complex accumulators, and the eight warp partials of every output are combined in a fixed tree, so each output has a
// fixed order of summation.  The products may be contracted (FMA).
// lcsd_cond_kernel then takes a frequency row per CTA: it scales the sums, completes Sxx by conjugation, factors it
// (complex Cholesky in shared memory) and solves for every target, a warp per target.
// ---------------------------------------------------------------------------------------------------------------
constexpr int kGramThreads = 256;
constexpr int kGramRows = 8;        // witnesses per tile
constexpr int kGramCols = 32;       // series per tile
constexpr int kGramChunk = 64;      // segments staged per step
constexpr int kCondThreads = 256;
constexpr int kCondMaxWitnesses = 64;
constexpr double kCondPivotTol = 1e-10;

struct GramParams {
    const double2* seg;        // lcsd_segment_kernel's table [cx + cy][nslots]
    long long nslots;
    const LpsdFreq* plan;
    int nf;
    long long cx, cy;
    long long row_tiles, col_tiles;  // block tiles: row_tiles x col_tiles, then ceil(cy / kGramCols) diagonal tiles
    double* sxx;               // [cx][cx][nf] (re, im): upper triangle written here
    double* syy;               // [cy][nf]
    double* sxy;               // [cx][cy][nf] (re, im)
};

__global__ void __launch_bounds__(kGramThreads, 3) lcsd_gram_kernel(const GramParams G) {
    constexpr int kWarps = kGramThreads / 32;
    // staging (rows [k][kGramRows + 1], columns [k][kGramCols + 1]: padded so neither the stores nor the reads of a
    // warp meet bank conflicts) and, after the segment loop, the warp partials [kWarps][kGramRows * kGramCols]
    constexpr int kRowBytes = kGramChunk * (kGramRows + 1) * 16, kColBytes = kGramChunk * (kGramCols + 1) * 16;
    constexpr int kRedBytes = kWarps * kGramRows * kGramCols * 16;
    constexpr int kSmem = kRowBytes + kColBytes > kRedBytes ? kRowBytes + kColBytes : kRedBytes;
    __shared__ __align__(16) unsigned char smem[kSmem];
    double2* srow = reinterpret_cast<double2*>(smem);
    double2* scol = reinterpret_cast<double2*>(smem + kRowBytes);
    double2* red = reinterpret_cast<double2*>(smem);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long tile = blockIdx.x;
    const long long nblock = G.row_tiles * G.col_tiles;
    const bool diag = tile >= nblock;
    long long a0 = 0, b0;
    if (diag) {
        b0 = G.cx + (tile - nblock) * kGramCols;  // target diagonals b0 .. b0 + 31
    } else {
        a0 = (tile / G.col_tiles) * kGramRows;
        b0 = (tile % G.col_tiles) * kGramCols;
        if (b0 + kGramCols <= a0) return;  // wholly below the diagonal of Sxx
    }
    const long long ns = G.cx + G.cy;
    const int ri = lane >> 3, ci = lane & 7;  // block tiles: rows 2 ri, 2 ri + 1; columns ci + 8 m
    for (int j = blockIdx.y; j < G.nf; j += gridDim.y) {
        const LpsdFreq F = G.plan[j];
        const double2* base = G.seg + F.group0 * kLpsdGroup;
        double2 acc[2][4];
#pragma unroll
        for (int r = 0; r < 2; ++r)
#pragma unroll
            for (int m = 0; m < 4; ++m) acc[r][m] = make_double2(0.0, 0.0);
        for (long long k0 = 0; k0 < F.K; k0 += kGramChunk) {
            __syncthreads();  // the previous chunk's (or row's) reads of the staging area are done
            for (int i = tid; i < kGramCols * kGramChunk; i += kGramThreads) {
                const int c = i / kGramChunk, k = i % kGramChunk;
                const long long b = b0 + c;
                scol[k * (kGramCols + 1) + c] =
                    (b < ns && k0 + k < F.K) ? base[b * G.nslots + k0 + k] : make_double2(0.0, 0.0);
            }
            if (!diag) {
                for (int i = tid; i < kGramRows * kGramChunk; i += kGramThreads) {
                    const int r = i / kGramChunk, k = i % kGramChunk;
                    const long long a = a0 + r;
                    srow[k * (kGramRows + 1) + r] =
                        (a < G.cx && k0 + k < F.K) ? base[a * G.nslots + k0 + k] : make_double2(0.0, 0.0);
                }
            }
            __syncthreads();
            if (diag) {
#pragma unroll 4
                for (int k = warp; k < kGramChunk; k += kWarps) {
                    const double2 q = scol[k * (kGramCols + 1) + lane];
                    acc[0][0].x = fma(q.x, q.x, acc[0][0].x);
                    acc[0][0].x = fma(q.y, q.y, acc[0][0].x);
                }
            } else {
#pragma unroll 1
                for (int k = warp; k < kGramChunk; k += kWarps) {
                    double2 p[2], q[4];
#pragma unroll
                    for (int r = 0; r < 2; ++r) p[r] = srow[k * (kGramRows + 1) + 2 * ri + r];
#pragma unroll
                    for (int m = 0; m < 4; ++m) q[m] = scol[k * (kGramCols + 1) + ci + 8 * m];
                    // A conj(B) = (p.x q.x + p.y q.y) + i (p.y q.x - p.x q.y)
#pragma unroll
                    for (int r = 0; r < 2; ++r)
#pragma unroll
                        for (int m = 0; m < 4; ++m) {
                            acc[r][m].x = fma(p[r].x, q[m].x, acc[r][m].x);
                            acc[r][m].x = fma(p[r].y, q[m].y, acc[r][m].x);
                            acc[r][m].y = fma(p[r].y, q[m].x, acc[r][m].y);
                            acc[r][m].y = fma(-p[r].x, q[m].y, acc[r][m].y);
                        }
                }
            }
        }
        __syncthreads();  // staging reads done: the area now holds the warp partials
        if (diag) {
            red[warp * kGramCols + lane] = acc[0][0];
        } else {
#pragma unroll
            for (int r = 0; r < 2; ++r)
#pragma unroll
                for (int m = 0; m < 4; ++m) red[warp * (kGramRows * kGramCols) + (2 * ri + r) * kGramCols + ci + 8 * m] = acc[r][m];
        }
        __syncthreads();
        const int nout = diag ? kGramCols : kGramRows * kGramCols;
        if (tid < nout) {
            const int stride = diag ? kGramCols : kGramRows * kGramCols;
            double2 w[kWarps];
#pragma unroll
            for (int v = 0; v < kWarps; ++v) w[v] = red[v * stride + tid];
            const double re = ((w[0].x + w[1].x) + (w[2].x + w[3].x)) + ((w[4].x + w[5].x) + (w[6].x + w[7].x));
            const double im = ((w[0].y + w[1].y) + (w[2].y + w[3].y)) + ((w[4].y + w[5].y) + (w[6].y + w[7].y));
            if (diag) {
                const long long b = b0 + tid;
                if (b < ns) G.syy[(b - G.cx) * G.nf + j] = re;
            } else {
                const long long a = a0 + tid / kGramCols, b = b0 + tid % kGramCols;
                if (a < G.cx && b < ns) {
                    if (b >= G.cx) {
                        double* o = G.sxy + 2 * ((a * G.cy + (b - G.cx)) * G.nf + j);
                        o[0] = re;
                        o[1] = im;
                    } else if (b >= a) {
                        double* o = G.sxx + 2 * ((a * G.cx + b) * G.nf + j);
                        o[0] = re;
                        o[1] = im;
                    }
                }
            }
        }
    }
}

struct CondParams {
    LpsdParams P;              // the plan and window (for S2_j); series pointers unused
    long long cx, cy;
    double fs;
    double* sxx;               // [cx][cx][nf] (re, im): upper triangle in raw sums on entry, the full matrix on exit
    double* syy;               // [cy][nf]: raw sums on entry, scaled on exit
    double* sxy;               // [cx][cy][nf] (re, im): likewise
    double* h;                 // [cx][cy][nf] (re, im)
    double* sres;              // [cy][nf]
    double* mcoh;              // [cy][nf]
    double* enbw;              // [nf]
};

DFK_D double2 cmul(double2 a, double2 b) { return make_double2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
DFK_D double2 cmul_conj(double2 a, double2 b) { return make_double2(a.x * b.x + a.y * b.y, a.y * b.x - a.x * b.y); }  // a conj(b)

// Per frequency row: window sums, scaling of every sum lcsd's way (2 (sum / K) / (fs S2)), Sxx completed by
// conjugation; then the Cholesky factor L of Sxx (lower triangle of the shared matrix, leading dimension cx + 1) and,
// for each target, L z = Sxy[:,t], L^H H = z, Sres = Syy - |z|^2.  Dynamic shared memory: cx (cx + 1) double2.
__global__ void __launch_bounds__(kCondThreads) lcsd_cond_kernel(const CondParams C) {
    constexpr int kWarps = kCondThreads / 32;
    extern __shared__ double2 M[];
    __shared__ double r1[kWarps], r2[kWarps];
    __shared__ double diag0[kCondMaxWitnesses];
    __shared__ int singular;
    const int j = blockIdx.x;
    const int nf = C.P.nf;
    const LpsdFreq F = C.P.plan[j];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int cx = static_cast<int>(C.cx), ld = cx + 1;
    const long long cy = C.cy;
    double s1, s2;
    lpsd_window_sums<kCondThreads>(C.P, F, r1, r2, s1, s2);
    const double K = static_cast<double>(F.K), den = C.fs * s2;
    for (int i = tid; i < cx * cx; i += kCondThreads) {
        const int a = i / cx, b = i % cx;
        if (b < a) continue;
        double* o = C.sxx + 2 * ((static_cast<long long>(a) * cx + b) * nf + j);
        const double re = 2.0 * (o[0] / K) / den, im = a == b ? 0.0 : 2.0 * (o[1] / K) / den;
        o[0] = re;
        o[1] = im;
        M[a * ld + b] = make_double2(re, im);
        if (a != b) {
            double* t = C.sxx + 2 * ((static_cast<long long>(b) * cx + a) * nf + j);
            t[0] = re;
            t[1] = -im;
            M[b * ld + a] = make_double2(re, -im);
        } else {
            diag0[a] = re;
        }
    }
    for (long long i = tid; i < cx * cy; i += kCondThreads) {
        double* o = C.sxy + 2 * (i * nf + j);
        o[0] = 2.0 * (o[0] / K) / den;
        o[1] = 2.0 * (o[1] / K) / den;
    }
    for (long long t = tid; t < cy; t += kCondThreads) C.syy[t * nf + j] = 2.0 * (C.syy[t * nf + j] / K) / den;
    if (tid == 0) {
        C.enbw[j] = C.fs * s2 / (s1 * s1);
        singular = F.K < cx;
    }
    __syncthreads();
    // Cholesky, right-looking: column k of L, then the trailing lower triangle
    for (int k = 0; k < cx && !singular; ++k) {
        const double d = M[k * ld + k].x;
        if (!(d > kCondPivotTol * diag0[k])) {  // also NaN and a zero witness
            __syncthreads();                    // every thread has read d before the flag changes
            if (tid == 0) singular = 1;
            __syncthreads();
            break;
        }
        const double l = sqrt(d);
        for (int i = k + 1 + tid; i < cx; i += kCondThreads) {
            const double2 v = M[i * ld + k];
            M[i * ld + k] = make_double2(v.x / l, v.y / l);
        }
        __syncthreads();
        if (tid == 0) M[k * ld + k] = make_double2(l, 0.0);
        const int m = cx - k - 1;
        for (int i = tid; i < m * m; i += kCondThreads) {
            const int r = k + 1 + i / m, c = k + 1 + i % m;
            if (c > r) continue;
            const double2 u = cmul_conj(M[r * ld + k], M[c * ld + k]);
            M[r * ld + c].x -= u.x;
            M[r * ld + c].y -= u.y;
        }
        __syncthreads();
    }
    const bool bad = singular;
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    // a warp per target; lane owns rows lane and lane + 32 of the solves
    for (long long t = warp; t < cy; t += kWarps) {
        const double syy = C.syy[t * nf + j];
        double2 z0 = make_double2(0.0, 0.0), z1 = z0;
        if (lane < cx) {
            const double* o = C.sxy + 2 * ((lane * cy + t) * nf + j);
            z0 = make_double2(o[0], o[1]);
        }
        if (lane + 32 < cx) {
            const double* o = C.sxy + 2 * (((lane + 32) * cy + t) * nf + j);
            z1 = make_double2(o[0], o[1]);
        }
        double zz = 0.0;
        if (!bad) {
            // forward: L z = b, column by column
            for (int k = 0; k < cx; ++k) {
                const double2 own = k < 32 ? z0 : z1;
                const double l = M[k * ld + k].x;
                double2 zk;
                zk.x = __shfl_sync(0xffffffffu, own.x, k & 31) / l;
                zk.y = __shfl_sync(0xffffffffu, own.y, k & 31) / l;
                zz += zk.x * zk.x + zk.y * zk.y;
                if (lane == (k & 31)) {
                    if (k < 32) z0 = zk; else z1 = zk;
                }
                if (lane > k && lane < cx) {
                    const double2 u = cmul(M[lane * ld + k], zk);
                    z0.x -= u.x;
                    z0.y -= u.y;
                }
                if (lane + 32 > k && lane + 32 < cx) {
                    const double2 u = cmul(M[(lane + 32) * ld + k], zk);
                    z1.x -= u.x;
                    z1.y -= u.y;
                }
            }
            // backward: L^H h = z, column by column from the last row
            for (int k = cx - 1; k >= 0; --k) {
                const double2 own = k < 32 ? z0 : z1;
                const double l = M[k * ld + k].x;
                double2 hk;
                hk.x = __shfl_sync(0xffffffffu, own.x, k & 31) / l;
                hk.y = __shfl_sync(0xffffffffu, own.y, k & 31) / l;
                if (lane == (k & 31)) {
                    if (k < 32) z0 = hk; else z1 = hk;
                }
                // row i < k of L^H holds conj(L[k][i]) in column k
                if (lane < k) {
                    const double2 u = cmul_conj(hk, M[k * ld + lane]);
                    z0.x -= u.x;
                    z0.y -= u.y;
                }
                if (lane + 32 < k) {
                    const double2 u = cmul_conj(hk, M[k * ld + lane + 32]);
                    z1.x -= u.x;
                    z1.y -= u.y;
                }
            }
        }
        if (lane < cx) {
            double* o = C.h + 2 * ((lane * cy + t) * nf + j);
            o[0] = bad ? nan : z0.x;
            o[1] = bad ? nan : z0.y;
        }
        if (lane + 32 < cx) {
            double* o = C.h + 2 * (((lane + 32) * cy + t) * nf + j);
            o[0] = bad ? nan : z1.x;
            o[1] = bad ? nan : z1.y;
        }
        if (lane == 0) {
            const double res = bad ? nan : syy - zz;
            C.sres[t * nf + j] = res;
            C.mcoh[t * nf + j] = (bad || syy == 0.0) ? nan : 1.0 - res / syy;
        }
    }
}

}  // namespace dfk
