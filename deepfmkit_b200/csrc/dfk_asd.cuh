// 'asd'-mode physics of the reference on the device (physics.py:423-440, 557-611, 615-722), batched over Monte-Carlo
// trials: the exact model the Experiment runner simulates once per trial (experiments.py:15-88).
//   g(t)        = waveform(w_mod t + psi) / max|waveform|                      (unitless frequency modulation)
//   phi_mod(t)  = (2 pi / fs) cumsum((df + n_df(t)) g(t))                      (physics.py:675)
//   tau_dl(t)   = (A_arm sin(w_arm t + psi_arm) + phi lambda / 2 pi) / c       (dynamic main channel)
//   Phi(t)      = w0 ((tau_m + tau_dl) - tau_r) + interp(t - tau_m - tau_dl) - interp(t - tau_r)
//   y(t)        = (A + n_amp(t)) (1 + C cos Phi(t))
// with n_df, n_amp white, sigma = asd sqrt(fs / 2) (physics.py:591-597).  The coloured sources (laser frequency and
// arm-length noise) come from the third-party pyplnoise in the reference and are not generated here; like the
// reference's engine (generate(..., external_noise=...), physics.py:430-434) the kernel takes pre-computed noise series
// for all four sources instead -- laser frequency n_f(t) (w0 -> 2 pi (f0 + n_f)), amplitude, df and, on a dynamic
// channel, arm length (added to the path) -- which then replace the internal draws.
// One CTA per trial: block-wide prefix sum of the frequency waveform into an L2-resident scratch row, then the
// delayed-time interpolation np.interp performs, sample by sample.
#pragma once
#include "dfk_common.cuh"
#include "dfk_rng.cuh"

namespace dfk {

constexpr int kAsdThreads = 256;
constexpr int kAsdPerThread = 4;
constexpr int kAsdTerms = 6;
constexpr double kLightSpeed = 299792458.0;  // speed of light in m/s, the exact SI value the reference uses

struct AsdTrial {  // one Monte-Carlo trial, 26 doubles
    double amp, vis, df, w_mod, psi;
    double omega0;               // 2 pi c / lambda
    double tau_r, tau_m;         // arm delays
    double path0;                // phi lambda / (2 pi)
    double arm_amp, arm_w, arm_psi;
    double sigma_amp, sigma_df;  // white-noise standard deviations per sample
    double seed;                 // noise key (trial number), < 2^53
    double nterms;               // > 0: g = sum_k a_k cos(h_k theta + p_k);  0: g from the waveform table
    double table;                // waveform table row when nterms == 0
    double term[kAsdTerms][3];   // h_k, a_k, p_k   (only the first nterms)
    double dynamic;              // != 0: the channel's arm moves (takes the external arm-length noise)
    double noise_row;            // >= 0: row of the external noise series this trial reads; < 0: internal white noise
};
static_assert(sizeof(AsdTrial) == (19 + 3 * kAsdTerms) * sizeof(double), "AsdTrial layout");

struct AsdParams {
    const AsdTrial* trials;
    long long ntrials;
    long long N;            // samples per trial
    double fs;
    double scale;           // 2 pi / (1 / dt) with dt = t[1] - t[0], as physics.py:672-675 forms it
    const double* tables;   // [ntables][N] unnormalised waveform rows (arbitrary host-evaluated waveforms)
    double* scratch;        // [ntrials][N] running sum of the frequency waveform
    double* y;              // [ntrials][ld]
    long long ld;
    double* truth;          // optional [ntrials][ld]: ground-truth phase w0 ((tau_m + tau_dl) - tau_r)
    // external noise series [rows][N], each optional: laser frequency, amplitude, df, arm length (physics.py:430-434)
    const double* ext_fn;
    const double* ext_amp;
    const double* ext_df;
    const double* ext_arm;
};

DFK_D double asd_waveform(const AsdTrial& tr, const AsdParams& P, long long i) {
    const int nt = static_cast<int>(tr.nterms);
    if (nt == 0) return P.tables[static_cast<long long>(tr.table) * P.N + i];
    const double theta = tr.w_mod * (static_cast<double>(i) / P.fs) + tr.psi;  // omega_mod * time_axis + psi
    double g = 0.0;
    for (int k = 0; k < nt; ++k) g += tr.term[k][1] * cos(tr.term[k][0] * theta + tr.term[k][2]);
    return g;
}

// np.interp(x, t, f) on the uniform grid t_j = j / fs with the end values held outside it
DFK_D double asd_interp(const double* __restrict__ f, long long N, double fs, double scale, double x) {
    if (!(x > 0.0)) return scale * f[0];
    double u = x * fs;
    long long j = static_cast<long long>(u);
    if (j >= N - 1) return scale * f[N - 1];
    // guard the rounding of x * fs against the grid the reference searches (t_j = j / fs)
    double tj = static_cast<double>(j) / fs;
    if (tj > x) {
        --j;
        tj = static_cast<double>(j) / fs;
    }
    const double tj1 = static_cast<double>(j + 1) / fs;
    const double f0 = scale * f[j], f1 = scale * f[j + 1];
    const double slope = (f1 - f0) / (tj1 - tj);
    return slope * (x - tj) + f0;
}

__global__ void __launch_bounds__(kAsdThreads) synth_asd_kernel(const AsdParams P) {
    __shared__ double red[kAsdThreads / 32];
    __shared__ double carry_sh;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (long long j = blockIdx.x; j < P.ntrials; j += gridDim.x) {
        AsdTrial tr = P.trials[j];
        const unsigned long long key = static_cast<unsigned long long>(tr.seed);
        const bool ext = tr.noise_row >= 0.0;
        const long long erow = ext ? static_cast<long long>(tr.noise_row) * P.N : 0;
        const double* e_fn = ext && P.ext_fn ? P.ext_fn + erow : nullptr;
        const double* e_amp = ext && P.ext_amp ? P.ext_amp + erow : nullptr;
        const double* e_df = ext && P.ext_df ? P.ext_df + erow : nullptr;
        const double* e_arm = ext && P.ext_arm && tr.dynamic != 0.0 ? P.ext_arm + erow : nullptr;
        if (ext) tr.sigma_amp = tr.sigma_df = 0.0;  // external series replace the internal draws, missing ones are zero
        double* phi = P.scratch + j * P.N;
        // ---- normalisation of the waveform: max |g| over the trial (physics.py:668-669) ----
        double gmax = 0.0;
        for (long long i = threadIdx.x; i < P.N; i += kAsdThreads) gmax = fmax(gmax, fabs(asd_waveform(tr, P, i)));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) gmax = fmax(gmax, __shfl_xor_sync(0xffffffffu, gmax, o));
        __syncthreads();
        if (lane == 0) red[warp] = gmax;
        __syncthreads();
        gmax = 0.0;
#pragma unroll
        for (int w = 0; w < kAsdThreads / 32; ++w) gmax = fmax(gmax, red[w]);
        const double ginv = gmax != 0.0 ? 1.0 / gmax : 0.0;
        // ---- running sum of (df + n_df) g: tiles of 1024 samples, four consecutive samples per thread ----
        if (threadIdx.x == 0) carry_sh = 0.0;
        __syncthreads();
        for (long long base = 0; base < P.N; base += kAsdThreads * kAsdPerThread) {
            const long long i0 = base + static_cast<long long>(threadIdx.x) * kAsdPerThread;
            double v[kAsdPerThread];
            float z[4];
            if (tr.sigma_df != 0.0) normal4(key, static_cast<unsigned long long>(i0 >> 2), 0xdf00u, z);
            double run = 0.0;
#pragma unroll
            for (int e = 0; e < kAsdPerThread; ++e) {
                const long long i = i0 + e;
                double inc = 0.0;
                if (i < P.N) {
                    const double g = asd_waveform(tr, P, i) * ginv;
                    const double dfn = e_df ? tr.df + e_df[i]
                                            : (tr.sigma_df != 0.0 ? tr.df + tr.sigma_df * static_cast<double>(z[e]) : tr.df);
                    inc = dfn * g;
                }
                run += inc;
                v[e] = run;
            }
            // exclusive scan of the thread totals over the CTA
            double inc = run;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const double t = __shfl_up_sync(0xffffffffu, inc, o);
                if (lane >= o) inc += t;
            }
            if (lane == 31) red[warp] = inc;
            __syncthreads();
            double before = carry_sh + inc - run;
            for (int w = 0; w < warp; ++w) before += red[w];
#pragma unroll
            for (int e = 0; e < kAsdPerThread; ++e)
                if (i0 + e < P.N) phi[i0 + e] = before + v[e];
            __syncthreads();
            if (threadIdx.x == kAsdThreads - 1) carry_sh = before + run;
            __syncthreads();
        }
        // ---- delayed-time interpolation and the interferometer output ----
        const double scale = P.scale;
        for (long long i0 = static_cast<long long>(threadIdx.x) * 4; i0 < P.N; i0 += kAsdThreads * 4) {
            float z[4];
            if (tr.sigma_amp != 0.0) normal4(key, static_cast<unsigned long long>(i0 >> 2), 0xa300u, z);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const long long i = i0 + e;
                if (i >= P.N) break;
                const double t = static_cast<double>(i) / P.fs;
                double path;
                if (e_arm)  // physics.py:686-688: modulation + noise + static offset, in this order
                    path = (tr.arm_amp != 0.0 ? tr.arm_amp * sin(tr.arm_w * t + tr.arm_psi) : 0.0) + e_arm[i] + tr.path0;
                else
                    path = tr.arm_amp != 0.0 ? tr.arm_amp * sin(tr.arm_w * t + tr.arm_psi) + 0.0 + tr.path0 : tr.path0;
                const double tau_dl = path / kLightSpeed;
                const double pm_meas = asd_interp(phi, P.N, P.fs, scale, t - (tr.tau_m + tau_dl));
                const double pm_ref = asd_interp(phi, P.N, P.fs, scale, t - tr.tau_r);
                const double lag = (tr.tau_m + tau_dl) - tr.tau_r;
                const double geom = tr.omega0 * lag;
                // physics.py:703-705: the carrier term with the noisy optical frequency f0 + n_f(t)
                const double carrier = e_fn ? (2.0 * kPi * (tr.omega0 / (2.0 * kPi) + e_fn[i])) * lag : geom;
                const double phase = carrier + (pm_meas - pm_ref);
                const double a = e_amp ? tr.amp + e_amp[i]
                                       : (tr.sigma_amp != 0.0 ? tr.amp + tr.sigma_amp * static_cast<double>(z[e]) : tr.amp);
                P.y[j * P.ld + i] = a * (1.0 + tr.vis * cos(phase));
                if (P.truth) P.truth[j * P.ld + i] = geom;
            }
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Reduction of a batch of trial results to the statistics Experiment.run reports per grid point
// (experiments.py:432-446): nanmean, nanstd (population), nanmin, nanmax and the "worst" trial, the value farthest
// from the mean (or from center[point][col] when given).  values[point][trial][col] with a column stride.
// A grid point's trials are cut into slices, one CTA per (slice, point); a thread takes whole rows, so that the table
// is read by coalesced row loads once per pass whatever the number of columns (a CTA per (point, column) striding over
// the rows ran at 0.5 TB/s on the 19 x 1e6 table of the Monte-Carlo sweep).  Pass 1: sum, count, min, max per slice.
// Pass 2: every CTA forms the point's mean from the slice partials, then its slice's centred sum of squares and
// farthest trial.  Finish: one thread per (point, column) combines the slices in slice order (deterministic).
// ---------------------------------------------------------------------------------------------------------------
constexpr int kStatThreads = 256;
constexpr int kStatMaxCols = 8;
constexpr int kStatMaxSlices = 64;

struct TrialStats {
    double mean, std, min, max, worst, count;
};
struct StatPart1 {
    double sum, cnt, mn, mx;
};
struct StatPart2 {
    double q, far;
    long long far_t;
    long long pad;
};

// CTA blockIdx.x = point * nslices + slice
DFK_D void stat_slice(long long ntrials, int nslices, long long& point, int& slice, long long& lo, long long& hi) {
    point = blockIdx.x / nslices;
    slice = static_cast<int>(blockIdx.x - point * nslices);
    const long long per = (ntrials + nslices - 1) / nslices;
    lo = slice * per;
    hi = lo + per < ntrials ? lo + per : ntrials;
}

__global__ void __launch_bounds__(kStatThreads) trial_stats_pass1(const double* __restrict__ values, long long ntrials,
                                                                  int ncols, long long col_stride, int nslices,
                                                                  StatPart1* __restrict__ part) {
    __shared__ double sh[kStatThreads / 32][kStatMaxCols][4];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    long long point, lo, hi;
    int slice;
    stat_slice(ntrials, nslices, point, slice, lo, hi);
    const double* v = values + point * ntrials * col_stride;
    const double inf = __longlong_as_double(0x7ff0000000000000ll);
    double s[kStatMaxCols], n[kStatMaxCols], mn[kStatMaxCols], mx[kStatMaxCols];
#pragma unroll
    for (int c = 0; c < kStatMaxCols; ++c) {
        s[c] = n[c] = 0.0;
        mn[c] = inf;
        mx[c] = -inf;
    }
    for (long long t = lo + threadIdx.x; t < hi; t += kStatThreads) {
        const double* row = v + t * col_stride;
#pragma unroll
        for (int c = 0; c < kStatMaxCols; ++c) {
            if (c < ncols) {
                const double x = row[c];
                if (x == x) {
                    s[c] += x;
                    n[c] += 1.0;
                    mn[c] = fmin(mn[c], x);
                    mx[c] = fmax(mx[c], x);
                }
            }
        }
    }
#pragma unroll
    for (int c = 0; c < kStatMaxCols; ++c) {
        if (c < ncols) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                s[c] += __shfl_xor_sync(0xffffffffu, s[c], o);
                n[c] += __shfl_xor_sync(0xffffffffu, n[c], o);
                mn[c] = fmin(mn[c], __shfl_xor_sync(0xffffffffu, mn[c], o));
                mx[c] = fmax(mx[c], __shfl_xor_sync(0xffffffffu, mx[c], o));
            }
            if (lane == 0) {
                sh[warp][c][0] = s[c];
                sh[warp][c][1] = n[c];
                sh[warp][c][2] = mn[c];
                sh[warp][c][3] = mx[c];
            }
        }
    }
    __syncthreads();
    if (threadIdx.x < ncols) {
        const int c = threadIdx.x;
        StatPart1 r = {0.0, 0.0, inf, -inf};
        for (int w = 0; w < kStatThreads / 32; ++w) {
            r.sum += sh[w][c][0];
            r.cnt += sh[w][c][1];
            r.mn = fmin(r.mn, sh[w][c][2]);
            r.mx = fmax(r.mx, sh[w][c][3]);
        }
        part[(point * nslices + slice) * ncols + c] = r;
    }
}

__global__ void __launch_bounds__(kStatThreads) trial_stats_pass2(const double* __restrict__ values, long long ntrials,
                                                                  int ncols, long long col_stride, int nslices,
                                                                  const double* __restrict__ center,
                                                                  const StatPart1* __restrict__ part1,
                                                                  StatPart2* __restrict__ part2) {
    __shared__ double mean_sh[kStatMaxCols], ref_sh[kStatMaxCols];
    __shared__ double shq[kStatThreads / 32][kStatMaxCols], shf[kStatThreads / 32][kStatMaxCols];
    __shared__ long long sht[kStatThreads / 32][kStatMaxCols];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    long long point, lo, hi;
    int slice;
    stat_slice(ntrials, nslices, point, slice, lo, hi);
    const double* v = values + point * ntrials * col_stride;
    if (threadIdx.x < ncols) {
        const int c = threadIdx.x;
        double s = 0.0, n = 0.0;
        for (int k = 0; k < nslices; ++k) {
            s += part1[(point * nslices + k) * ncols + c].sum;
            n += part1[(point * nslices + k) * ncols + c].cnt;
        }
        const double mean = n > 0.0 ? s / n : __longlong_as_double(0x7ff8000000000000ll);
        mean_sh[c] = mean;
        ref_sh[c] = center ? center[point * ncols + c] : mean;
    }
    __syncthreads();
    double mean[kStatMaxCols], ref[kStatMaxCols], q[kStatMaxCols], far[kStatMaxCols];
    long long far_t[kStatMaxCols];
#pragma unroll
    for (int c = 0; c < kStatMaxCols; ++c) {
        mean[c] = c < ncols ? mean_sh[c] : 0.0;
        ref[c] = c < ncols ? ref_sh[c] : 0.0;
        q[c] = 0.0;
        far[c] = -1.0;
        far_t[c] = 0x7fffffffffffffffll;
    }
    for (long long t = lo + threadIdx.x; t < hi; t += kStatThreads) {
        const double* row = v + t * col_stride;
#pragma unroll
        for (int c = 0; c < kStatMaxCols; ++c) {
            if (c < ncols) {
                const double x = row[c];
                if (x == x) {
                    const double d = x - mean[c];
                    q[c] = fma(d, d, q[c]);
                    const double ad = fabs(x - ref[c]);
                    if (ad > far[c]) {  // (a thread's trials ascend: the first of equals stays)
                        far[c] = ad;
                        far_t[c] = t;
                    }
                }
            }
        }
    }
#pragma unroll
    for (int c = 0; c < kStatMaxCols; ++c) {
        if (c < ncols) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                q[c] += __shfl_xor_sync(0xffffffffu, q[c], o);
                const double of = __shfl_xor_sync(0xffffffffu, far[c], o);
                const long long ot = __shfl_xor_sync(0xffffffffu, far_t[c], o);
                if (of > far[c] || (of == far[c] && ot < far_t[c])) {
                    far[c] = of;
                    far_t[c] = ot;
                }
            }
            if (lane == 0) {
                shq[warp][c] = q[c];
                shf[warp][c] = far[c];
                sht[warp][c] = far_t[c];
            }
        }
    }
    __syncthreads();
    if (threadIdx.x < ncols) {
        const int c = threadIdx.x;
        StatPart2 r = {0.0, -1.0, 0x7fffffffffffffffll, 0};
        for (int w = 0; w < kStatThreads / 32; ++w) {
            r.q += shq[w][c];
            if (shf[w][c] > r.far || (shf[w][c] == r.far && sht[w][c] < r.far_t)) {
                r.far = shf[w][c];
                r.far_t = sht[w][c];
            }
        }
        part2[(point * nslices + slice) * ncols + c] = r;
    }
}

__global__ void trial_stats_finish(const double* __restrict__ values, long long npoints, long long ntrials, int ncols,
                                   long long col_stride, int nslices, const StatPart1* __restrict__ part1,
                                   const StatPart2* __restrict__ part2, TrialStats* __restrict__ out) {
    const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (i >= npoints * ncols) return;
    const long long point = i / ncols;
    const int c = static_cast<int>(i - point * ncols);
    const double nan = __longlong_as_double(0x7ff8000000000000ll), inf = __longlong_as_double(0x7ff0000000000000ll);
    double s = 0.0, cnt = 0.0, mn = inf, mx = -inf, q = 0.0, far = -1.0;
    long long far_t = 0x7fffffffffffffffll;
    for (int k = 0; k < nslices; ++k) {
        const StatPart1 a = part1[(point * nslices + k) * ncols + c];
        const StatPart2 b = part2[(point * nslices + k) * ncols + c];
        s += a.sum;
        cnt += a.cnt;
        mn = fmin(mn, a.mn);
        mx = fmax(mx, a.mx);
        q += b.q;
        if (b.far > far || (b.far == far && b.far_t < far_t)) {
            far = b.far;
            far_t = b.far_t;
        }
    }
    TrialStats r;
    r.mean = cnt > 0.0 ? s / cnt : nan;
    r.std = cnt > 0.0 ? sqrt(q / cnt) : nan;
    r.min = cnt > 0.0 ? mn : nan;
    r.max = cnt > 0.0 ? mx : nan;
    // far < 0: no trial had a finite distance (a column holding both +inf and -inf has a NaN mean; a NaN centre),
    // so far_t still holds its sentinel and there is no trial to report
    r.worst = (cnt > 0.0 && far >= 0.0) ? values[(point * ntrials + far_t) * col_stride + c] : nan;
    r.count = cnt;
    out[i] = r;
}

}  // namespace dfk
