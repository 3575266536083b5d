// Time-domain stability of C series (NIST SP 1065, Riley 2008; the conventions of allantools): overlapping Allan,
// modified Allan, time and overlapping Hadamard deviations at a list of averaging factors m.
//
// With x the phase series (the input for 'phase' data; x_0 = 0, x_n = sum_{i<n} y_i for 'freq' data, in units of
// samples: tau0 is applied only in the final scaling) and S_k = sum_{i<k} x_i, every term is a second or third
// difference of x or S at offsets m.  Those differences are tiny against the running sums they are taken from: in fp64
// the running sum of a drifting series loses the difference to cancellation (the cumsum route of allantools).  Here the
// running sums are carried in double-double (hi, lo), every difference is formed in double-double and rounded once to
// fp64 before it is squared, so each term is the correctly rounded difference of running sums that are themselves
// exact to 2^-106 (exact for series on a grid whose sums stay below 2^106 grid steps).
//
// Device work per call: the running sum X by a three-phase scan per channel ('freq'; 'phase' data is only copied),
// the same scan over X for S when mdev or tdev is requested, one terms launch over a host-built table of slices
// (m, first term) and one finish launch.  Every sum is formed in a fixed order and no atomics are used, so results
// are bit-identical between runs, for a channel alone or in a batch, over strides, and for an m alone or in a list.
//
// The double-double helpers are __host__ __device__ and round every operation explicitly (__dadd_rn, fma), so a g++
// build with -ffp-contract=off (tests/host/stability_harness.cpp) computes the same terms.
#pragma once
#include "dfk_common.cuh"

namespace dfk {

struct DDval {
    double hi, lo;
};

DFK_HD double dd_plus(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}
DFK_HD double dd_minus(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dsub_rn(a, b);
#else
    return a - b;
#endif
}

// a + b = s + e exactly (Knuth)
DFK_HD DDval two_sum(double a, double b) {
    const double s = dd_plus(a, b);
    const double bb = dd_minus(s, a);
    const double e = dd_plus(dd_minus(a, dd_minus(s, bb)), dd_minus(b, bb));
    return {s, e};
}

// a + b = s + e exactly when |a| >= |b| (Dekker)
DFK_HD DDval fast_two_sum(double a, double b) {
    const double s = dd_plus(a, b);
    return {s, dd_minus(b, dd_minus(s, a))};
}

// double-double sum with the error of both halves carried (QD's accurate addition)
DFK_HD DDval dd_add(DDval a, DDval b) {
    DDval s = two_sum(a.hi, b.hi);
    const DDval t = two_sum(a.lo, b.lo);
    s = fast_two_sum(s.hi, dd_plus(s.lo, t.hi));
    return fast_two_sum(s.hi, dd_plus(s.lo, t.lo));
}

DFK_HD DDval dd_neg(DDval a) { return {-a.hi, -a.lo}; }

// k a for a small integer k (here +-2, +-3): k hi = p + e exactly by fma; k lo + e rounded once
DFK_HD DDval dd_mul_small(DDval a, double k) {
    const double p = k * a.hi;
    const double e = fma(k, a.hi, -p);
    return fast_two_sum(p, fma(k, a.lo, e));
}

DFK_HD double dd_round(DDval a) { return dd_plus(a.hi, a.lo); }

// x_{i+2m} - 2 x_{i+m} + x_i, rounded once
DFK_HD double stab_second_diff(DDval x0, DDval x1, DDval x2) {
    return dd_round(dd_add(dd_add(x2, x0), dd_mul_small(x1, -2.0)));
}

// x_{i+3m} - 3 x_{i+2m} + 3 x_{i+m} - x_i = (x3 - x0) - 3 (x2 - x1), rounded once
DFK_HD double stab_third_diff(DDval x0, DDval x1, DDval x2, DDval x3) {
    return dd_round(dd_add(dd_add(x3, dd_neg(x0)), dd_mul_small(dd_add(x2, dd_neg(x1)), -3.0)));
}

// Slots of the outputs, in the ABI's order, and the three sums the terms kernel forms (tdev comes from mdev's).
constexpr int kStabOadev = 0, kStabMdev = 1, kStabTdev = 2, kStabOhdev = 3;
constexpr int kStabSums = 3;  // sums of squared terms: oadev, mdev, ohdev

// Term counts of averaging factor m on Nx phase points (<= 0: that kind has no term at m).
DFK_HD long long stab_n_oadev(long long Nx, long long m) { return Nx - 2 * m; }
DFK_HD long long stab_n_mdev(long long Nx, long long m) { return Nx - 3 * m + 1; }
DFK_HD long long stab_n_ohdev(long long Nx, long long m) { return Nx - 3 * m; }

// The deviations of one (m, channel) from its sums of squared terms.  scale = 1 for 'freq' data (x is in units of
// samples times tau0, so tau0 cancels), fs for 'phase' data.  dev[4] in slot order; a kind with n <= 0 gives NaN.
DFK_HD void stab_finish_one(const double sums[kStabSums], long long m, long long Nx, double fs, double scale,
                            double dev[4]) {
    const double md = static_cast<double>(m), nan = ::nan("");
    const long long na = stab_n_oadev(Nx, m), nm = stab_n_mdev(Nx, m), nh = stab_n_ohdev(Nx, m);
    dev[kStabOadev] = na > 0 ? scale * std::sqrt(sums[0] / (2.0 * md * md * static_cast<double>(na))) : nan;
    dev[kStabMdev] = nm > 0 ? scale * std::sqrt(sums[1] / (2.0 * static_cast<double>(nm))) / (md * md) : nan;
    dev[kStabTdev] = md / fs * dev[kStabMdev] / std::sqrt(3.0);
    dev[kStabOhdev] = nh > 0 ? scale * std::sqrt(sums[2] / (6.0 * md * md * static_cast<double>(nh))) : nan;
}

// Scan geometry: a tile of 2048 samples per CTA, 8 consecutive samples per thread.
constexpr int kStabScanThreads = 256;
constexpr int kStabScanItems = 8;
constexpr int kStabTile = kStabScanThreads * kStabScanItems;
// Terms geometry: a slice of 4096 consecutive terms of one (m, channel) per CTA, thread t taking terms
// first + t + 256 r (r < 16) in order, then a fixed tree over the 256 threads.
constexpr int kStabTermThreads = 256;
constexpr int kStabTermsPerThread = 16;
constexpr long long kStabSlice = static_cast<long long>(kStabTermThreads) * kStabTermsPerThread;
constexpr int kStabFinishThreads = 128;

// One slice of the terms launch: averaging factor m, terms [first, first + kStabSlice) clipped to each kind's count.
struct StabSlice {
    long long m, first;
};

// One averaging factor of the finish launch: its slices are [e0, e0 + ns) of the table.
struct StabTau {
    long long m, e0, ns;
};

#if defined(__CUDACC__)

// Input of one scan: sample i of series c is v[c ld_c + i stride] (fp64, lo = 0) or X[c ld_c + i] (double-double).
struct StabScanParams {
    const double* v;
    const double2* X;
    long long ld_c, stride;
    long long L;        // input samples per series; the output has L + 1: out[0] = 0, out[k] = sum_{i<k} in_i
    long long ntiles;   // ceil(L / kStabTile)
    double2* tsum;      // [C][ntiles]: tile sums, then (after the carry pass) the exclusive carries
    double2* out;       // [C][ld_out]
    long long ld_out;
    int* bad;           // [C]: set to 1 by the fp64 input pass when a sample is not finite
};

DFK_D DDval dd_load(const double2* p) {
    const double2 v = *p;
    return {v.x, v.y};
}
DFK_D void dd_store(double2* p, DDval a) { *p = make_double2(a.hi, a.lo); }

DFK_D DDval dd_shfl_up(DDval a, int off) {
    return {__shfl_up_sync(0xffffffffu, a.hi, off), __shfl_up_sync(0xffffffffu, a.lo, off)};
}

// Inclusive scan over the lanes of a warp (Hillis-Steele, fixed order).
DFK_D DDval warp_incl_scan(DDval a, int lane) {
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const DDval o = dd_shfl_up(a, off);
        if (lane >= off) a = dd_add(o, a);
    }
    return a;
}

// shared-memory index of tile element i: one pad slot per 8 keeps a thread's 8 consecutive elements off the banks of
// its neighbours'
DFK_D int stab_pad(int i) { return i + (i >> 3); }

// kWrite = false: phase 1, the tile's sum to tsum (and, for fp64 input, the non-finite flag).  kWrite = true: phase 3,
// the in-tile inclusive scan plus the tile's carry, written to out[idx + 1] (and out[0] = 0).
template <bool kDD, bool kWrite>
__global__ void __launch_bounds__(kStabScanThreads) stab_scan_kernel(StabScanParams P) {
    __shared__ double2 sm[kStabTile + kStabTile / 8];
    __shared__ double2 wsum[kStabScanThreads / 32];
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const long long c = static_cast<long long>(blockIdx.x) / P.ntiles;
    const long long tile = static_cast<long long>(blockIdx.x) - c * P.ntiles;
    const long long base = tile * kStabTile;
    bool nonfinite = false;
#pragma unroll
    for (int k = 0; k < kStabScanItems; ++k) {
        const int i = k * kStabScanThreads + t;
        const long long idx = base + i;
        double2 x = make_double2(0.0, 0.0);
        if (idx < P.L) {
            if (kDD) {
                x = P.X[c * P.ld_c + idx];
            } else {
                x.x = P.v[c * P.ld_c + idx * P.stride];
                nonfinite |= !isfinite(x.x);
            }
        }
        sm[stab_pad(i)] = x;
    }
    if (!kDD && !kWrite && nonfinite) P.bad[c] = 1;  // every writer stores the same value
    __syncthreads();
    DDval loc[kStabScanItems];
    DDval run = dd_load(&sm[stab_pad(t * kStabScanItems)]);
    loc[0] = run;
#pragma unroll
    for (int k = 1; k < kStabScanItems; ++k) {
        run = dd_add(run, dd_load(&sm[stab_pad(t * kStabScanItems + k)]));
        loc[k] = run;
    }
    const DDval wincl = warp_incl_scan(run, lane);
    DDval wexcl = dd_shfl_up(wincl, 1);
    if (lane == 31) dd_store(&wsum[warp], wincl);
    __syncthreads();
    DDval off = {0.0, 0.0};
    for (int w = 0; w < warp; ++w) off = dd_add(off, dd_load(&wsum[w]));
    if (lane > 0) off = dd_add(off, wexcl);
    if (!kWrite) {
        if (t == kStabScanThreads - 1) dd_store(&P.tsum[c * P.ntiles + tile], dd_add(off, run));
        return;
    }
    const DDval pre = dd_add(dd_load(&P.tsum[c * P.ntiles + tile]), off);
#pragma unroll
    for (int k = 0; k < kStabScanItems; ++k) dd_store(&sm[stab_pad(t * kStabScanItems + k)], dd_add(pre, loc[k]));
    __syncthreads();
    double2* out = P.out + c * P.ld_out;
#pragma unroll
    for (int k = 0; k < kStabScanItems; ++k) {
        const int i = k * kStabScanThreads + t;
        if (base + i < P.L) out[base + i + 1] = sm[stab_pad(i)];
    }
    if (tile == 0 && t == 0) out[0] = make_double2(0.0, 0.0);
}

// Phase 2: one warp per channel turns its tile sums into exclusive carries, 32 tiles at a time in tile order.
__global__ void __launch_bounds__(128) stab_carry_kernel(double2* tsum, long long ntiles, long long C) {
    const long long c = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (c >= C) return;  // whole warps
    double2* ts = tsum + c * ntiles;
    DDval carry = {0.0, 0.0};
    for (long long k0 = 0; k0 < ntiles; k0 += 32) {
        const long long k = k0 + lane;
        const DDval a = k < ntiles ? dd_load(&ts[k]) : DDval{0.0, 0.0};
        const DDval incl = warp_incl_scan(a, lane);
        const DDval excl = dd_shfl_up(incl, 1);
        if (k < ntiles) dd_store(&ts[k], lane > 0 ? dd_add(carry, excl) : carry);
        const DDval total = {__shfl_sync(0xffffffffu, incl.hi, 31), __shfl_sync(0xffffffffu, incl.lo, 31)};
        carry = dd_add(carry, total);
    }
}

// 'phase' data: X = the input with lo = 0, on the scan's tiles.
__global__ void __launch_bounds__(kStabScanThreads) stab_load_kernel(StabScanParams P) {
    const long long c = static_cast<long long>(blockIdx.x) / P.ntiles;
    const long long base = (static_cast<long long>(blockIdx.x) - c * P.ntiles) * kStabTile;
    bool nonfinite = false;
#pragma unroll
    for (int k = 0; k < kStabScanItems; ++k) {
        const long long idx = base + k * kStabScanThreads + threadIdx.x;
        if (idx < P.L) {
            const double v = P.v[c * P.ld_c + idx * P.stride];
            nonfinite |= !isfinite(v);
            P.out[c * P.ld_out + idx] = make_double2(v, 0.0);
        }
    }
    if (nonfinite) P.bad[c] = 1;
}

struct StabTermsParams {
    const double2* X;   // [C][ld]
    const double2* S;   // [C][ld] or nullptr
    long long ld, Nx;
    const StabSlice* slices;
    long long nslices;  // per channel
    int want_a, want_m, want_h;
    double* part;       // [C][nslices][kStabSums]
};

// One CTA per (slice, channel), channel-major so that the slices of one (m, channel) run together and the reads at
// offsets m, 2m, 3m of one running sum meet in L2.
__global__ void __launch_bounds__(kStabTermThreads) stab_terms_kernel(StabTermsParams P) {
    __shared__ double red[kStabSums][kStabTermThreads];
    if (P.nslices == 0) return;
    const int t = threadIdx.x;
    const long long c = static_cast<long long>(blockIdx.x) / P.nslices;
    const long long e = static_cast<long long>(blockIdx.x) - c * P.nslices;
    const StabSlice sl = P.slices[e];
    const long long m = sl.m;
    const long long na = stab_n_oadev(P.Nx, m), nm = stab_n_mdev(P.Nx, m), nh = stab_n_ohdev(P.Nx, m);
    const double2* x = P.X + c * P.ld;
    const double2* s = P.S ? P.S + c * P.ld : nullptr;
    double acc_a = 0.0, acc_m = 0.0, acc_h = 0.0;
    for (int r = 0; r < kStabTermsPerThread; ++r) {
        const long long j = sl.first + static_cast<long long>(r) * kStabTermThreads + t;
        if ((P.want_a || P.want_h) && j < na) {
            const DDval x0 = dd_load(&x[j]), x1 = dd_load(&x[j + m]), x2 = dd_load(&x[j + 2 * m]);
            if (P.want_a) {
                const double d = stab_second_diff(x0, x1, x2);
                acc_a = fma(d, d, acc_a);
            }
            if (P.want_h && j < nh) {
                const double d = stab_third_diff(x0, x1, x2, dd_load(&x[j + 3 * m]));
                acc_h = fma(d, d, acc_h);
            }
        }
        if (P.want_m && j < nm) {
            const double d = stab_third_diff(dd_load(&s[j]), dd_load(&s[j + m]), dd_load(&s[j + 2 * m]),
                                             dd_load(&s[j + 3 * m]));
            acc_m = fma(d, d, acc_m);
        }
    }
    red[0][t] = acc_a;
    red[1][t] = acc_m;
    red[2][t] = acc_h;
    __syncthreads();
#pragma unroll
    for (int w = kStabTermThreads / 2; w > 0; w >>= 1) {
        if (t < w) {
#pragma unroll
            for (int k = 0; k < kStabSums; ++k) red[k][t] = dd_plus(red[k][t], red[k][t + w]);
        }
        __syncthreads();
    }
    if (t < kStabSums) P.part[(c * P.nslices + e) * kStabSums + t] = red[t][0];
}

// One thread per (m, channel): the slices' partials summed in slice order, scaled; out[4][C][n_m].
__global__ void __launch_bounds__(kStabFinishThreads) stab_finish_kernel(const StabTau* taus, int n_m, long long C,
                                                                        const double* part, long long nslices,
                                                                        const int* bad, long long Nx, double fs,
                                                                        double scale, double* out) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= C * n_m) return;
    const long long c = i / n_m;
    const int ti = static_cast<int>(i - c * n_m);
    const StabTau tau = taus[ti];
    double sums[kStabSums] = {0.0, 0.0, 0.0};
    for (long long e = tau.e0; e < tau.e0 + tau.ns; ++e)
        for (int k = 0; k < kStabSums; ++k) sums[k] = dd_plus(sums[k], part[(c * nslices + e) * kStabSums + k]);
    double dev[4];
    stab_finish_one(sums, tau.m, Nx, fs, scale, dev);
    const bool poisoned = bad[c] != 0;
    for (int k = 0; k < 4; ++k) out[(k * C + c) * n_m + ti] = poisoned ? ::nan("") : dev[k];
}

#endif  // __CUDACC__

}  // namespace dfk
