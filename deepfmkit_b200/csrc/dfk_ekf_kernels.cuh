// EKF kernels: per-channel record statistics (initial dc and default measurement variance,
// fitters.py:253,256) and the tracking loop itself, one thread per channel (fitters.py:274-308).
#pragma once
#include <type_traits>

#include "dfk_ekf_core.cuh"

namespace dfk {

constexpr int kStatsThreads = 256;
constexpr int kEkfTile = 32;    // samples per staged tile and thread
constexpr int kEkfStages = 3;   // tiles in flight per thread (cp.async groups)

// slab[c] = {mean(z_c), var(z_c)} over the T samples given, numpy's two-pass definition of var (ddof = 0).
// With acc != nullptr the slab's moments are merged into the running {n, mean, M2} of the channel (Chan et al.),
// which is how a record streamed in slabs gets its whole-record mean and variance.
__global__ void __launch_bounds__(kStatsThreads) channel_stats_kernel(const double* __restrict__ z, long long T,
                                                                      long long C, long long ld_t, long long ld_c,
                                                                      double* __restrict__ stats,
                                                                      double* __restrict__ acc) {
    __shared__ double red[kStatsThreads / 32];
    __shared__ double mean_sh;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    for (long long c = blockIdx.x; c < C; c += gridDim.x) {
        const double* zc = z + c * ld_c;
        double sum = 0.0;
        for (long long t = tid; t < T; t += kStatsThreads) sum += zc[t * ld_t];
        sum = warp_sum(sum);
        __syncthreads();
        if (lane == 0) red[warp] = sum;
        __syncthreads();
        if (tid == 0) {
            double v = 0.0;
            for (int w = 0; w < kStatsThreads / 32; ++w) v += red[w];
            mean_sh = v / static_cast<double>(T);
        }
        __syncthreads();
        const double mean = mean_sh;
        sum = 0.0;
        for (long long t = tid; t < T; t += kStatsThreads) {
            const double d = zc[t * ld_t] - mean;
            sum = fma(d, d, sum);
        }
        sum = warp_sum(sum);
        __syncthreads();
        if (lane == 0) red[warp] = sum;
        __syncthreads();
        if (tid == 0) {
            double m2 = 0.0;
            for (int w = 0; w < kStatsThreads / 32; ++w) m2 += red[w];
            if (stats) {
                stats[2 * c] = mean;
                stats[2 * c + 1] = m2 / static_cast<double>(T);
            }
            if (acc) {
                double* a = acc + 3 * c;
                const double na = a[0], nb = static_cast<double>(T), n = na + nb;
                const double delta = mean - a[1];
                a[1] += delta * (nb / n);
                a[2] += m2 + delta * delta * (na * nb / n);
                a[0] = n;
            }
        }
    }
}

// The same moments for time-major records ([T][C], ld_c == 1), where a CTA per channel would touch one 8-byte sample
// per 32-byte sector: lanes take 32 adjacent channels (coalesced rows), the warps of a block and the blocks of
// grid.y split the time axis, and per-block partial sums land in part[split][C] to be added in a fixed order.
// pass 0: part = sum z; pass 1: part = sum (z - mean)^2 with mean = (sum over splits of pass 0) / T.
__global__ void __launch_bounds__(kStatsThreads) stats_tm_kernel(const double* __restrict__ z, long long T, long long C,
                                                                 long long ld_t, int pass, const double* __restrict__ sums,
                                                                 int nsplit_prev, double* __restrict__ part) {
    __shared__ double red[kStatsThreads / 32][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long c = blockIdx.x * 32ll + lane;
    const long long per = (T + gridDim.y - 1) / gridDim.y;
    const long long lo = blockIdx.y * per, hi = (lo + per < T) ? lo + per : T;
    double mean = 0.0;
    if (pass == 1 && c < C) {
        for (int sidx = 0; sidx < nsplit_prev; ++sidx) mean += sums[sidx * C + c];
        mean /= static_cast<double>(T);
    }
    double acc = 0.0;
    if (c < C) {
        for (long long t = lo + warp; t < hi; t += kStatsThreads / 32) {
            const double v = z[t * ld_t + c];
            if (pass == 0) {
                acc += v;
            } else {
                const double d = v - mean;
                acc = fma(d, d, acc);
            }
        }
    }
    red[warp][lane] = acc;
    __syncthreads();
    if (warp == 0 && c < C) {
        double v = 0.0;
        for (int w = 0; w < kStatsThreads / 32; ++w) v += red[w][lane];
        part[blockIdx.y * C + c] = v;
    }
}

// stats[c] = {mean, var} from the two sets of partial sums; merged into acc like channel_stats_kernel when given.
__global__ void stats_tm_finish_kernel(const double* __restrict__ sums, const double* __restrict__ sq, int nsplit,
                                       long long T, long long C, double* __restrict__ stats, double* __restrict__ acc) {
    const long long c = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (c >= C) return;
    double s1 = 0.0, m2 = 0.0;
    for (int i = 0; i < nsplit; ++i) {
        s1 += sums[i * C + c];
        m2 += sq[i * C + c];
    }
    const double mean = s1 / static_cast<double>(T);
    if (stats) {
        stats[2 * c] = mean;
        stats[2 * c + 1] = m2 / static_cast<double>(T);
    }
    if (acc) {
        double* a = acc + 3 * c;
        const double na = a[0], nb = static_cast<double>(T), n = na + nb;
        const double delta = mean - a[1];
        a[1] += delta * (nb / n);
        a[2] += m2 + delta * delta * (na * nb / n);
        a[0] = n;
    }
}

// stats[c] = {mean, M2 / n} from the merged moments.
__global__ void stats_finish_kernel(const double* __restrict__ acc, long long C, double* __restrict__ stats) {
    const long long c = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (c >= C) return;
    stats[2 * c] = acc[3 * c + 1];
    stats[2 * c + 1] = acc[3 * c + 2] / acc[3 * c];
}

// doubles per channel in a carried state: x at [0, 5), the covariance's upper triangle at [5, 20) in tri(i, j) order
// (EkfState::P, the pending update applied), [20, 30) unused, r at [30], [31] unused
constexpr int kEkfStateStride = 32;

struct EkfLaunch {
    long long k0;   // absolute index of the first sample of this call (a multiple of R)
    double* state;  // carried filter state, C x kEkfStateStride (nullptr: single-call mode)
    double init[4];
    double init_dc;  // NaN -> per-channel mean from stats
    double p0[5];
    double q[5];
    double r_val;  // NaN -> per-channel variance from stats
    double w_m, f_samp;
    int cpw;  // channels per warp (power of two <= 32): lanes cpw..31 of every one-warp block idle
};

DFK_D void cp_async8(double* smem_dst, const double* gmem_src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_addr(smem_dst)), "l"(gmem_src) : "memory");
}
DFK_D void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
DFK_D void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

// One-warp blocks, one thread per channel.  The filter is a serial chain per channel, so a warp's pace does not
// depend on how many of its lanes are active; with C channels and 4 sub-partitions per SM the launcher picks the
// fewest channels per warp that still gives every warp a sub-partition of its own (cfg 4: 4096 channels -> 8 per
// warp, 512 warps on 592 sub-partitions).  Samples arrive through each thread's private shared-memory column by
// cp.async, kEkfStages tiles ahead: no registers, no barrier (a thread only ever reads what it copied itself),
// and either record layout ([C][T] or [T][C]) costs one 8-byte copy per sample.
__global__ void __launch_bounds__(32) ekf_kernel(const double* __restrict__ z, long long T, long long C,
                                                 long long ld_t, long long ld_c, long long R, EkfLaunch a,
                                                 const double* __restrict__ stats, double* __restrict__ rows) {
    __shared__ double stage[kEkfStages][kEkfTile][32];
    __shared__ double saved[20][32];  // filter state at the entry of the current tile (per-thread columns)
    const int lane = threadIdx.x;
    const long long c = blockIdx.x * static_cast<long long>(a.cpw) + lane;
    if (lane >= a.cpw || c >= C) return;
    EkfState s;
    EkfConsts k;
    k.w_m = a.w_m;
    k.f_samp = a.f_samp;
    k.inv_fs = 1.0 / a.f_samp;
#pragma unroll
    for (int i = 0; i < 5; ++i) k.q[i] = a.q[i];
    double* carried = a.state ? a.state + c * kEkfStateStride : nullptr;
    if (carried && a.k0 > 0) {  // continuation slab: resume the filter where the previous call left it
#pragma unroll
        for (int i = 0; i < 5; ++i) s.x[i] = carried[i];
#pragma unroll
        for (int i = 0; i < 15; ++i) s.P[i] = carried[5 + i];
        k.r = carried[30];
    } else {
        // (fresh state below)
#pragma unroll
        for (int i = 0; i < 4; ++i) s.x[i] = a.init[i];
        s.x[4] = (a.init_dc == a.init_dc) ? a.init_dc : stats[2 * c];
#pragma unroll
        for (int i = 0; i < 15; ++i) s.P[i] = 0.0;
        s.P[0] = a.p0[0]; s.P[5] = a.p0[1]; s.P[9] = a.p0[2]; s.P[12] = a.p0[3]; s.P[14] = a.p0[4];
        k.r = (a.r_val == a.r_val) ? a.r_val : stats[2 * c + 1];
    }

#pragma unroll
    for (int i = 0; i < 5; ++i) s.kp[i] = s.hp[i] = 0.0;
    const double* zc = z + c * ld_c;
    const long long nbuf = T / R;
    double* out = rows + c * nbuf * 8;
    const long long ntiles = (T + kEkfTile - 1) / kEkfTile;
    auto issue = [&](long long tile) {
        if (tile < ntiles) {
            double* dst = &stage[tile % kEkfStages][0][lane];
            const long long t0 = tile * kEkfTile;
            const int lim = (T - t0 < kEkfTile) ? static_cast<int>(T - t0) : kEkfTile;
            const double* src = zc + t0 * ld_t;
#pragma unroll 8
            for (int i = 0; i < lim; ++i) cp_async8(dst + i * 32, src + i * ld_t);
        }
        cp_async_commit();  // an empty group keeps the wait arithmetic uniform at the tail
    };
#pragma unroll
    for (int p = 0; p < kEkfStages - 1; ++p) issue(p);

    long long until_snap = R;  // samples left before the next state snapshot
    long long snaps = 0;
    double kd = static_cast<double>(a.k0);  // absolute sample index, exact in a double
    // Runs of samples between snapshot points go through a loop without a single branch: the step uses the
    // range-limited sincos / reciprocal and only reports whether every argument stayed in range.  A tile that ever
    // left the range (|angle| >= 1e6, S out of the normal range, NaN) is replayed from its saved entry state with
    // the checked routines -- in practice never, so the compiler can schedule the hot loop as one block.
    auto run_tile = [&](auto fast_tag, const double* src, int lim, EkfState& st, double& kdl, long long& us,
                        long long& sn) -> bool {
        constexpr bool FAST = decltype(fast_tag)::value;
        bool ok = true;
        int pos = 0;
        while (pos < lim) {
            const int run = (us < lim - pos) ? static_cast<int>(us) : lim - pos;
            double A = carrier_angle(kdl, k);
#pragma unroll 1
            for (int i = 0; i < run; ++i) {
                kdl += 1.0;
                const double A_next = carrier_angle(kdl, k);  // off the chain: ready before the next step needs it
                ok &= ekf_step<FAST>(st, src[(pos + i) * 32], A, k);
                A = A_next;
            }
            pos += run;
            us -= run;
            if (us == 0) {
                if (sn < nbuf) {
                    double* row = out + sn * 8;
                    row[0] = st.x[0]; row[1] = st.x[1]; row[2] = st.x[2]; row[3] = st.x[3]; row[4] = st.x[4];
                    row[5] = 0.0; row[6] = 1.0; row[7] = 0.0;  // ssq = 0, fitok = 1 (fitters.py:313-318)
                }
                ++sn;
                us = R;
            }
        }
        return ok;
    };
    for (long long tile = 0; tile < ntiles; ++tile) {
        issue(tile + kEkfStages - 1);
        cp_async_wait<kEkfStages - 1>();
        const double* src = &stage[tile % kEkfStages][0][lane];
        const long long t0 = tile * kEkfTile;
        const int lim = (T - t0 < kEkfTile) ? static_cast<int>(T - t0) : kEkfTile;
        double* sv = &saved[0][lane];
        ekf_flush(s);  // the saved entry state (and the carried one) hold a fully updated covariance
#pragma unroll
        for (int i = 0; i < 5; ++i) sv[i * 32] = s.x[i];
#pragma unroll
        for (int i = 0; i < 15; ++i) sv[(5 + i) * 32] = s.P[i];
        const double kd0 = kd;
        const long long us0 = until_snap, sn0 = snaps;
        if (!run_tile(std::true_type{}, src, lim, s, kd, until_snap, snaps)) {
#pragma unroll
            for (int i = 0; i < 5; ++i) s.x[i] = sv[i * 32];
#pragma unroll
            for (int i = 0; i < 15; ++i) s.P[i] = sv[(5 + i) * 32];
#pragma unroll
            for (int i = 0; i < 5; ++i) s.kp[i] = s.hp[i] = 0.0;
            kd = kd0;
            until_snap = us0;
            snaps = sn0;
            run_tile(std::false_type{}, src, lim, s, kd, until_snap, snaps);
        }
    }
    if (carried) {
        ekf_flush(s);
#pragma unroll
        for (int i = 0; i < 5; ++i) carried[i] = s.x[i];
#pragma unroll
        for (int i = 0; i < 15; ++i) carried[5 + i] = s.P[i];
        carried[30] = k.r;
    }
}

}  // namespace dfk
