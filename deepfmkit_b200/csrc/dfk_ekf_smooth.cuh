// EKF fixed-interval smoother: a Rauch-Tung-Striebel pass over a resident window, one thread per channel.
//
// Window: the T samples of a channel starting at absolute sample k0 (a multiple of R).  x_f[k], P_f[k]: the filter's
// state and covariance after the update with sample k, the pending update applied (what ekf_flush leaves; the
// filter is ekf_kernel's, step for step).  With F = I (fitters.py:276):
//     x_s[T-1] = x_f[T-1],  P_s[T-1] = P_f[T-1]
//     for k = T-2 .. 0:  Pp  = P_f[k] + diag(q)                   the filter's own prediction for step k+1
//                        G   = P_f[k] Pp^-1                       by a 5x5 Cholesky factorisation of Pp
//                        x_s[k] = x_f[k] + G (x_s[k+1] - x_f[k])
//                        P_s[k] = P_f[k] + G (P_s[k+1] - Pp) G^T  carried as its upper triangle, tri(i, j) order
// This is the Kalman smoother of the linearisation the filter used (the measurement linearised at the predicted
// states), so no step is re-linearised.  Row b is the state at k_b = (b+1) R - 1, b < T / R, the sample ekf_kernel
// snapshots; samples after the last snapshot still count as data.  A non-positive or NaN Cholesky pivot, or a NaN
// sample, makes that channel's smoothed states and variances NaN from that step back to the window's start; the
// filtered outputs and the other channels are unaffected.
//
// Device: the forward kernel runs the filter as ekf_kernel does (same step, same 32-sample tiles with the fast /
// checked replay decision per tile, same cp.async staging), writes the filtered rows and variances and checkpoints
// (x, flushed P) every B samples.  B is a multiple of kEkfTile, so a checkpoint is a tile entry and a replay from it is
// bit-identical to the forward run.  The backward kernel walks each channel's blocks from last to first: it re-runs
// the filter from the block's checkpoint into a block store ([step][20][lane] per CTA, lanes coalesced), then runs the
// recursion back through the block.  Neither kernel communicates between threads.
#pragma once
#include "dfk_ekf_core.cuh"

namespace dfk {

constexpr int kSmoothDoubles = 20;  // x[5] and the upper triangle of P [15] per stored step / checkpoint
// Checkpoint interval B when the caller leaves the choice to the library (capped at the window rounded up to a tile).
constexpr long long kSmoothBlockDefault = 256;

DFK_HD int sym(int i, int j) { return i <= j ? tri(i, j) : tri(j, i); }  // index of P_ij in the upper triangle

// One backward step.  xf, Pf: the filtered state and covariance (tri order) at step k; xs, Ps: the smoothed ones at
// k+1 on entry, at k on return.  Every product that meets a sum is an explicit fma or mul_rn, so host and device
// round alike.  Returns false on breakdown (a pivot not > 0): xs and Ps are then NaN.
DFK_HD bool rts_step(const double* xf, const double* Pf, const double* q, double* xs, double* Ps) {
    double L[5][5], inv[5], Pp[15];
#pragma unroll
    for (int i = 0; i < 15; ++i) Pp[i] = Pf[i];
#pragma unroll
    for (int j = 0; j < 5; ++j) Pp[tri(j, j)] = Pf[tri(j, j)] + q[j];
    bool ok = true;
#pragma unroll
    for (int j = 0; j < 5; ++j) {
        double d = Pp[tri(j, j)];
#pragma unroll
        for (int k = 0; k < j; ++k) d = fma(-L[j][k], L[j][k], d);
        ok &= d > 0.0;
        L[j][j] = sqrt(d);
        inv[j] = 1.0 / L[j][j];
#pragma unroll
        for (int i = j + 1; i < 5; ++i) {
            double v = Pp[tri(j, i)];
#pragma unroll
            for (int k = 0; k < j; ++k) v = fma(-L[i][k], L[j][k], v);
            L[i][j] = mul_rn(v, inv[j]);
        }
    }
    // G[c][i] = (Pp^-1 Pf)[i][c]: column c of Pf through L and L^T
    double G[5][5];
#pragma unroll
    for (int c = 0; c < 5; ++c) {
        double y[5];
#pragma unroll
        for (int i = 0; i < 5; ++i) {
            double v = Pf[sym(i, c)];
#pragma unroll
            for (int k = 0; k < i; ++k) v = fma(-L[i][k], y[k], v);
            y[i] = mul_rn(v, inv[i]);
        }
#pragma unroll
        for (int i = 4; i >= 0; --i) {
            double v = y[i];
#pragma unroll
            for (int k = i + 1; k < 5; ++k) v = fma(-L[k][i], y[k], v);
            y[i] = mul_rn(v, inv[i]);
        }
#pragma unroll
        for (int i = 0; i < 5; ++i) G[c][i] = y[i];
    }
    double d[5];
#pragma unroll
    for (int i = 0; i < 5; ++i) d[i] = xs[i] - xf[i];
#pragma unroll
    for (int i = 0; i < 5; ++i) {
        double v = xf[i];
#pragma unroll
        for (int j = 0; j < 5; ++j) v = fma(G[i][j], d[j], v);
        xs[i] = v;
    }
    double M[15];  // P_s[k+1] - Pp
#pragma unroll
    for (int i = 0; i < 15; ++i) M[i] = Ps[i] - Pp[i];
#pragma unroll
    for (int c = 0; c < 5; ++c) {
        double w[5];  // (M G^T)[:, c]
#pragma unroll
        for (int j = 0; j < 5; ++j) {
            double v = mul_rn(M[sym(j, 0)], G[c][0]);
#pragma unroll
            for (int l = 1; l < 5; ++l) v = fma(M[sym(j, l)], G[c][l], v);
            w[j] = v;
        }
#pragma unroll
        for (int i = 0; i <= c; ++i) {
            double v = Pf[tri(i, c)];
#pragma unroll
            for (int j = 0; j < 5; ++j) v = fma(G[i][j], w[j], v);
            Ps[tri(i, c)] = v;
        }
    }
    if (!ok) {
        const double nan = __builtin_nan("");
#pragma unroll
        for (int i = 0; i < 5; ++i) xs[i] = nan;
#pragma unroll
        for (int i = 0; i < 15; ++i) Ps[i] = nan;
    }
    return ok;
}

}  // namespace dfk

#if defined(__CUDACC__)
#include "dfk_ekf_kernels.cuh"

namespace dfk {

struct SmoothLaunch {
    EkfLaunch f;          // filter settings; f.state: the carried state the window starts from (read only) or nullptr
    long long B;          // checkpoint interval, a multiple of kEkfTile
    double* ckpt;         // [ceil(T / B)][20][C]
    double* store;        // per CTA: [B][20][width], width = the CTA's channels
    double* rows;         // [C][nbuf][8] smoothed rows
    double* var;          // [C][nbuf][5] smoothed variances (or nullptr)
    double* filt_rows;    // [C][nbuf][8] filtered rows (or nullptr)
    double* filt_var;     // [C][nbuf][5] filtered variances (or nullptr)
};

// The filter's starting state and constants for channel c, as ekf_kernel sets them up.
DFK_D void smooth_init(const EkfLaunch& a, const double* stats, long long c, EkfState& s, EkfConsts& k) {
    k.w_m = a.w_m;
    k.f_samp = a.f_samp;
    k.inv_fs = 1.0 / a.f_samp;
#pragma unroll
    for (int i = 0; i < 5; ++i) k.q[i] = a.q[i];
    if (a.state) {
        const double* carried = a.state + c * kEkfStateStride;
#pragma unroll
        for (int i = 0; i < 5; ++i) s.x[i] = carried[i];
#pragma unroll
        for (int i = 0; i < 15; ++i) s.P[i] = carried[5 + i];
        k.r = carried[30];
    } else {
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
}

// The filter over samples [t_lo, t_hi) of a window (t_lo a multiple of kEkfTile, s the state at t_lo with no pending
// update, kd = k0 + t_lo), tile by tile exactly as ekf_kernel runs it: cp.async staging kEkfStages tiles ahead into
// the thread's own columns of stage, the fast step on a whole tile, and a replay of the tile from its saved entry
// state with the checked step if any argument left the fast range.
//   on_entry(t0, s):  at each tile entry, s flushed;
//   on_step(t, s):    after the step with sample t (s's pending update not applied);
//   on_snap(sn, s):   after sample t with (t + 1) % R == 0, sn = (t + 1) / R - 1 (us: samples to the next one).
// A replayed tile repeats its on_step and on_snap calls, so outputs they write end up as the replay's.
template <class OnEntry, class OnStep, class OnSnap>
DFK_D void smooth_filter(double (*stage)[kEkfTile][32], double (*saved)[32], int lane, const double* zc, long long ld_t,
                         long long t_lo, long long t_hi, EkfState& s, const EkfConsts& k, double kd, long long R,
                         long long us, long long sn, OnEntry on_entry, OnStep on_step, OnSnap on_snap) {
    const long long ntiles = (t_hi - t_lo + kEkfTile - 1) / kEkfTile;
    auto issue = [&](long long tile) {
        if (tile < ntiles) {
            double* dst = &stage[tile % kEkfStages][0][lane];
            const long long t0 = t_lo + tile * kEkfTile;
            const int lim = (t_hi - t0 < kEkfTile) ? static_cast<int>(t_hi - t0) : kEkfTile;
            const double* src = zc + t0 * ld_t;
#pragma unroll 8
            for (int i = 0; i < lim; ++i) cp_async8(dst + i * 32, src + i * ld_t);
        }
        cp_async_commit();
    };
#pragma unroll
    for (int p = 0; p < kEkfStages - 1; ++p) issue(p);
    auto run_tile = [&](auto fast_tag, const double* src, long long t0, int lim, double& kdl, long long& usl,
                        long long& snl) -> bool {
        constexpr bool FAST = decltype(fast_tag)::value;
        bool ok = true;
        int pos = 0;
        while (pos < lim) {
            const int run = (usl < lim - pos) ? static_cast<int>(usl) : lim - pos;
            double A = carrier_angle(kdl, k);
#pragma unroll 1
            for (int i = 0; i < run; ++i) {
                kdl += 1.0;
                const double A_next = carrier_angle(kdl, k);
                ok &= ekf_step<FAST>(s, src[(pos + i) * 32], A, k);
                on_step(t0 + pos + i, s);
                A = A_next;
            }
            pos += run;
            usl -= run;
            if (usl == 0) {
                on_snap(snl, s);
                ++snl;
                usl = R;
            }
        }
        return ok;
    };
    double* sv = &saved[0][lane];
    for (long long tile = 0; tile < ntiles; ++tile) {
        issue(tile + kEkfStages - 1);
        cp_async_wait<kEkfStages - 1>();
        const double* src = &stage[tile % kEkfStages][0][lane];
        const long long t0 = t_lo + tile * kEkfTile;
        const int lim = (t_hi - t0 < kEkfTile) ? static_cast<int>(t_hi - t0) : kEkfTile;
        ekf_flush(s);
        on_entry(t0, s);
#pragma unroll
        for (int i = 0; i < 5; ++i) sv[i * 32] = s.x[i];
#pragma unroll
        for (int i = 0; i < 15; ++i) sv[(5 + i) * 32] = s.P[i];
        const double kd0 = kd;
        const long long us0 = us, sn0 = sn;
        if (!run_tile(std::true_type{}, src, t0, lim, kd, us, sn)) {
#pragma unroll
            for (int i = 0; i < 5; ++i) s.x[i] = sv[i * 32];
#pragma unroll
            for (int i = 0; i < 15; ++i) s.P[i] = sv[(5 + i) * 32];
#pragma unroll
            for (int i = 0; i < 5; ++i) s.kp[i] = s.hp[i] = 0.0;
            kd = kd0;
            us = us0;
            sn = sn0;
            run_tile(std::false_type{}, src, t0, lim, kd, us, sn);
        }
    }
}

// Forward pass: filtered rows and variances at the snapshots, a checkpoint at every block entry.
__global__ void __launch_bounds__(32) ekf_smooth_forward_kernel(const double* __restrict__ z, long long T, long long C,
                                                                long long ld_t, long long ld_c, long long R,
                                                                SmoothLaunch a, const double* __restrict__ stats) {
    __shared__ double stage[kEkfStages][kEkfTile][32];
    __shared__ double saved[20][32];
    const int lane = threadIdx.x;
    const long long c = blockIdx.x * static_cast<long long>(a.f.cpw) + lane;
    if (lane >= a.f.cpw || c >= C) return;
    EkfState s;
    EkfConsts k;
    smooth_init(a.f, stats, c, s, k);
    const long long nbuf = T / R;
    double* rows = a.filt_rows ? a.filt_rows + c * nbuf * 8 : nullptr;
    double* var = a.filt_var ? a.filt_var + c * nbuf * 5 : nullptr;
    const long long B = a.B;
    auto on_entry = [&](long long t0, const EkfState& st) {
        if (t0 % B == 0) {
            double* ck = a.ckpt + (t0 / B) * kSmoothDoubles * C + c;
#pragma unroll
            for (int i = 0; i < 5; ++i) ck[i * C] = st.x[i];
#pragma unroll
            for (int i = 0; i < 15; ++i) ck[(5 + i) * C] = st.P[i];
        }
    };
    auto on_step = [](long long, const EkfState&) {};
    auto on_snap = [&](long long sn, const EkfState& st) {
        if (sn >= nbuf) return;
        if (rows) {
            double* row = rows + sn * 8;
            row[0] = st.x[0]; row[1] = st.x[1]; row[2] = st.x[2]; row[3] = st.x[3]; row[4] = st.x[4];
            row[5] = 0.0; row[6] = 1.0; row[7] = 0.0;
        }
        if (var) {
            EkfState f = st;
            ekf_apply_pending(f);
            double* v = var + sn * 5;
            v[0] = f.P[0]; v[1] = f.P[5]; v[2] = f.P[9]; v[3] = f.P[12]; v[4] = f.P[14];
        }
    };
    smooth_filter(stage, saved, lane, z + c * ld_c, ld_t, 0, T, s, k, static_cast<double>(a.f.k0), R, R, 0, on_entry,
                  on_step, on_snap);
}

// Backward pass: per block, from last to first, the filter re-run from its checkpoint into the block store, then the
// recursion back through the block.
__global__ void __launch_bounds__(32) ekf_smooth_backward_kernel(const double* __restrict__ z, long long T, long long C,
                                                                 long long ld_t, long long ld_c, long long R,
                                                                 SmoothLaunch a, const double* __restrict__ stats) {
    __shared__ double stage[kEkfStages][kEkfTile][32];
    __shared__ double saved[20][32];
    const int lane = threadIdx.x;
    const long long c0 = blockIdx.x * static_cast<long long>(a.f.cpw);
    const long long c = c0 + lane;
    if (lane >= a.f.cpw || c >= C) return;
    const long long width = (C - c0 < a.f.cpw) ? C - c0 : a.f.cpw;
    double* store = a.store + c0 * a.B * kSmoothDoubles + lane;  // step i, entry j at store[(i * 20 + j) * width]
    EkfState s;
    EkfConsts k;
    smooth_init(a.f, stats, c, s, k);
    const long long nbuf = T / R;
    double* rows = a.rows + c * nbuf * 8;
    double* var = a.var ? a.var + c * nbuf * 5 : nullptr;
    const long long B = a.B;
    const long long nblk = (T + B - 1) / B;
    const double* zc = z + c * ld_c;
    double xs[5], Ps[15];
    auto on_entry = [](long long, const EkfState&) {};
    auto on_snap = [](long long, const EkfState&) {};
    for (long long blk = nblk - 1; blk >= 0; --blk) {
        const long long t_lo = blk * B, t_hi = (t_lo + B < T) ? t_lo + B : T;
        const double* ck = a.ckpt + blk * kSmoothDoubles * C + c;
#pragma unroll
        for (int i = 0; i < 5; ++i) s.x[i] = ck[i * C];
#pragma unroll
        for (int i = 0; i < 15; ++i) s.P[i] = ck[(5 + i) * C];
#pragma unroll
        for (int i = 0; i < 5; ++i) s.kp[i] = s.hp[i] = 0.0;
        auto on_step = [&](long long t, const EkfState& st) {
            EkfState f = st;
            ekf_apply_pending(f);
            double* dst = store + (t - t_lo) * kSmoothDoubles * width;
#pragma unroll
            for (int i = 0; i < 5; ++i) dst[i * width] = f.x[i];
#pragma unroll
            for (int i = 0; i < 15; ++i) dst[(5 + i) * width] = f.P[i];
        };
        // no snapshots in the replay: the countdown never reaches zero
        smooth_filter(stage, saved, lane, zc, ld_t, t_lo, t_hi, s, k, static_cast<double>(a.f.k0 + t_lo), R,
                      t_hi - t_lo + 1, 0, on_entry, on_step, on_snap);
        long long to_snap = t_hi % R;  // (t + 1) % R at t = t_hi - 1
#pragma unroll 1
        for (long long t = t_hi - 1; t >= t_lo; --t) {
            const double* src = store + (t - t_lo) * kSmoothDoubles * width;
            double xf[5], Pf[15];
#pragma unroll
            for (int i = 0; i < 5; ++i) xf[i] = src[i * width];
#pragma unroll
            for (int i = 0; i < 15; ++i) Pf[i] = src[(5 + i) * width];
            if (t == T - 1) {
#pragma unroll
                for (int i = 0; i < 5; ++i) xs[i] = xf[i];
#pragma unroll
                for (int i = 0; i < 15; ++i) Ps[i] = Pf[i];
            } else {
                rts_step(xf, Pf, k.q, xs, Ps);
            }
            if (to_snap == 0) {
                const long long b = (t + 1) / R - 1;
                double* row = rows + b * 8;
                row[0] = xs[0]; row[1] = xs[1]; row[2] = xs[2]; row[3] = xs[3]; row[4] = xs[4];
                row[5] = 0.0; row[6] = 1.0; row[7] = 0.0;
                if (var) {
                    double* v = var + b * 5;
                    v[0] = Ps[0]; v[1] = Ps[5]; v[2] = Ps[9]; v[3] = Ps[12]; v[4] = Ps[14];
                }
                to_snap = R;
            }
            --to_snap;
        }
    }
}

}  // namespace dfk
#endif  // __CUDACC__
