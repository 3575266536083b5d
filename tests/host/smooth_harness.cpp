// Host build of the EKF smoother's core (ekf_step + rts_step, dfk_ekf_smooth.cuh), for the CPU-side smoother tests.
// The driver mirrors the device passes: the filter forward with a checkpoint every B samples, then per block, from last
// to first, a replay from the checkpoint into a block store and the recursion back through the block.
#include <cstdint>
#include <cstring>
#include <vector>

#include "../../deepfmkit_b200/csrc/dfk_ekf_smooth.cuh"

using namespace dfk;

extern "C" {

// One channel's window of T samples from absolute sample k0, prior x0[5] and P0 (upper triangle, tri order), noise
// q[5] and r.  At snapshot b (sample (b+1) R - 1): xs/vs = smoothed state / variances, xf/vf = filtered ones, [nbuf][5].
void sh_smooth(const double* z, int64_t T, int64_t R, int64_t k0, double f_samp, double f_mod, const double* x0,
               const double* P0, const double* q, double r, int64_t B, double* xs_out, double* vs_out, double* xf_out,
               double* vf_out) {
    EkfConsts c;
    c.w_m = 2 * kPi * f_mod;
    c.f_samp = f_samp;
    c.inv_fs = 1.0 / f_samp;
    for (int i = 0; i < 5; ++i) c.q[i] = q[i];
    c.r = r;
    EkfState s;
    std::memcpy(s.x, x0, sizeof(s.x));
    std::memcpy(s.P, P0, sizeof(s.P));
    for (int i = 0; i < 5; ++i) s.kp[i] = s.hp[i] = 0.0;
    const int64_t nblk = (T + B - 1) / B;
    std::vector<double> ckpt(nblk * kSmoothDoubles), store(B * kSmoothDoubles);
    for (int64_t t = 0; t < T; ++t) {
        if (t % B == 0) {
            ekf_flush(s);
            std::memcpy(&ckpt[(t / B) * kSmoothDoubles], s.x, 5 * sizeof(double));
            std::memcpy(&ckpt[(t / B) * kSmoothDoubles + 5], s.P, 15 * sizeof(double));
        }
        ekf_step<false>(s, z[t], carrier_angle(static_cast<double>(k0 + t), c), c);
        if ((t + 1) % R == 0) {
            EkfState f = s;
            ekf_apply_pending(f);
            const int64_t b = (t + 1) / R - 1;
            for (int i = 0; i < 5; ++i) {
                xf_out[b * 5 + i] = f.x[i];
                vf_out[b * 5 + i] = f.P[tri(i, i)];
            }
        }
    }
    double xs[5], Ps[15];
    for (int64_t blk = nblk - 1; blk >= 0; --blk) {
        const int64_t lo = blk * B, hi = lo + B < T ? lo + B : T;
        std::memcpy(s.x, &ckpt[blk * kSmoothDoubles], 5 * sizeof(double));
        std::memcpy(s.P, &ckpt[blk * kSmoothDoubles + 5], 15 * sizeof(double));
        for (int i = 0; i < 5; ++i) s.kp[i] = s.hp[i] = 0.0;
        for (int64_t t = lo; t < hi; ++t) {
            ekf_step<false>(s, z[t], carrier_angle(static_cast<double>(k0 + t), c), c);
            EkfState f = s;
            ekf_apply_pending(f);
            std::memcpy(&store[(t - lo) * kSmoothDoubles], f.x, 5 * sizeof(double));
            std::memcpy(&store[(t - lo) * kSmoothDoubles + 5], f.P, 15 * sizeof(double));
        }
        for (int64_t t = hi - 1; t >= lo; --t) {
            const double* xf = &store[(t - lo) * kSmoothDoubles];
            if (t == T - 1) {
                std::memcpy(xs, xf, 5 * sizeof(double));
                std::memcpy(Ps, xf + 5, 15 * sizeof(double));
            } else {
                rts_step(xf, xf + 5, c.q, xs, Ps);
            }
            if ((t + 1) % R == 0) {
                const int64_t b = (t + 1) / R - 1;
                for (int i = 0; i < 5; ++i) {
                    xs_out[b * 5 + i] = xs[i];
                    vs_out[b * 5 + i] = Ps[tri(i, i)];
                }
            }
        }
    }
}

}  // extern "C"
