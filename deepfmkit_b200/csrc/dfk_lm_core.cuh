// Levenberg-Marquardt core for the 4-parameter DFMI harmonic model, G lanes cooperating per fit.
//
// Follows the reference solver fit.py:68-362 step for step (same damping ladder, same
// first-improvement acceptance, same stopping rule, same fallback and normalisation); only the
// evaluation strategy is different: harmonics are strided over the G lanes of a group, Bessel
// values come from a Miller recurrence kept in a per-lane column, cos/sin(j*psi) come from a
// rotation recurrence, and the damped 4x4 system is solved in registers by Gaussian elimination
// with partial pivoting (what np.linalg.solve/LAPACK gesv does, including "exactly singular ->
// no step", fit.py:197-204) on the block structure the model's Jacobian has (see NormalEq).
#pragma once
#include "dfk_bessel.cuh"
#include "dfk_common.cuh"

namespace dfk {

// ---- cooperation of G lanes (G = 1 on the host build) ---------------------------------------
template <int G>
struct Coop {
    static DFK_HD int rank() {
#if defined(__CUDA_ARCH__)
        return static_cast<int>(threadIdx.x) & (G - 1);
#else
        return 0;
#endif
    }
    static DFK_HD unsigned mask() {
#if defined(__CUDA_ARCH__)
        if (G == 32) return 0xffffffffu;
        const unsigned lane = threadIdx.x & 31u;
        return static_cast<unsigned>((1ull << G) - 1ull) << (lane & ~static_cast<unsigned>(G - 1));
#else
        return 1u;
#endif
    }
    static DFK_HD double sum(double v) {
#if defined(__CUDA_ARCH__)
        if (G > 1) {
            const unsigned m = mask();
#pragma unroll
            for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(m, v, o);
        }
#endif
        return v;
    }
    static DFK_HD double bcast(double v, int src_rank) {
#if defined(__CUDA_ARCH__)
        if (G > 1) v = __shfl_sync(mask(), v, src_rank, G);
#endif
        (void)src_rank;
        return v;
    }
    // (value, index) argmin with "first index wins" on ties, like a sequential strict-< scan.
    static DFK_HD void argmin(double& v, int& idx) {
#if defined(__CUDA_ARCH__)
        if (G > 1) {
            const unsigned m = mask();
#pragma unroll
            for (int o = G / 2; o > 0; o >>= 1) {
                const double ov = __shfl_xor_sync(m, v, o);
                const int oi = __shfl_xor_sync(m, idx, o);
                const bool take = (oi >= 0) && (idx < 0 || ov < v || (ov == v && oi < idx));
                if (take) {
                    v = ov;
                    idx = oi;
                }
            }
        }
#endif
    }
};

// ---- normal equations ------------------------------------------------------------------------
// The model's two rows of harmonic j are  a q_j J_j(m) (cos j psi, -sin j psi)  with q_j = cos(phi + j pi/2).
// Rotating the data pair (Q_j, I_j) by j psi instead of the model,
//     u_j = c Q_j - s I_j,   v_j = s Q_j + c I_j      (c, s = cos, sin of j psi),
// the residual pair becomes (u_j - env_j, v_j) with env_j = a q_j J_j, the amplitude / depth / phase columns
// of the Jacobian (fit.py:125-140) all point along the first rotated axis and the psi column (fit.py:143-144)
// along the second.  J^T J is therefore block diagonal -- a 3x3 block and the scalar psi-psi entry; the
// reference's fourth row/column holds only its rounding noise (~1e-17 of the diagonal) -- and J^T r needs one
// product per column.  Same numbers as fit.py:68-150 to rounding, about half the arithmetic.
struct NormalEq {
    double ssq;
    double a00, a01, a02, a11, a12, a22;  // amplitude, depth, phase block of J^T J (upper triangle)
    double a33;                           // psi-psi entry
    double g0, g1, g2, g3;                // J^T r
};

// quarter-turn factors: cos(phi + j*pi/2) and its phi-derivative cos(phi + j*pi/2 + pi/2) (fit.py:100,137)
DFK_HD void quarter_terms(int j, double cphi, double sphi, double& q, double& dq) {
    switch (j & 3) {
        case 0: q = cphi; dq = -sphi; break;
        case 1: q = -sphi; dq = -cphi; break;
        case 2: q = -cphi; dq = sphi; break;
        default: q = sphi; dq = cphi; break;
    }
}

// (q, dq) at harmonic j -> harmonic j + G (G a power of two)
template <int G>
DFK_HD void quarter_advance(double& q, double& dq) {
    if (G == 1) {
        const double t = q;
        q = dq;
        dq = -t;
    } else if (G == 2) {
        q = -q;
        dq = -dq;
    }
}

// Sum of squares, J^T J and J^T r at p (fit.py:68-150).  qi[k*qs]: harmonic vector of this fit;
// bes[k*bs]: this lane's column holding J_0..J_{N+1}(p[1]).
template <int G>
DFK_HD void eval_state(int N, const double* qi, int qs, const double* bes, int bs, const double* p, NormalEq& ne) {
    const double a = p[0], phi = p[2], psi = p[3];
    double sphi, cphi;
    sincos_hd(phi, &sphi, &cphi);
    const int r = Coop<G>::rank();
    double s, c, sg, cg;
    sincos_hd(static_cast<double>(r + 1) * psi, &s, &c);
    if (G == 1) {
        sg = s;
        cg = c;
    } else {
        sincos_hd(static_cast<double>(G) * psi, &sg, &cg);
    }
    double q, dq;
    quarter_terms(r + 1, cphi, sphi, q, dq);
    NormalEq t = {};
    const double a_on = (a != 0.0) ? 1.0 : 0.0;  // fit.py:126: amplitude column stays zero at a == 0
    double fj = static_cast<double>(r + 1);
    const double* qq = qi + r * qs;
    const double* qv = qi + (N + r) * qs;
    const double* bb = bes + (r + 1) * bs;
    double b_lo = bes[r * bs];  // J_{j-1}
    for (int j = r + 1; j <= N; j += G) {
        const double B = bb[0];
        const double b_hi = bb[bs];
        const double dB = 0.5 * (b_lo - b_hi);  // fit.py:108
        const double Qj = qq[0], Ij = qv[0];
        const double u = c * Qj - s * Ij;  // data rotated by j*psi
        const double v = s * Qj + c * Ij;
        const double shape = q * B;
        const double env = a * shape;  // fit.py:111
        const double e = u - env;
        const double x0 = a_on * shape, x1 = (a * q) * dB, x2 = (a * dq) * B, x3 = -(env * fj);
        t.ssq += e * e + v * v;
        t.a00 += x0 * x0;
        t.a01 += x0 * x1;
        t.a02 += x0 * x2;
        t.a11 += x1 * x1;
        t.a12 += x1 * x2;
        t.a22 += x2 * x2;
        t.a33 += x3 * x3;
        t.g0 += x0 * e;
        t.g1 += x1 * e;
        t.g2 += x2 * e;
        t.g3 += x3 * v;
        const double cn = c * cg - s * sg;  // advance cos/sin(j*psi) by G harmonics
        s = s * cg + c * sg;
        c = cn;
        quarter_advance<G>(q, dq);
        fj += static_cast<double>(G);
        qq += G * qs;
        qv += G * qs;
        if (G == 1) {
            b_lo = B;
        } else if (j + G <= N) {
            b_lo = bb[(G - 1) * bs];  // J_{j+G-1}; past the last harmonic the column ends
        }
        bb += G * bs;
    }
    ne.ssq = Coop<G>::sum(t.ssq);
    ne.a00 = Coop<G>::sum(t.a00); ne.a01 = Coop<G>::sum(t.a01); ne.a02 = Coop<G>::sum(t.a02);
    ne.a11 = Coop<G>::sum(t.a11); ne.a12 = Coop<G>::sum(t.a12); ne.a22 = Coop<G>::sum(t.a22);
    ne.a33 = Coop<G>::sum(t.a33);
    ne.g0 = Coop<G>::sum(t.g0); ne.g1 = Coop<G>::sum(t.g1); ne.g2 = Coop<G>::sum(t.g2);
    ne.g3 = Coop<G>::sum(t.g3);
}

// Residual sum of squares only (fit.py:152-167).
template <int G>
DFK_HD double eval_ssq(int N, const double* qi, int qs, const double* bes, int bs, const double* p) {
    const double a = p[0], phi = p[2], psi = p[3];
    double sphi, cphi;
    sincos_hd(phi, &sphi, &cphi);
    const int r = Coop<G>::rank();
    double s, c, sg, cg;
    sincos_hd(static_cast<double>(r + 1) * psi, &s, &c);
    if (G == 1) {
        sg = s;
        cg = c;
    } else {
        sincos_hd(static_cast<double>(G) * psi, &sg, &cg);
    }
    double q, dq;
    quarter_terms(r + 1, cphi, sphi, q, dq);
    double aq = a * q, adq = a * dq;  // a * cos(phi + j*pi/2) and the next quarter turn
    double acc = 0.0;
    const double* qq = qi + r * qs;
    const double* qv = qi + (N + r) * qs;
    const double* bb = bes + (r + 1) * bs;
    for (int j = r + 1; j <= N; j += G) {
        const double Qj = qq[0], Ij = qv[0];
        const double e = (c * Qj - s * Ij) - aq * bb[0];
        const double v = s * Qj + c * Ij;
        acc += e * e + v * v;
        const double cn = c * cg - s * sg;
        s = s * cg + c * sg;
        c = cn;
        quarter_advance<G>(aq, adq);
        qq += G * qs;
        qv += G * qs;
        bb += G * bs;
    }
    return Coop<G>::sum(acc);
}

// (J^T J + lam diag(J^T J)) dp = g (fit.py:169-206): elimination with partial pivoting on the 3x3 block, a
// division for psi.  Returns false (dp = 0) when a pivot is exactly zero -- numpy's LinAlgError branch.
DFK_HD bool damped_solve(const NormalEq& ne, double lam, double* dp) {
    double A[3][4] = {{ne.a00 + lam * ne.a00, ne.a01, ne.a02, ne.g0},
                      {ne.a01, ne.a11 + lam * ne.a11, ne.a12, ne.g1},
                      {ne.a02, ne.a12, ne.a22 + lam * ne.a22, ne.g2}};
    const double d33 = ne.a33 + lam * ne.a33;
    bool ok = d33 != 0.0;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        int piv = c;
        double best = fabs(A[c][c]);
#pragma unroll
        for (int r = c + 1; r < 3; ++r) {
            const double v = fabs(A[r][c]);
            if (v > best) {
                best = v;
                piv = r;
            }
        }
        if (!(best > 0.0)) ok = false;
#pragma unroll
        for (int r = c + 1; r < 3; ++r) {
            if (piv == r) {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const double tmp = A[c][k];
                    A[c][k] = A[r][k];
                    A[r][k] = tmp;
                }
            }
        }
        const double inv = 1.0 / A[c][c];
#pragma unroll
        for (int r = c + 1; r < 3; ++r) {
            const double f = A[r][c] * inv;
#pragma unroll
            for (int k = c + 1; k < 4; ++k) A[r][k] -= f * A[c][k];
        }
    }
    if (!ok) {
        dp[0] = dp[1] = dp[2] = dp[3] = 0.0;
        return false;
    }
    const double x2 = A[2][3] / A[2][2];
    const double x1 = (A[1][3] - A[1][2] * x2) / A[1][1];
    const double x0 = (A[0][3] - A[0][1] * x1 - A[0][2] * x2) / A[0][0];
    dp[0] = x0; dp[1] = x1; dp[2] = x2; dp[3] = ne.g3 / d33;
    return true;
}

DFK_HD double lambda_of(int i) {  // fit.py:222
    switch (i) {
        case 0: return 0.0;
        case 1: return 1e-7;
        case 2: return 1e-5;
        case 3: return 1e-3;
        case 4: return 1e-1;
        case 5: return 1.0;
        case 6: return 10.0;
        default: return 100.0;
    }
}

// LM loop (fit.py:208-258).  p is updated in place; returns the final ssq and the number of accepted steps.
template <int G>
DFK_HD double lm_descend(int N, const double* qi, int qs, double* bes, int bs, const LmOpts& o, double* p,
                         int& accepted_steps, LmCounts& cnt) {
    NormalEq ne;
    cnt.n_bessel_steps += bessel_j_upto(p[1], N + 1, bes, bs);
    // m the Bessel column currently holds: near convergence the steps of neighbouring dampings differ by less than
    // an ulp of m, the trial m is then bit-identical and the column (a pure function of m) need not be rebuilt
    double m_held = p[1];
    eval_state<G>(N, qi, qs, bes, bs, p, ne);
    cnt.n_state++;
    double ssq = ne.ssq;
    accepted_steps = 0;
    for (int it = 0; it < o.max_steps; ++it) {
        double best_ssq = ssq;
        double pb[4] = {p[0], p[1], p[2], p[3]};
        bool improved = false;
        for (int l = 0; l < 8; ++l) {
            double dp[4];
            damped_solve(ne, lambda_of(l), dp);
            cnt.n_solve++;
            const double nrm = sqrt(dp[0] * dp[0] + dp[1] * dp[1] + dp[2] * dp[2] + dp[3] * dp[3]);
            if (nrm < 1e-15) continue;  // fit.py:230
            const double pt[4] = {p[0] + dp[0], p[1] + dp[1], p[2] + dp[2], p[3] + dp[3]};
            if (pt[1] != m_held) {
                cnt.n_bessel_steps += bessel_j_upto(pt[1], N + 1, bes, bs);
                m_held = pt[1];
            }
            const double st = eval_ssq<G>(N, qi, qs, bes, bs, pt);
            cnt.n_ssq++;
            if (st < best_ssq) {  // first strictly better damping wins (fit.py:240-243)
                best_ssq = st;
                pb[0] = pt[0]; pb[1] = pt[1]; pb[2] = pt[2]; pb[3] = pt[3];
                improved = true;
                break;
            }
        }
        if (!improved) break;  // fit.py:246
        const double d0 = pb[0] - p[0], d1 = pb[1] - p[1], d2 = pb[2] - p[2], d3 = pb[3] - p[3];
        p[0] = pb[0]; p[1] = pb[1]; p[2] = pb[2]; p[3] = pb[3];
        // the Bessel column still holds J_k(p[1]) from the accepted trial
        eval_state<G>(N, qi, qs, bes, bs, p, ne);
        cnt.n_state++;
        ssq = ne.ssq;
        ++accepted_steps;
        const double moved = sqrt(d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3);
        if ((ssq - best_ssq) < o.conv_improve && moved < o.conv_param) break;  // fit.py:255
    }
    return ssq;
}

// Number of m values np.arange(min, max + step, step) produces (fit.py:270).
DFK_HD int grid_points(const LmOpts& o) {
    const double n = ceil((o.grid_max + o.grid_step - o.grid_min) / o.grid_step);
    if (!(n > 0.0)) return 0;
    return n > 100000.0 ? 100000 : static_cast<int>(n);
}

// Fallback initialiser (fit.py:260-320): lanes of the group take m candidates round robin; each
// evaluates its candidates alone (G = 1 arithmetic on its own Bessel column), then the group picks
// the first minimum.  seed = 0 when no candidate qualified.
template <int G>
DFK_HD void grid_seed(int N, const double* qi, int qs, double* bes, int bs, const LmOpts& o, double* seed,
                      LmCounts& cnt) {
    const int npts = grid_points(o);
    double best_ssq = 9e99;
    int best_idx = -1;
    double best_a = 0.0, best_phi = 0.0;
    for (int i = Coop<G>::rank(); i < npts; i += G) {
        const double m_try = o.grid_min + static_cast<double>(i) * o.grid_step;
        cnt.n_bessel_steps += bessel_j_upto(m_try, N + 1, bes, bs);
        double s_sum = 0.0, c_sum = 0.0;
        int n_s = 0, n_c = 0;
        for (int j = 1; j <= N; ++j) {
            const double w = bes[j * bs];  // * cos(j*0); the sine-half weight is -J*sin(0) = 0 and never qualifies
            if (fabs(w) > o.bessel_thr) {
                const double r = qi[(j - 1) * qs] / w;
                switch (j & 3) {
                    case 0: c_sum += r; ++n_c; break;
                    case 1: s_sum -= r; ++n_s; break;
                    case 2: c_sum -= r; ++n_c; break;
                    default: s_sum += r; ++n_s; break;
                }
            }
        }
        if (n_s == 0 || n_c == 0) continue;
        const double phi_try = atan2(s_sum / n_s, c_sum / n_c);
        double sp, cp;
        sincos_hd(phi_try, &sp, &cp);
        double a_sum = 0.0;
        int n_a = 0;
        for (int j = 1; j <= N; ++j) {
            const double w = bes[j * bs];
            double f;
            switch (j & 3) {
                case 0: f = cp; break;
                case 1: f = -sp; break;
                case 2: f = -cp; break;
                default: f = sp; break;
            }
            if (fabs(w) > o.bessel_thr && fabs(f) > o.sincos_thr) {
                a_sum += qi[(j - 1) * qs] / (f * w);
                ++n_a;
            }
        }
        if (n_a == 0) continue;
        const double cand[4] = {a_sum / n_a, m_try, phi_try, 0.0};
        const double cs = eval_ssq<1>(N, qi, qs, bes, bs, cand);
        cnt.n_ssq++;
        if (cs < best_ssq) {
            best_ssq = cs;
            best_idx = i;
            best_a = cand[0];
            best_phi = phi_try;
        }
    }
    Coop<G>::argmin(best_ssq, best_idx);
    if (best_idx < 0) {
        seed[0] = seed[1] = seed[2] = seed[3] = 0.0;
        return;
    }
    const int owner = best_idx % G;
    seed[0] = Coop<G>::bcast(best_a, owner);
    seed[1] = o.grid_min + static_cast<double>(best_idx) * o.grid_step;
    seed[2] = Coop<G>::bcast(best_phi, owner);
    seed[3] = 0.0;
}

// Sign normalisation and phase wrap (fit.py:351-360); psi is left unwrapped.
DFK_HD void normalise_params(double* p) {
    if (p[0] < 0.0) {
        p[0] = -p[0];
        p[2] += kPi;
    }
    if (p[1] < 0.0) {
        p[1] = -p[1];
        p[2] += kPi;
    }
    // (phi + pi) % (2 pi) - pi with Python's sign convention.  fmod is exact, and so are the two shortcuts: for
    // t in [2 pi, 4 pi) the difference t - 2 pi is exact (Sterbenz), and for t in [-2 pi, 0) Python's own result
    // is fmod's (t itself) plus 2 pi, rounded once.
    const double t = p[2] + kPi;
    double r;
    if (t >= 0.0 && t < kTwoPi) {
        r = t;
    } else if (t >= kTwoPi && t < 2.0 * kTwoPi) {
        r = t - kTwoPi;
    } else if (t < 0.0 && t > -kTwoPi) {
        r = t + kTwoPi;
    } else {
        r = fmod(t, kTwoPi);
        if (r != 0.0) {
            if (r < 0.0) r += kTwoPi;
        } else {
            r = 0.0;
        }
    }
    p[2] = r - kPi;
}

// Covariance of a fit's reported parameters: the standard NLS estimate s^2 (J^T J)^-1 with s^2 = ssq / (2N - 4), J^T J
// evaluated at the row's own (normalised, wrapped) parameters -- the model is invariant under that normalisation.
// The reference computes the same inv(J^T J) sigma^2 only at the true parameters, for its Cramer-Rao bound
// (helpers.py:16-45, 60-96).  J^T J is block diagonal (see NormalEq), so the result is one 3x3 inverse -- elimination
// with partial pivoting on unit right-hand sides, as damped_solve at lambda = 0 -- and a division for psi; the psi
// cross terms are identically zero and not stored.
//   row: [a, m, phi, psi, dc, ssq, ...];  bes[k*bs]: scratch column of N + 2 doubles (J_0..J_{N+1}(m) on return)
//   cov: [C_aa, C_am, C_aphi, C_mm, C_mphi, C_phiphi, C_psipsi, s^2]  (kCovStride doubles)
// Degenerate cases:
//   2N - 4 <= 0, or a non-finite a, m, phi or psi: all eight entries NaN;
//   a zero pivot in the 3x3 block (e.g. a = 0: the amplitude column vanishes, fit.py:126): the six block entries NaN;
//   a33 = 0: C_psipsi NaN;
//   ssq = 0 (noise-free input): the finite entries are zeros.
// Computed whatever the row's fitok; callers filter on fitok as they do for the parameters.
constexpr int kCovStride = 8;

DFK_HD void fit_covariance(int N, const double* qi, int qs, double* bes, int bs, const double* row, double* cov) {
    const double nan = std::nan("");
    const int dof = 2 * N - 4;
    const double p[4] = {row[0], row[1], row[2], row[3]};
    if (dof <= 0 || !std::isfinite(p[0]) || !std::isfinite(p[1]) || !std::isfinite(p[2]) || !std::isfinite(p[3])) {
        for (int k = 0; k < kCovStride; ++k) cov[k] = nan;
        return;
    }
    const double s2 = row[5] / static_cast<double>(dof);
    bessel_j_upto(p[1], N + 1, bes, bs);
    NormalEq ne;
    eval_state<1>(N, qi, qs, bes, bs, p, ne);
    // [A | I] -> [U | L^-1 P]
    double A[3][6] = {{ne.a00, ne.a01, ne.a02, 1.0, 0.0, 0.0},
                      {ne.a01, ne.a11, ne.a12, 0.0, 1.0, 0.0},
                      {ne.a02, ne.a12, ne.a22, 0.0, 0.0, 1.0}};
    bool ok = true;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        int piv = c;
        double best = fabs(A[c][c]);
#pragma unroll
        for (int r = c + 1; r < 3; ++r) {
            const double v = fabs(A[r][c]);
            if (v > best) {
                best = v;
                piv = r;
            }
        }
        if (!(best > 0.0)) ok = false;
#pragma unroll
        for (int r = c + 1; r < 3; ++r) {
            if (piv == r) {
#pragma unroll
                for (int k = 0; k < 6; ++k) {
                    const double tmp = A[c][k];
                    A[c][k] = A[r][k];
                    A[r][k] = tmp;
                }
            }
        }
        const double inv = 1.0 / A[c][c];
#pragma unroll
        for (int r = c + 1; r < 3; ++r) {
            const double f = A[r][c] * inv;
#pragma unroll
            for (int k = c + 1; k < 6; ++k) A[r][k] -= f * A[c][k];
        }
    }
    // back substitution, one column of the inverse per right-hand side
    double X[3][3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        X[2][k] = A[2][3 + k] / A[2][2];
        X[1][k] = (A[1][3 + k] - A[1][2] * X[2][k]) / A[1][1];
        X[0][k] = (A[0][3 + k] - A[0][1] * X[1][k] - A[0][2] * X[2][k]) / A[0][0];
    }
    auto scaled = [s2](double x) { return s2 == 0.0 ? 0.0 : s2 * x; };  // no -0 for a noise-free record
    cov[0] = ok ? scaled(X[0][0]) : nan;
    cov[1] = ok ? scaled(X[0][1]) : nan;
    cov[2] = ok ? scaled(X[0][2]) : nan;
    cov[3] = ok ? scaled(X[1][1]) : nan;
    cov[4] = ok ? scaled(X[1][2]) : nan;
    cov[5] = ok ? scaled(X[2][2]) : nan;
    cov[6] = ne.a33 != 0.0 ? s2 / ne.a33 : nan;
    cov[7] = s2;
}

// Retry stage of fit.py:336-349 for a fit whose first descent ended at (p, ssq) >= threshold.
template <int G>
DFK_HD int retry_fit(int N, const double* qi, int qs, double* bes, int bs, const LmOpts& o, double* p, double& ssq,
                     int& steps, LmCounts& cnt) {
    double seed[4];
    grid_seed<G>(N, qi, qs, bes, bs, o, seed, cnt);
    cnt.n_grid++;
    if (seed[0] != 0.0 || seed[1] != 0.0 || seed[2] != 0.0 || seed[3] != 0.0) {  // np.any (NaN counts as true)
        int steps2 = 0;
        const double ssq2 = lm_descend<G>(N, qi, qs, bes, bs, o, seed, steps2, cnt);
        if (ssq2 < ssq) {
            ssq = ssq2;
            p[0] = seed[0]; p[1] = seed[1]; p[2] = seed[2]; p[3] = seed[3];
            steps = steps2;
        }
    }
    return ssq < o.fitok_threshold ? 1 : 2;
}

// One complete fit (fit.py:322-362) by a single group; used by the host build and the small-batch path.
template <int G>
DFK_HD int fit_full(int N, const double* qi, int qs, double* bes, int bs, const LmOpts& o, double* p, double& ssq,
                    int& steps, LmCounts& cnt) {
    ssq = lm_descend<G>(N, qi, qs, bes, bs, o, p, steps, cnt);
    int status = 0;
    if (!(ssq < o.fitok_threshold)) status = retry_fit<G>(N, qi, qs, bes, bs, o, p, ssq, steps, cnt);
    normalise_params(p);
    return status;
}

}  // namespace dfk
