// Lock-in demodulation kernels (sm_100a).
//
// Reference computation (fit.py:55-64 + fitters.py:45-49,57): per buffer of R samples,
//   Q_k = mean(x[t] * cos(fl((k)*w0)*t)),  I_k = mean(x[t] * sin(fl(k*w0)*t)),  k = 1..N,  dc = mean(x),
// with t restarting at 0 in every buffer.
//
// The kernels, chosen by the launcher in dfk_b200.cu from the geometry (dfk_demod_plan.h):
//
// demod_fold_kernel   -- long fold lengths (P > 256, e.g. 1 MHz / 1 kHz).  Needs a whole even number P of samples
//   that holds whole modulation periods, and whole folds per buffer.  A persistent CTA streams its buffers from
//   HBM with 1-D TMA bulk copies (cp.async.bulk, one elected producer lane, mbarrier ring) and folds the periods
//   onto one: S_j = sum_c x[j + cP] -- one DADD per 8 bytes (plus one DFMA for the optional drift sum).  The N
//   harmonics are then taken from the folded period with the j <-> P-j symmetry (cos(k th_j) even, sin(k th_j)
//   odd) by a rotation recurrence per lane and a warp-shuffle reduction.
// demod_tile_kernel   -- short fold lengths (P <= 256): no CTA-wide synchronisation, a warp owns its group of
//   buffers from the TMA stage to the outputs, harmonics by a product with a twiddle table in shared memory.
// demod_period_kernel -- one period per buffer (R = P, P % 4 == 0): the tile scheme with quarter-wave symmetry and
//   a 2 x 4 register tile per lane, because at this shape the product, not HBM, is the bound.
// demod_fold_long_kernel -- fold lengths beyond 2048 samples in column chunks; in STORE mode the folded period of an
//   interleaved (time-major) multi-channel buffer for project_interleaved_kernel.
// demod_direct_kernel / demod_direct_pair_kernel -- anything else (incommensurate period, unaligned pointer, strided
//   channels): a warp per buffer (or 16 384-sample chunk of a long one; two per warp when there are enough), cos/sin
//   of the lane-independent part of the angle from a shared-memory table, two FMAs per sample and harmonic; 8 to 16
//   harmonics per pass, further passes re-read the record; direct_combine_kernel adds the chunks up.
//
// In the TMA kernels every sample is read from HBM exactly once: 8 B/sample + 8(2N+1) B/buffer written.
#pragma once
#include "dfk_common.cuh"
#include "dfk_demod_plan.h"

namespace dfk {

constexpr int kFoldConsumerWarps = 8;
constexpr int kFoldConsumers = kFoldConsumerWarps * 32;  // 256
constexpr int kFoldThreads = kFoldConsumers + 32;        // + producer warp
constexpr int kFoldStageBytes = 16384;

struct FoldParams {
    const double* x;
    double* qi;
    double* dc;
    long long nbuf;
    long long bpc;   // buffers per channel record
    long long ld_c;  // samples between the starts of consecutive channel records
    int R, P, periods, N;
    int kmul;     // modulation periods per fold length P (harmonic k of f_mod = harmonic kmul*k of the fold)
    int pps;      // periods per pipeline stage
    int nstages;  // ring depth
    double delta[kMaxHarmonics];
};

// shared-memory carve-up, identical on host (size) and device (pointers)
struct FoldSmem {
    int stage_doubles;  // pps * P
    size_t off_stage, off_s, off_u, off_cmb, off_tw, off_step, off_bar, total;
};

inline __host__ __device__ FoldSmem fold_smem_layout(int P, int pps, int nstages, int N, bool drift) {
    FoldSmem L;
    L.stage_doubles = pps * P;
    size_t o = 0;
    L.off_stage = o;
    o += static_cast<size_t>(nstages) * L.stage_doubles * 8;
    L.off_s = o;
    o += static_cast<size_t>(P) * 8;
    L.off_u = o;
    o += drift ? static_cast<size_t>(P) * 8 : 0;
    o = (o + 15) & ~static_cast<size_t>(15);
    L.off_cmb = o;
    o += static_cast<size_t>(P / 2 + 1) * (drift ? 32 : 16);
    L.off_tw = o;
    o += static_cast<size_t>(N + 1) * 32 * 16;
    L.off_step = o;
    o += static_cast<size_t>(N + 1) * 16;
    L.off_bar = o;
    o += static_cast<size_t>(2 * nstages) * 8;
    L.total = o;
    return L;
}

DFK_D void consumer_bar() { asm volatile("bar.sync 1, %0;" ::"n"(kFoldConsumers) : "memory"); }

DFK_D void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_addr(bar)) : "memory");
}

// SLOTS = ceil(P / 2 / 256): column pairs per consumer thread (all but the last slot are full for every thread)
template <bool DRIFT, int SLOTS>
__global__ void __launch_bounds__(kFoldThreads, 2) demod_fold_kernel(const FoldParams p) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const FoldSmem L = fold_smem_layout(p.P, p.pps, p.nstages, p.N, DRIFT);
    double* stage_base = reinterpret_cast<double*>(smem_raw + L.off_stage);
    double* sm_s = reinterpret_cast<double*>(smem_raw + L.off_s);
    double* sm_u = reinterpret_cast<double*>(smem_raw + L.off_u);
    double* sm_cmb = reinterpret_cast<double*>(smem_raw + L.off_cmb);
    double2* sm_tw = reinterpret_cast<double2*>(smem_raw + L.off_tw);
    double2* sm_step = reinterpret_cast<double2*>(smem_raw + L.off_step);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + L.off_bar);
    uint64_t* empty = full + p.nstages;

    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    const int P = p.P, N = p.N, half = P >> 1;
    const int chunks = (p.periods + p.pps - 1) / p.pps;

    if (tid == 0) {
        for (int s = 0; s < p.nstages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], kFoldConsumerWarps);
        }
        mbar_fence_init();
    }
    // twiddles: start value for (harmonic k, lane) and the 32-column step of harmonic k; the same
    // for every buffer because the lock-in phase restarts at each buffer.
    for (int i = tid; i < (N + 1) * 32; i += kFoldThreads) {
        const int k = i >> 5, l = i & 31;
        const long long r = (static_cast<long long>(k) * p.kmul * l) % P;
        double s, c;
        sincospi(2.0 * static_cast<double>(r) / static_cast<double>(P), &s, &c);
        sm_tw[i] = make_double2(c, s);
    }
    for (int k = tid; k <= N; k += kFoldThreads) {
        const long long r = (static_cast<long long>(k) * p.kmul * 32) % P;
        double s, c;
        sincospi(2.0 * static_cast<double>(r) / static_cast<double>(P), &s, &c);
        sm_step[k] = make_double2(c, s);
    }
    __syncthreads();

    if (warp == kFoldConsumerWarps) {
        // ---------------- producer: one lane feeds the ring -----------------------------------
        if (lane == 0) {
            const uint64_t pol = l2_evict_first_policy();
            int stage = 0;
            uint32_t phase = 0;
            for (long long b = blockIdx.x; b < p.nbuf; b += gridDim.x) {
                const double* src = p.x + (b / p.bpc) * p.ld_c + (b % p.bpc) * static_cast<long long>(p.R);
                for (int q = 0; q < chunks; ++q) {
                    const int np = min(p.pps, p.periods - q * p.pps);
                    const uint32_t bytes = static_cast<uint32_t>(np) * static_cast<uint32_t>(P) * 8u;
                    mbar_wait(&empty[stage], phase ^ 1u);
                    mbar_arrive_expect_tx(&full[stage], bytes);
                    bulk_load(stage_base + static_cast<size_t>(stage) * L.stage_doubles,
                              src + static_cast<size_t>(q) * p.pps * P, bytes, &full[stage], pol);
                    if (++stage == p.nstages) {
                        stage = 0;
                        phase ^= 1u;
                    }
                }
            }
        }
        return;
    }

    // ---------------- consumers: fold, then harmonics -----------------------------------------
    int stage = 0;
    uint32_t phase = 0;
    for (long long b = blockIdx.x; b < p.nbuf; b += gridDim.x) {
        double2 accS[SLOTS], accT[SLOTS];
#pragma unroll
        for (int s = 0; s < SLOTS; ++s) {
            accS[s] = make_double2(0.0, 0.0);
            accT[s] = make_double2(0.0, 0.0);
        }
        const bool last_ok = tid + (SLOTS - 1) * kFoldConsumers < half;
        for (int q = 0; q < chunks; ++q) {
            const int np = min(p.pps, p.periods - q * p.pps);
            mbar_wait(&full[stage], phase);
            const double2* row = reinterpret_cast<const double2*>(stage_base + static_cast<size_t>(stage) * L.stage_doubles) + tid;
            double cg = static_cast<double>(q * p.pps);
#pragma unroll 4
            for (int c = 0; c < np; ++c) {
#pragma unroll
                for (int s = 0; s < SLOTS; ++s) {
                    if (s < SLOTS - 1 || last_ok) {
                        const double2 v = row[s * kFoldConsumers];
                        accS[s].x += v.x;
                        accS[s].y += v.y;
                        if (DRIFT) {
                            accT[s].x = fma(cg, v.x, accT[s].x);
                            accT[s].y = fma(cg, v.y, accT[s].y);
                        }
                    }
                }
                row += half;
                if (DRIFT) cg += 1.0;
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[stage]);
            if (++stage == p.nstages) {
                stage = 0;
                phase ^= 1u;
            }
        }

        consumer_bar();  // everyone is done with the previous buffer's folded arrays
#pragma unroll
        for (int s = 0; s < SLOTS; ++s) {
            const int pair = tid + s * kFoldConsumers;
            if (pair < half) {
                reinterpret_cast<double2*>(sm_s)[pair] = accS[s];
                if (DRIFT) {
                    // U_j = sum_c (j + cP) x[j + cP] = j S_j + P T_j
                    const double j0 = static_cast<double>(2 * pair);
                    const double Pd = static_cast<double>(P);
                    reinterpret_cast<double2*>(sm_u)[pair] =
                        make_double2(fma(Pd, accT[s].x, j0 * accS[s].x), fma(Pd, accT[s].y, (j0 + 1.0) * accS[s].y));
                }
            }
        }
        consumer_bar();
        // symmetric / antisymmetric combinations over j <-> P - j  (j = 0 and j = P/2 pair with nothing)
        double2* cmb_s = reinterpret_cast<double2*>(sm_cmb);  // (A_j, B_j)   = (S_j + S_{P-j}, S_j - S_{P-j})
        double2* cmb_u = cmb_s + (half + 1);                  // (AU_j, BU_j) likewise from U
        for (int j = tid; j <= half; j += kFoldConsumers) {
            const bool self = (j == 0) || (j == half);
            const double sa = sm_s[j], sb = self ? 0.0 : sm_s[P - j];
            cmb_s[j] = make_double2(sa + sb, self ? 0.0 : sa - sb);
            if (DRIFT) {
                const double ua = sm_u[j], ub = self ? 0.0 : sm_u[P - j];
                cmb_u[j] = make_double2(ua + ub, self ? 0.0 : ua - ub);
            }
        }
        consumer_bar();

        // harmonic k (k = 0 is the mean) is owned by warp k % 8, two harmonics (k, k + 8) per pass so that
        // the folded period is read once for both; lanes stride the half period by 32 columns
        const double Rd = static_cast<double>(p.R);
        for (int k0 = warp; k0 <= N; k0 += 2 * kFoldConsumerWarps) {
            const int k1 = k0 + kFoldConsumerWarps;
            const bool two = k1 <= N;
            const double2 wa = sm_tw[k0 * 32 + lane], sta = sm_step[k0];
            const double2 wb = two ? sm_tw[k1 * 32 + lane] : make_double2(0.0, 0.0);
            const double2 stb = two ? sm_step[k1] : make_double2(1.0, 0.0);
            double ca = wa.x, sa = wa.y, cb = wb.x, sb = wb.y;
            double acc[2][4] = {{0.0, 0.0, 0.0, 0.0}, {0.0, 0.0, 0.0, 0.0}};  // Q, I, Q drift, I drift
            for (int j = lane; j <= half; j += 32) {
                const double2 ab = cmb_s[j];
                acc[0][0] = fma(ab.x, ca, acc[0][0]);
                acc[0][1] = fma(ab.y, sa, acc[0][1]);
                acc[1][0] = fma(ab.x, cb, acc[1][0]);
                acc[1][1] = fma(ab.y, sb, acc[1][1]);
                if (DRIFT) {
                    const double2 uab = cmb_u[j];
                    acc[0][2] = fma(uab.y, sa, acc[0][2]);
                    acc[0][3] = fma(uab.x, ca, acc[0][3]);
                    acc[1][2] = fma(uab.y, sb, acc[1][2]);
                    acc[1][3] = fma(uab.x, cb, acc[1][3]);
                }
                const double cna = ca * sta.x - sa * sta.y;
                sa = fma(sa, sta.x, ca * sta.y);
                ca = cna;
                const double cnb = cb * stb.x - sb * stb.y;
                sb = fma(sb, stb.x, cb * stb.y);
                cb = cnb;
            }
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int k = h == 0 ? k0 : k1;
                if (h == 1 && !two) break;
                double aq = warp_sum(acc[h][0]), ai = 0.0, aqu = 0.0, aiu = 0.0;
                if (k > 0) {
                    ai = warp_sum(acc[h][1]);
                    if (DRIFT) {
                        aqu = warp_sum(acc[h][2]);
                        aiu = warp_sum(acc[h][3]);
                    }
                }
                if (lane == 0) {
                    if (k == 0) {
                        p.dc[b] = aq / Rd;
                    } else {
                        double qv = aq, iv = ai;
                        if (DRIFT) {
                            const double d = p.delta[k - 1];
                            qv = fma(-d, aqu, qv);
                            iv = fma(d, aiu, iv);
                        }
                        double* out = p.qi + b * static_cast<long long>(2 * N);
                        out[k - 1] = qv / Rd;
                        out[N + k - 1] = iv / Rd;
                    }
                }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// demod_fold_long_kernel -- fold lengths beyond the register kernel's 2048 samples (e.g. 10 MHz / 1 kHz = 10 000).
// The period is cut into column chunks of kLongChunk samples.  For a chunk, the producer streams that chunk's slice
// of every period of the buffer (rows P samples apart in HBM, one bulk copy each), the consumers fold it in
// registers exactly as demod_fold_kernel does, park the folded slice in shared memory and project it on the
// harmonics -- warp k % 8 owns harmonics k and k + 8, lanes stride the slice by 32 columns with a rotation
// recurrence started from an exact sincospi per chunk -- accumulating over the chunks in registers.  No j <-> P - j
// pairing (the partners live in different chunks), so the projection covers the whole period: still a small
// fraction of the fold's time.  Every sample is read from HBM once: the same 8 B/sample roofline.
constexpr int kLongChunk = 4 * 2 * kFoldConsumers;  // 2048 columns: four column pairs per consumer thread
constexpr int kLongPasses = (kMaxHarmonics + 2 * kFoldConsumerWarps) / (2 * kFoldConsumerWarps);  // 5: harmonics 0..64, two per warp and pass

struct FoldLongSmem {
    int stage_doubles;  // pps * kLongChunk
    size_t off_stage, off_s, off_u, off_step, off_bar, total;
};

inline __host__ __device__ FoldLongSmem fold_long_smem_layout(int pps, int nstages, int N, bool drift) {
    FoldLongSmem L;
    L.stage_doubles = pps * kLongChunk;
    size_t o = 0;
    L.off_stage = o;
    o += static_cast<size_t>(nstages) * L.stage_doubles * 8;
    L.off_s = o;
    o += static_cast<size_t>(kLongChunk) * 8;
    L.off_u = o;
    o += drift ? static_cast<size_t>(kLongChunk) * 8 : 0;
    L.off_step = o;
    o += static_cast<size_t>(N + 1) * 16;
    L.off_bar = o;
    o += static_cast<size_t>(2 * nstages) * 8;
    L.total = o;
    return L;
}

// STORE: instead of projecting, the folded sums S (and, with DRIFT, T_g = sum_k k x[g + k P]) of every buffer are
// written out -- p.qi and p.dc then point at [nbuf][P] scratch arrays.  That is the first half of the lock-in of
// time-major records (fold_interleaved below): an interleaved [T][C] buffer folds like a single channel whose period is
// P C samples, and the per-channel harmonics are taken from the folded super-period by project_interleaved_kernel.
template <bool DRIFT, bool STORE = false>
__global__ void __launch_bounds__(kFoldThreads, 1) demod_fold_long_kernel(const FoldParams p) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const FoldLongSmem L = fold_long_smem_layout(p.pps, p.nstages, p.N, DRIFT);
    double* stage_base = reinterpret_cast<double*>(smem_raw + L.off_stage);
    double* sm_s = reinterpret_cast<double*>(smem_raw + L.off_s);
    double* sm_u = reinterpret_cast<double*>(smem_raw + L.off_u);
    double2* sm_step = reinterpret_cast<double2*>(smem_raw + L.off_step);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + L.off_bar);
    uint64_t* empty = full + p.nstages;
    constexpr int SLOTS = 4;

    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    const int P = p.P, N = p.N;
    const int nchunks = (P + kLongChunk - 1) / kLongChunk;
    const int stages_per_chunk = (p.periods + p.pps - 1) / p.pps;

    if (tid == 0) {
        for (int s = 0; s < p.nstages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], kFoldConsumerWarps);
        }
        mbar_fence_init();
    }
    for (int k = tid; k <= N; k += kFoldThreads) {  // 32-column step of harmonic k
        const long long r = (static_cast<long long>(k) * p.kmul * 32) % P;
        double s, c;
        sincospi(2.0 * static_cast<double>(r) / static_cast<double>(P), &s, &c);
        sm_step[k] = make_double2(c, s);
    }
    __syncthreads();

    if (warp == kFoldConsumerWarps) {
        if (lane == 0) {
            const uint64_t pol = l2_evict_first_policy();
            int stage = 0;
            uint32_t phase = 0;
            for (long long b = blockIdx.x; b < p.nbuf; b += gridDim.x) {
                const double* src = p.x + (b / p.bpc) * p.ld_c + (b % p.bpc) * static_cast<long long>(p.R);
                for (int w = 0; w < nchunks; ++w) {
                    const int wc = min(kLongChunk, P - w * kLongChunk);  // columns of this chunk (even)
                    for (int q = 0; q < stages_per_chunk; ++q) {
                        const int np = min(p.pps, p.periods - q * p.pps);
                        mbar_wait(&empty[stage], phase ^ 1u);
                        mbar_arrive_expect_tx(&full[stage], static_cast<uint32_t>(np) * static_cast<uint32_t>(wc) * 8u);
                        double* dst = stage_base + static_cast<size_t>(stage) * L.stage_doubles;
                        for (int c = 0; c < np; ++c)
                            bulk_load(dst + static_cast<size_t>(c) * wc,
                                      src + static_cast<size_t>(q * p.pps + c) * P + static_cast<size_t>(w) * kLongChunk,
                                      static_cast<uint32_t>(wc) * 8u, &full[stage], pol);
                        if (++stage == p.nstages) {
                            stage = 0;
                            phase ^= 1u;
                        }
                    }
                }
            }
        }
        return;
    }

    int stage = 0;
    uint32_t phase = 0;
    const double Rd = static_cast<double>(p.R);
    for (long long b = blockIdx.x; b < p.nbuf; b += gridDim.x) {
        // running harmonic sums of this warp's harmonics (up to four passes of two: N <= 64)
        double hacc[kLongPasses][2][4];
#pragma unroll
        for (int a = 0; a < kLongPasses; ++a)
#pragma unroll
            for (int h = 0; h < 2; ++h)
#pragma unroll
                for (int e = 0; e < 4; ++e) hacc[a][h][e] = 0.0;
        for (int w = 0; w < nchunks; ++w) {
            const int wc = min(kLongChunk, P - w * kLongChunk);
            const int whalf = wc >> 1;
            double2 accS[SLOTS], accT[SLOTS];
#pragma unroll
            for (int s = 0; s < SLOTS; ++s) {
                accS[s] = make_double2(0.0, 0.0);
                accT[s] = make_double2(0.0, 0.0);
            }
            for (int q = 0; q < stages_per_chunk; ++q) {
                const int np = min(p.pps, p.periods - q * p.pps);
                mbar_wait(&full[stage], phase);
                const double2* row = reinterpret_cast<const double2*>(stage_base + static_cast<size_t>(stage) * L.stage_doubles) + tid;
                double cg = static_cast<double>(q * p.pps);
                for (int c = 0; c < np; ++c) {
#pragma unroll
                    for (int s = 0; s < SLOTS; ++s) {
                        if (tid + s * kFoldConsumers < whalf) {
                            const double2 v = row[s * kFoldConsumers];
                            accS[s].x += v.x;
                            accS[s].y += v.y;
                            if (DRIFT) {
                                accT[s].x = fma(cg, v.x, accT[s].x);
                                accT[s].y = fma(cg, v.y, accT[s].y);
                            }
                        }
                    }
                    row += whalf;
                    if (DRIFT) cg += 1.0;
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty[stage]);
                if (++stage == p.nstages) {
                    stage = 0;
                    phase ^= 1u;
                }
            }
            if (STORE) {
                double2* fs = reinterpret_cast<double2*>(p.qi + b * static_cast<long long>(P) + static_cast<long long>(w) * kLongChunk);
                double2* ft = reinterpret_cast<double2*>(p.dc + b * static_cast<long long>(P) + static_cast<long long>(w) * kLongChunk);
#pragma unroll
                for (int s = 0; s < SLOTS; ++s) {
                    const int pair = tid + s * kFoldConsumers;
                    if (pair < whalf) {
                        fs[pair] = accS[s];
                        if (DRIFT) ft[pair] = accT[s];
                    }
                }
                continue;
            }
            consumer_bar();  // the previous chunk's projection is over
#pragma unroll
            for (int s = 0; s < SLOTS; ++s) {
                const int pair = tid + s * kFoldConsumers;
                if (pair < whalf) {
                    reinterpret_cast<double2*>(sm_s)[pair] = accS[s];
                    if (DRIFT) {
                        // U_j = sum_c (j + cP) x[j + cP] = j S_j + P T_j with the global column j
                        const double j0 = static_cast<double>(w * kLongChunk + 2 * pair);
                        const double Pd = static_cast<double>(P);
                        reinterpret_cast<double2*>(sm_u)[pair] =
                            make_double2(fma(Pd, accT[s].x, j0 * accS[s].x), fma(Pd, accT[s].y, (j0 + 1.0) * accS[s].y));
                    }
                }
            }
            consumer_bar();
            int pass = 0;
            for (int k0 = warp; k0 <= N; k0 += 2 * kFoldConsumerWarps, ++pass) {
                const int k1 = k0 + kFoldConsumerWarps;
                const bool two = k1 <= N;
                const long long col = static_cast<long long>(w) * kLongChunk + lane;
                double sa, ca, sb = 0.0, cb = 0.0;
                sincospi(2.0 * static_cast<double>((static_cast<long long>(k0) * p.kmul * col) % P) / static_cast<double>(P), &sa, &ca);
                if (two)
                    sincospi(2.0 * static_cast<double>((static_cast<long long>(k1) * p.kmul * col) % P) / static_cast<double>(P), &sb, &cb);
                const double2 sta = sm_step[k0];
                const double2 stb = two ? sm_step[k1] : make_double2(1.0, 0.0);
                double acc[2][4] = {{0.0, 0.0, 0.0, 0.0}, {0.0, 0.0, 0.0, 0.0}};  // Q, I, Q drift, I drift
                for (int j = lane; j < wc; j += 32) {
                    const double v = sm_s[j];
                    acc[0][0] = fma(v, ca, acc[0][0]);
                    acc[0][1] = fma(v, sa, acc[0][1]);
                    acc[1][0] = fma(v, cb, acc[1][0]);
                    acc[1][1] = fma(v, sb, acc[1][1]);
                    if (DRIFT) {
                        const double u = sm_u[j];
                        acc[0][2] = fma(u, sa, acc[0][2]);
                        acc[0][3] = fma(u, ca, acc[0][3]);
                        acc[1][2] = fma(u, sb, acc[1][2]);
                        acc[1][3] = fma(u, cb, acc[1][3]);
                    }
                    const double cna = ca * sta.x - sa * sta.y;
                    sa = fma(sa, sta.x, ca * sta.y);
                    ca = cna;
                    const double cnb = cb * stb.x - sb * stb.y;
                    sb = fma(sb, stb.x, cb * stb.y);
                    cb = cnb;
                }
#pragma unroll
                for (int a = 0; a < kLongPasses; ++a) {
                    if (a == pass) {
#pragma unroll
                        for (int h = 0; h < 2; ++h)
#pragma unroll
                            for (int e = 0; e < 4; ++e) hacc[a][h][e] += acc[h][e];
                    }
                }
            }
        }
        if (STORE) continue;
        int pass = 0;
        for (int k0 = warp; k0 <= N; k0 += 2 * kFoldConsumerWarps, ++pass) {
            const int k1 = k0 + kFoldConsumerWarps;
            const bool two = k1 <= N;
            double acc[2][4];
#pragma unroll
            for (int a = 0; a < kLongPasses; ++a) {
                if (a == pass) {
#pragma unroll
                    for (int h = 0; h < 2; ++h)
#pragma unroll
                        for (int e = 0; e < 4; ++e) acc[h][e] = hacc[a][h][e];
                }
            }
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int k = h == 0 ? k0 : k1;
                if (h == 1 && !two) break;
                double aq = warp_sum(acc[h][0]), ai = 0.0, aqu = 0.0, aiu = 0.0;
                if (k > 0) {
                    ai = warp_sum(acc[h][1]);
                    if (DRIFT) {
                        aqu = warp_sum(acc[h][2]);
                        aiu = warp_sum(acc[h][3]);
                    }
                }
                if (lane == 0) {
                    if (k == 0) {
                        p.dc[b] = aq / Rd;
                    } else {
                        double qv = aq, iv = ai;
                        if (DRIFT) {
                            const double d = p.delta[k - 1];
                            qv = fma(-d, aqu, qv);
                            iv = fma(d, aiu, iv);
                        }
                        double* out = p.qi + b * static_cast<long long>(2 * N);
                        out[k - 1] = qv / Rd;
                        out[N + k - 1] = iv / Rd;
                    }
                }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// project_interleaved_kernel -- second half of the time-major lock-in.  fs[b][j][c] (and ft) hold the folded sums of
// time buffer b, time column j of the period, channel c; a thread takes one (buffer, channel) and walks the columns
// (adjacent threads read adjacent channels: coalesced) in j <-> P - j pairs -- the cosine sums need S_j + S_{P-j}, the
// sine sums S_j - S_{P-j}, which halves the work -- accumulating kProjBlock harmonics at a time with a rotation
// recurrence restarted from an exact sincospi every kProjResync pairs.  Output rows are channel-major:
// unit u = c * bpc + b.  The folded arrays are 1/n of the record (n periods per buffer), so this pass reads little.
constexpr int kProjBlock = 6;
constexpr int kProjResync = 32;

template <bool DRIFT>
__global__ void __launch_bounds__(128) project_interleaved_kernel(const double* __restrict__ fs, const double* __restrict__ ft,
                                                                   long long nbuf_t, int C, int P, int R, int N, int kmul,
                                                                   const double* __restrict__ delta, double* __restrict__ qi,
                                                                   double* __restrict__ dc) {
    const long long idx = blockIdx.x * 128ll + threadIdx.x;
    if (idx >= nbuf_t * C) return;
    const long long b = idx / C;
    const int c = static_cast<int>(idx - b * C);
    const double* s = fs + (b * P) * static_cast<long long>(C) + c;
    const double* t = DRIFT ? ft + (b * P) * static_cast<long long>(C) + c : nullptr;
    const double Rd = static_cast<double>(R);
    const long long u = static_cast<long long>(c) * nbuf_t + b;
    double* out = qi + u * static_cast<long long>(2 * N);
    const double Pd = static_cast<double>(P);
    const int half = P >> 1;  // P is even
    for (int k0 = 0; k0 <= N; k0 += kProjBlock) {
        double aq[kProjBlock], ai[kProjBlock], uq[kProjBlock], ui[kProjBlock], cs[kProjBlock], sn[kProjBlock], cst[kProjBlock],
            snt[kProjBlock];
#pragma unroll
        for (int h = 0; h < kProjBlock; ++h) {
            aq[h] = ai[h] = uq[h] = ui[h] = 0.0;
            const long long r1 = (static_cast<long long>(k0 + h) * kmul) % P;
            sincospi(2.0 * static_cast<double>(r1) / Pd, &snt[h], &cst[h]);  // one-column step of harmonic k0 + h
        }
        for (int j0 = 0; j0 <= half; j0 += kProjResync) {
#pragma unroll
            for (int h = 0; h < kProjBlock; ++h) {
                const long long r0 = (static_cast<long long>(k0 + h) * kmul * j0) % P;
                sincospi(2.0 * static_cast<double>(r0) / Pd, &sn[h], &cs[h]);
            }
            const int j1 = min(half + 1, j0 + kProjResync);
            // four column pairs per trip, their (independent, L2 / HBM latency) loads issued before any arithmetic
            for (int jb = j0; jb < j1; jb += 4) {
                double v1[4], v2[4], t1[4], t2[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int j = jb + e;
                    const bool live = j < j1, self = j == 0 || j == half;
                    v1[e] = live ? s[static_cast<long long>(j) * C] : 0.0;
                    v2[e] = (live && !self) ? s[static_cast<long long>(P - j) * C] : 0.0;
                    if (DRIFT) {
                        t1[e] = live ? t[static_cast<long long>(j) * C] : 0.0;
                        t2[e] = (live && !self) ? t[static_cast<long long>(P - j) * C] : 0.0;
                    }
                }
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int j = jb + e;
                    if (j >= j1) break;
                    const bool self = j == 0 || j == half;  // columns that pair with themselves
                    const double va = v1[e] + v2[e], vd = self ? 0.0 : v1[e] - v2[e];
                    double wa = 0.0, wd = 0.0;
                    if (DRIFT) {  // U_j = j S_j + P T_j
                        const double w1 = fma(Pd, t1[e], static_cast<double>(j) * v1[e]);
                        const double w2 = self ? 0.0 : fma(Pd, t2[e], static_cast<double>(P - j) * v2[e]);
                        wa = w1 + w2;
                        wd = self ? 0.0 : w1 - w2;
                    }
#pragma unroll
                    for (int h = 0; h < kProjBlock; ++h) {
                        aq[h] = fma(va, cs[h], aq[h]);
                        ai[h] = fma(vd, sn[h], ai[h]);
                        if (DRIFT) {
                            uq[h] = fma(wd, sn[h], uq[h]);
                            ui[h] = fma(wa, cs[h], ui[h]);
                        }
                        const double cn = cs[h] * cst[h] - sn[h] * snt[h];
                        sn[h] = fma(sn[h], cst[h], cs[h] * snt[h]);
                        cs[h] = cn;
                    }
                }
            }
        }
#pragma unroll
        for (int h = 0; h < kProjBlock; ++h) {
            const int k = k0 + h;
            if (k > N) break;
            if (k == 0) {
                dc[u] = aq[h] / Rd;
            } else {
                double qv = aq[h], iv = ai[h];
                if (DRIFT) {
                    qv = fma(-delta[k - 1], uq[h], qv);
                    iv = fma(delta[k - 1], ui[h], iv);
                }
                out[k - 1] = qv / Rd;
                out[N + k - 1] = iv / Rd;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// demod_tile_kernel -- short modulation periods (P <= 256: the 200 kHz configs).  A buffer is then small
// (32 kB at n = 20, 1.6 kB at n = 1) and the per-buffer block barriers of demod_fold_kernel dominate, so here
// nothing is synchronised across the CTA: the producer lane streams *groups* of NBW consecutive buffers through
// one CTA-wide TMA ring, group i of the CTA belongs to warp i % 8 alone, and that warp folds its buffers in
// registers, forms the j <-> P-j combinations through a private scratch column and takes all 2N+1 outputs of its
// NBW buffers as one small dense product with a twiddle table held in shared memory for the life of the CTA
// (lane = output row, NBW accumulators per lane, table value loaded once per NBW buffers).  No recurrence, no
// shuffles, no __syncthreads after set-up.
constexpr int kTileMaxPeriod = 256;
constexpr int kTileMaxSlots = kTileMaxPeriod / 2 / 32;  // column pairs per lane (4)
constexpr int kTileStageBytes = 16384;

struct TileParams {
    const double* x;
    double* qi;
    double* dc;
    long long nbuf;
    int R, P, periods, N;
    int kmul;     // modulation periods per fold length P
    int pps;      // periods per ring stage
    int cpg;      // stages per full group
    int nstages;  // ring depth
    double delta[kMaxHarmonics];
};

struct TileSmem {
    int ldt;         // table row stride in doubles (odd: lanes on consecutive rows hit distinct banks)
    int nv_pad;      // table rows, a multiple of 32
    int xrow;        // doubles per column j in a warp's operand block
    int stage_doubles;
    size_t off_t1, off_t2, off_scr, off_x, off_stage, off_bar, total;
    size_t scr_per_warp, x_per_warp;  // in doubles
};

inline __host__ __device__ TileSmem tile_smem_layout(int P, int N, int nbw, int pps, int nstages, bool drift) {
    TileSmem L;
    const int half = P / 2;
    L.ldt = (half + 1) | 1;
    L.nv_pad = ((2 * N + 1) + 31) / 32 * 32;
    const int ncomp = drift ? 4 : 2;
    L.xrow = ncomp * nbw + (nbw > 1 ? 2 : 0);
    L.stage_doubles = pps * P;
    L.scr_per_warp = static_cast<size_t>(P) * (drift ? 2 : 1);
    L.x_per_warp = static_cast<size_t>(half + 1) * L.xrow;
    size_t o = 0;
    L.off_stage = o;
    o += static_cast<size_t>(nstages) * L.stage_doubles * 8;
    o = (o + 15) & ~static_cast<size_t>(15);
    L.off_t1 = o;
    o += static_cast<size_t>(L.nv_pad) * L.ldt * 8;
    L.off_t2 = o;
    o += drift ? static_cast<size_t>(L.nv_pad) * L.ldt * 8 : 0;
    o = (o + 15) & ~static_cast<size_t>(15);
    L.off_scr = o;
    o += kFoldConsumerWarps * L.scr_per_warp * 8;
    o = (o + 15) & ~static_cast<size_t>(15);
    L.off_x = o;
    o += kFoldConsumerWarps * ((L.x_per_warp * 8 + 15) & ~static_cast<size_t>(15));
    L.off_bar = o;
    o += static_cast<size_t>(2 * nstages + 1) * 8;  // full[], empty[], issued-chunk counter
    L.total = o;
    return L;
}

template <bool DRIFT, int NBW>
__global__ void __launch_bounds__(kFoldThreads, 1) demod_tile_kernel(const TileParams p) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const TileSmem L = tile_smem_layout(p.P, p.N, NBW, p.pps, p.nstages, DRIFT);
    double* stage_base = reinterpret_cast<double*>(smem_raw + L.off_stage);
    double* t1 = reinterpret_cast<double*>(smem_raw + L.off_t1);
    double* t2 = reinterpret_cast<double*>(smem_raw + L.off_t2);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + L.off_bar);
    uint64_t* empty = full + p.nstages;
    // Chunks issued so far.  The warps run independently, so the owner of chunk q + nstages can reach its wait
    // before chunk q (same stage, opposite parity) has even been issued, and a parity wait cannot tell those two
    // phases apart; a warp therefore first waits until its chunk has been issued, then on the stage's barrier.
    volatile unsigned long long* issued = reinterpret_cast<volatile unsigned long long*>(empty + p.nstages);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int P = p.P, N = p.N, half = P >> 1, n = p.periods, NV = 2 * N + 1;
    const long long ngroups = (p.nbuf + NBW - 1) / NBW;
    // groups of this CTA: blockIdx.x, blockIdx.x + gridDim.x, ...
    const long long my_groups = ngroups > blockIdx.x ? (ngroups - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

    if (tid == 0) {
        for (int s = 0; s < p.nstages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 1);
        }
        *issued = 0ull;
        mbar_fence_init();
    }
    // twiddle table: row 0 = 1 (mean), rows 1..N = cos(2 pi k j / P), rows N+1..2N = sin(2 pi k j / P);
    // second table (drift term): -delta_k sin for the cosine rows, +delta_k cos for the sine rows
    for (int i = tid; i < L.nv_pad * L.ldt; i += kFoldThreads) {
        const int v = i / L.ldt, j = i - v * L.ldt;
        double a = 0.0, b = 0.0;
        if (v < NV && j <= half) {
            const int k = v <= N ? v : v - N;
            double sn, cs;
            sincospi(2.0 * static_cast<double>((static_cast<long long>(k) * p.kmul * j) % P) / static_cast<double>(P), &sn, &cs);
            a = v <= N ? cs : sn;
            if (DRIFT && v > 0) b = v <= N ? -p.delta[k - 1] * sn : p.delta[k - 1] * cs;
        }
        t1[i] = a;
        if (DRIFT) t2[i] = b;
    }
    __syncthreads();

    if (warp == kFoldConsumerWarps) {
        if (lane == 0) {
            const uint64_t pol = l2_evict_first_policy();
            int stage = 0;
            uint32_t phase = 0;
            unsigned long long count = 0;
            for (long long i = 0; i < my_groups; ++i) {
                const long long g = blockIdx.x + i * gridDim.x;
                const long long b0 = g * NBW;
                const int nb = static_cast<int>(min(static_cast<long long>(NBW), p.nbuf - b0));
                const int tot = nb * n;  // periods in this group
                const double* src = p.x + b0 * static_cast<long long>(p.R);
                for (int q0 = 0; q0 < tot; q0 += p.pps) {
                    const int np = min(p.pps, tot - q0);
                    const uint32_t bytes = static_cast<uint32_t>(np) * static_cast<uint32_t>(P) * 8u;
                    mbar_wait(&empty[stage], phase ^ 1u);
                    mbar_arrive_expect_tx(&full[stage], bytes);
                    bulk_load(stage_base + static_cast<size_t>(stage) * L.stage_doubles,
                              src + static_cast<size_t>(q0) * P, bytes, &full[stage], pol);
                    __threadfence_block();
                    *issued = ++count;
                    if (++stage == p.nstages) {
                        stage = 0;
                        phase ^= 1u;
                    }
                }
            }
        }
        return;
    }

    double* scr_s = reinterpret_cast<double*>(smem_raw + L.off_scr) + warp * L.scr_per_warp;
    double* scr_u = scr_s + P;
    double* X = reinterpret_cast<double*>(smem_raw + L.off_x + warp * ((L.x_per_warp * 8 + 15) & ~static_cast<size_t>(15)));
    const int xrow = L.xrow;
    const double Rd = static_cast<double>(p.R);

    // Ring position of chunk number q (CTA-wide count): stage q % nstages, phase (q / nstages) & 1.  Full groups
    // have cpg chunks; only the CTA's last group can be short, so the count before group i is i * cpg.
    for (long long i = warp; i < my_groups; i += kFoldConsumerWarps) {
        const long long g = blockIdx.x + i * gridDim.x;
        const long long b0 = g * NBW;
        const int nb = static_cast<int>(min(static_cast<long long>(NBW), p.nbuf - b0));
        const int tot = nb * n;
        long long q = i * p.cpg;
        if (!DRIFT && NBW > 1 && n == 1 && p.cpg == 1) {
            // One period per buffer (the Monte-Carlo shape) and the whole group in one stage: nothing to fold.
            // Lane j reads column j and P-j of all NBW rows and writes the combinations of column j for the NBW
            // buffers as contiguous 128-bit stores -- the transpose the product below wants, with every shared
            // memory access conflict-free.
            const int stage = static_cast<int>(q % p.nstages);
            const uint32_t phase = static_cast<uint32_t>((q / p.nstages) & 1);
            while (*issued <= static_cast<unsigned long long>(q)) __nanosleep(64);
            __threadfence_block();
            mbar_wait(&full[stage], phase);
            const double* sm = stage_base + static_cast<size_t>(stage) * L.stage_doubles;
            for (int j = lane; j <= half; j += 32) {
                const bool self = (j == 0) || (j == half);
                double a[NBW], b[NBW];
#pragma unroll
                for (int s = 0; s < NBW; ++s) {
                    const bool have = s < nb;
                    const double va = have ? sm[s * P + j] : 0.0;
                    const double vb = (have && !self) ? sm[s * P + (P - j)] : 0.0;
                    a[s] = va + vb;
                    b[s] = self ? 0.0 : va - vb;
                }
                double2* xr = reinterpret_cast<double2*>(X + j * xrow);
#pragma unroll
                for (int s = 0; s < NBW; s += 2) {
                    xr[s / 2] = make_double2(a[s], a[s + 1]);
                    xr[(NBW + s) / 2] = make_double2(b[s], b[s + 1]);
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[stage]);
        } else {
        double2 accS[kTileMaxSlots], accT[kTileMaxSlots];
#pragma unroll
        for (int s = 0; s < kTileMaxSlots; ++s) accS[s] = accT[s] = make_double2(0.0, 0.0);
        int pin = 0;   // period index inside the current buffer
        int slot = 0;  // buffer inside the group
        for (int q0 = 0; q0 < tot; q0 += p.pps, ++q) {
            const int np = min(p.pps, tot - q0);
            const int stage = static_cast<int>(q % p.nstages);
            const uint32_t phase = static_cast<uint32_t>((q / p.nstages) & 1);
            while (*issued <= static_cast<unsigned long long>(q)) __nanosleep(64);
            __threadfence_block();
            mbar_wait(&full[stage], phase);
            const double* sm = stage_base + static_cast<size_t>(stage) * L.stage_doubles;
            for (int c = 0; c < np; ++c) {
                const double2* row = reinterpret_cast<const double2*>(sm + c * P);
                const double cin = static_cast<double>(pin);
#pragma unroll
                for (int s = 0; s < kTileMaxSlots; ++s) {
                    const int pair = lane + 32 * s;
                    if (pair < half) {
                        const double2 v = row[pair];
                        accS[s].x += v.x;
                        accS[s].y += v.y;
                        if (DRIFT) {
                            accT[s].x = fma(cin, v.x, accT[s].x);
                            accT[s].y = fma(cin, v.y, accT[s].y);
                        }
                    }
                }
                if (++pin == n) {
                    // buffer complete: folded period -> scratch -> even/odd combinations -> operand block
#pragma unroll
                    for (int s = 0; s < kTileMaxSlots; ++s) {
                        const int pair = lane + 32 * s;
                        if (pair < half) {
                            reinterpret_cast<double2*>(scr_s)[pair] = accS[s];
                            if (DRIFT) {
                                const double j0 = static_cast<double>(2 * pair), Pd = static_cast<double>(P);
                                reinterpret_cast<double2*>(scr_u)[pair] = make_double2(
                                    fma(Pd, accT[s].x, j0 * accS[s].x), fma(Pd, accT[s].y, (j0 + 1.0) * accS[s].y));
                            }
                        }
                        accS[s] = accT[s] = make_double2(0.0, 0.0);
                    }
                    __syncwarp();
                    for (int j = lane; j <= half; j += 32) {
                        const bool self = (j == 0) || (j == half);
                        const double sa = scr_s[j], sb = self ? 0.0 : scr_s[P - j];
                        double* xr = X + j * xrow + slot;
                        xr[0] = sa + sb;
                        xr[NBW] = self ? 0.0 : sa - sb;
                        if (DRIFT) {
                            const double ua = scr_u[j], ub = self ? 0.0 : scr_u[P - j];
                            xr[2 * NBW] = ua + ub;
                            xr[3 * NBW] = self ? 0.0 : ua - ub;
                        }
                    }
                    __syncwarp();
                    pin = 0;
                    ++slot;
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[stage]);
        }
        }

        // outputs of the group: lane = output row (0 = mean, 1..N = Q_k, N+1..2N = I_k)
        for (int vb = 0; vb < NV; vb += 32) {
            const int v = vb + lane;
            const bool active = v < NV;
            const int vv = active ? v : 0;
            const double* trow = t1 + vv * L.ldt;
            const double* urow = t2 + vv * L.ldt;
            const double* x1 = X + (vv <= N ? 0 : NBW);          // cosine rows read A, sine rows read B
            const double* x2 = X + (vv <= N ? 3 * NBW : 2 * NBW);  // drift: cosine rows read BU, sine rows read AU
            double acc[NBW];
#pragma unroll
            for (int s = 0; s < NBW; ++s) acc[s] = 0.0;
#pragma unroll 4
            for (int j = 0; j <= half; ++j) {
                const double tv = trow[j];
                if (NBW == 1) {
                    acc[0] = fma(tv, x1[j * xrow], acc[0]);
                } else {
#pragma unroll
                    for (int s = 0; s < NBW; s += 2) {
                        const double2 xv = *reinterpret_cast<const double2*>(x1 + j * xrow + s);
                        acc[s] = fma(tv, xv.x, acc[s]);
                        acc[s + 1] = fma(tv, xv.y, acc[s + 1]);
                    }
                }
                if (DRIFT) {
                    const double uv = urow[j];
                    if (NBW == 1) {
                        acc[0] = fma(uv, x2[j * xrow], acc[0]);
                    } else {
#pragma unroll
                        for (int s = 0; s < NBW; s += 2) {
                            const double2 xv = *reinterpret_cast<const double2*>(x2 + j * xrow + s);
                            acc[s] = fma(uv, xv.x, acc[s]);
                            acc[s + 1] = fma(uv, xv.y, acc[s + 1]);
                        }
                    }
                }
            }
            if (active) {
#pragma unroll
                for (int s = 0; s < NBW; ++s) {
                    if (s < nb) {
                        const long long b = b0 + s;
                        const double val = acc[s] / Rd;
                        if (v == 0) {
                            p.dc[b] = val;
                        } else {
                            p.qi[b * static_cast<long long>(2 * N) + (v - 1)] = val;
                        }
                    }
                }
            }
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------------------
// demod_period_kernel -- one modulation period per buffer (R = P <= 256, P % 4 == 0): the Monte-Carlo shape
// (BASELINE config 5: 1.9e7 buffers of 1.6 kB).  Same CTA-wide ring and warp-owns-group scheme as the tile kernel
// with groups of 8 buffers, but the product is cut down twice more, because here it -- not HBM -- is the bound
// (the tile kernel's product keeps the shared-memory pipe > 90 % busy at this shape):
//   * quarter-wave symmetry on top of the half-wave one: with j' = P/2 - j,
//     cos(k th_j') = (-1)^k cos(k th_j) and sin(k th_j') = -(-1)^k sin(k th_j), so even and odd harmonics read
//     different combinations (AE, AO, BE, BO) and the column range halves to 0..P/4;
//   * every lane produces 2 output rows x 4 buffers (instead of 1 x 8), which loads 6 operands per 8 FMAs
//     instead of 9: shared-memory loads are charged per lane-byte, broadcast or not.
constexpr int kPeriodNbw = 8;
// Consumer warps of the one build of demod_period_kernel<WARPS> (+ one producer warp).  It stays a template: as a
// plain kernel its 128-byte-aligned smem_raw would be the module's first dynamic shared array, which moves the dynamic
// shared memory of synth_snr_kernel from byte 16 to byte 128.
constexpr int kPeriodWarps = 8;

struct PeriodParams {
    const double* x;
    double* qi;
    double* dc;
    long long nbuf;
    int P, N;
    int nstages;
};

struct PeriodSmem {
    int quarter, nrows, xrow, stage_doubles;
    size_t off_stage, off_t, off_x, off_rows, off_bar, total;
    size_t x_per_warp;  // doubles
};

// output rows in the order cos-even (k = 0, 2, ..), cos-odd, sin-even, sin-odd, each block padded to a multiple of
// four so that the four rows of a lane always read the same operand; total padded to a multiple of 32.
inline __host__ __device__ int period_rows(int N) {
    const int ce = N / 2 + 1, co = (N + 1) / 2, se = N / 2, so = (N + 1) / 2;
    const int tot = ((ce + 3) & ~3) + ((co + 3) & ~3) + ((se + 3) & ~3) + ((so + 3) & ~3);
    return (tot + 31) / 32 * 32;
}

// Where row r of the twiddle table sits inside its 32-row block: the block is stored as two halves of eight 16-byte
// chunks, chunk g of half h holding rows 4g + 2h, 4g + 2h + 1 -- so that the eight row groups of a warp read eight
// consecutive chunks with each of their two loads.
inline __host__ __device__ int period_row_slot(int r) { return (r & ~31) + ((r & 3) >> 1) * 16 + ((r >> 2) & 7) * 2 + (r & 1); }

inline __host__ __device__ PeriodSmem period_smem_layout(int P, int N, int nstages, int warps = kPeriodWarps) {
    PeriodSmem L;
    L.quarter = P / 4;
    L.nrows = period_rows(N);
    L.xrow = 4 * kPeriodNbw + 2;
    L.stage_doubles = kPeriodNbw * P;
    L.x_per_warp = static_cast<size_t>(L.quarter + 1) * L.xrow;
    size_t o = 0;
    L.off_stage = o;
    o += static_cast<size_t>(nstages) * L.stage_doubles * 8;
    L.off_t = o;
    o += static_cast<size_t>(L.quarter + 1) * L.nrows * 8;
    L.off_x = o;
    o += static_cast<size_t>(warps) * L.x_per_warp * 8;
    L.off_rows = o;
    o += static_cast<size_t>(L.nrows) * 2 * sizeof(int);  // row_type[], row_out[]
    o = (o + 7) & ~static_cast<size_t>(7);
    L.off_bar = o;
    o += static_cast<size_t>(2 * nstages + 1) * 8;
    L.total = o;
    return L;
}

// Row tables and twiddles of a CTA (all threads call it; it synchronises).
// row_out: -1 = padding, 0 = mean, k = Q_k (qi column k-1), N + k = I_k (qi column N+k-1).
DFK_D void period_build_tables(int P, int N, int nrows, int quarter, double* T, int* row_type, int* row_out, int tid,
                               int nthreads) {
    if (tid == 0) {
        int v = 0;
        for (int type = 0; type < 4; ++type) {
            const int k0 = (type == 0) ? 0 : (type == 2 ? 2 : 1);
            for (int k = k0; k <= N; k += 2, ++v) {
                row_type[v] = type;
                row_out[v] = type < 2 ? k : N + k;
            }
            for (; v & 3; ++v) {
                row_type[v] = type;
                row_out[v] = -1;
            }
        }
        for (; v < nrows; ++v) {
            row_type[v] = 3;
            row_out[v] = -1;
        }
    }
    __syncthreads();
    for (int i = tid; i < (quarter + 1) * nrows; i += nthreads) {
        const int j = i / nrows, v = i - j * nrows;
        const int out = row_out[v];
        double val = 0.0;
        if (out >= 0) {
            const int k = out <= N ? out : out - N;
            double sn, cs;
            sincospi(2.0 * static_cast<double>((static_cast<long long>(k) * j) % P) / static_cast<double>(P), &sn, &cs);
            val = out <= N ? cs : sn;
        }
        T[j * nrows + period_row_slot(v)] = val;
    }
    __syncthreads();
}

// Combinations of columns j, P-j, j' = P/2-j, P-j' of the eight buffers at sm (buffer s at sm + s*P), written
// transposed into the warp's scratch X: row j holds AE, AO, BE, BO, eight buffers each.  Buffers past the end of a
// ragged last group hold stale bytes; their outputs are never stored, so they are combined like the rest.
// Interior columns 0 < j < P/4 take the branch-free path; the two self-paired columns j = 0 and j = P/4 follow on two
// lanes.
template <bool EDGE>
DFK_D void period_combo_column(const double* sm, double* X, int P, int xrow, int j) {
    constexpr int NBW = kPeriodNbw;
    const int half = P >> 1, quarter = P >> 2;
    const int jp = half - j;
    const bool first = EDGE && j == 0, mid = EDGE && j == quarter;
    double2* xr = reinterpret_cast<double2*>(X + j * xrow);
    double ae[NBW], ao[NBW], be[NBW], bo[NBW];
#pragma unroll
    for (int s = 0; s < NBW; ++s) {
        const double* row = sm + s * P;
        const double s1 = row[j];
        const double s2 = first ? 0.0 : row[P - j];
        const double s3 = row[jp];
        const double s4 = first ? 0.0 : row[half + j];  // column P - j'
        const double aj = s1 + s2, bj = first ? 0.0 : s1 - s2;
        const double ap = s3 + s4, bp = first ? 0.0 : s3 - s4;
        ae[s] = mid ? aj : aj + ap;
        ao[s] = mid ? 0.0 : aj - ap;
        be[s] = mid ? 0.0 : bj - bp;
        bo[s] = mid ? bj : bj + bp;
    }
    // chunk (type, hb, half) = half * 8 + type * 2 + hb holds buffers 4 hb + 2 half, + 1: the product's two loads
    // per lane (half 0, half 1) each sweep eight consecutive chunks over the (type, hb) pairs of a warp
#pragma unroll
    for (int s = 0; s < NBW; s += 2) {
        const int c = ((s >> 1) & 1) * 8 + (s >> 2);
        xr[c + 0] = make_double2(ae[s], ae[s + 1]);
        xr[c + 2] = make_double2(ao[s], ao[s + 1]);
        xr[c + 4] = make_double2(be[s], be[s + 1]);
        xr[c + 6] = make_double2(bo[s], bo[s + 1]);
    }
}

DFK_D void period_combos(const double* sm, double* X, int P, int xrow, int lane) {
    const int quarter = P >> 2;
    for (int j = 1 + lane; j < quarter; j += 32) period_combo_column<false>(sm, X, P, xrow, j);
    if (lane < 2) period_combo_column<true>(sm, X, P, xrow, lane == 0 ? 0 : quarter);
}

// Product of the combinations with the twiddle table.  Lane = (row group g = lane % 8: rows 4g..4g+3 of each 32-row
// block, buffer half hb = (lane / 8) % 2: buffers 4hb..4hb+3, column parity = lane / 16): 16 accumulators fed by four
// 128-bit loads per column -- 4 bytes of shared memory per FMA instead of 6 -- the two half-warps taking alternate
// columns and adding up at the end.  The results of the group are laid out in the warp's scratch as they lie in
// memory (qi rows of consecutive buffers are contiguous) and leave with 128-bit stores.
// out_stage: 8 * 2N + 8 doubles of warp-private shared memory that the product no longer reads (the head of X).
DFK_D void period_product(double* X, const double* T, const int* row_type, const int* row_out, int P, int N, int nrows,
                          int xrow, int nb, long long b0, double* __restrict__ qi, double* __restrict__ dc, int lane) {
    const int quarter = P >> 2;
    const double inv_r = 1.0 / static_cast<double>(P);
    const int g = lane & 7, hb = (lane >> 3) & 1, par = lane >> 4;
    const int two_n = 2 * N;
    const bool staged = nrows == 32;  // one 32-row block (N <= 15): X is free once its loop ends
    for (int vb = 0; vb < nrows; vb += 32) {
        const int r0 = vb + 4 * g;
        const double* tp = T + vb + 2 * g;                     // + 16 for rows 2, 3 of the group
        const double* xp = X + (row_type[r0] * 2 + hb) * 2;   // + 16 for buffers 2, 3 of the half
        double acc[4][4];
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int s = 0; s < 4; ++s) acc[r][s] = 0.0;
#pragma unroll 2
        for (int j = par; j <= quarter; j += 2) {
            const double2 t01 = *reinterpret_cast<const double2*>(tp + j * nrows);
            const double2 t23 = *reinterpret_cast<const double2*>(tp + j * nrows + 16);
            const double2 xa = *reinterpret_cast<const double2*>(xp + j * xrow);
            const double2 xb = *reinterpret_cast<const double2*>(xp + j * xrow + 16);
            const double t[4] = {t01.x, t01.y, t23.x, t23.y};
            const double x[4] = {xa.x, xa.y, xb.x, xb.y};
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int s = 0; s < 4; ++s) acc[r][s] = fma(t[r], x[s], acc[r][s]);
        }
        // even + odd columns; the lower half-warp keeps rows 0, 1 of its group, the upper one rows 2, 3
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int s = 0; s < 4; ++s) acc[r][s] += __shfl_xor_sync(0xffffffffu, acc[r][s], 16);
        if (staged) __syncwarp();  // every lane is done reading X: its head becomes the output stage
        double* oq = X;              // [8][2N]
        double* od = X + 8 * two_n;  // [8]
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) {
            const int out = row_out[r0 + 2 * par + rr];
            if (out < 0) continue;
#pragma unroll
            for (int s = 0; s < 4; ++s) {
                const int slot = 4 * hb + s;
                const double val = (par == 0 ? acc[rr][s] : acc[2 + rr][s]) * inv_r;
                if (staged) {
                    if (out == 0) od[slot] = val; else oq[slot * two_n + (out - 1)] = val;
                } else if (slot < nb) {
                    if (out == 0) dc[b0 + slot] = val; else qi[(b0 + slot) * static_cast<long long>(two_n) + (out - 1)] = val;
                }
            }
        }
    }
    if (staged) {
        __syncwarp();
        double2* dst = reinterpret_cast<double2*>(qi + b0 * static_cast<long long>(two_n));  // 16-byte aligned: b0 % 8 == 0
        const double2* src = reinterpret_cast<const double2*>(X);
        for (int i = lane; i < nb * N; i += 32) dst[i] = src[i];
        if (lane < nb) dc[b0 + lane] = X[8 * two_n + lane];
        __syncwarp();  // the stage is X again for the next group
    }
}

template <int WARPS>
__global__ void __launch_bounds__((WARPS + 1) * 32, 1) demod_period_kernel(const PeriodParams p) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const PeriodSmem L = period_smem_layout(p.P, p.N, p.nstages, WARPS);
    double* stage_base = reinterpret_cast<double*>(smem_raw + L.off_stage);
    double* T = reinterpret_cast<double*>(smem_raw + L.off_t);
    int* row_type = reinterpret_cast<int*>(smem_raw + L.off_rows);
    int* row_out = row_type + L.nrows;
    uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + L.off_bar);
    uint64_t* empty = full + p.nstages;
    volatile unsigned long long* issued = reinterpret_cast<volatile unsigned long long*>(empty + p.nstages);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int P = p.P, N = p.N, nrows = L.nrows;
    constexpr int NBW = kPeriodNbw;
    const long long ngroups = (p.nbuf + NBW - 1) / NBW;
    const long long my_groups = ngroups > blockIdx.x ? (ngroups - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

    if (tid == 0) {
        for (int s = 0; s < p.nstages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 1);
        }
        *issued = 0ull;
        mbar_fence_init();
    }
    period_build_tables(P, N, nrows, L.quarter, T, row_type, row_out, tid, (WARPS + 1) * 32);

    if (warp == WARPS) {
        if (lane == 0) {
            const uint64_t pol = l2_evict_first_policy();
            int stage = 0;
            uint32_t phase = 0;
            unsigned long long count = 0;
            for (long long i = 0; i < my_groups; ++i) {
                const long long b0 = (blockIdx.x + i * gridDim.x) * NBW;
                const int nb = static_cast<int>(min(static_cast<long long>(NBW), p.nbuf - b0));
                const uint32_t bytes = static_cast<uint32_t>(nb) * static_cast<uint32_t>(P) * 8u;
                mbar_wait(&empty[stage], phase ^ 1u);
                mbar_arrive_expect_tx(&full[stage], bytes);
                bulk_load(stage_base + static_cast<size_t>(stage) * L.stage_doubles, p.x + b0 * static_cast<long long>(P),
                          bytes, &full[stage], pol);
                __threadfence_block();
                *issued = ++count;
                if (++stage == p.nstages) {
                    stage = 0;
                    phase ^= 1u;
                }
            }
        }
        return;
    }

    double* X = reinterpret_cast<double*>(smem_raw + L.off_x) + warp * L.x_per_warp;
    const bool own_stage = (p.nstages % WARPS) == 0;
    for (long long i = warp; i < my_groups; i += WARPS) {
        const long long b0 = (blockIdx.x + i * gridDim.x) * NBW;
        const int nb = static_cast<int>(min(static_cast<long long>(NBW), p.nbuf - b0));
        const int stage = static_cast<int>(i % p.nstages);
        const uint32_t phase = static_cast<uint32_t>((i / p.nstages) & 1);
        // A parity wait is only sound once the stage's previous occupant has landed.  When the ring depth is a
        // multiple of the consumer warps, a stage always belongs to the same warp, which consumed that occupant itself;
        // otherwise wait until the producer has issued this group (it could not before the occupant was released).
        if (!own_stage) {
            while (*issued <= static_cast<unsigned long long>(i)) __nanosleep(64);
            __threadfence_block();
        }
        mbar_wait(&full[stage], phase);
        period_combos(stage_base + static_cast<size_t>(stage) * L.stage_doubles, X, P, L.xrow, lane);
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[stage]);
        period_product(X, T, row_type, row_out, P, N, nrows, L.xrow, nb, b0, p.qi, p.dc, lane);
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------------------
// Lock-in for records that cannot fold (the modulation period is not a small rational number of samples, or the
// buffer is not whole fold lengths): every sample meets every harmonic, cos/sin of fl(w_k t) as the reference forms
// them (fit.py:55-64).  Lane l of a warp takes the samples t = l + 32 j of a piece, so that
//     w_k t = w_k l + w_k 32 j,
// the second term being the same for every lane and every piece: its cos/sin for j < steps live in a shared-memory
// table built once per launch (read as broadcasts), and a sample costs its load plus two FMAs per harmonic.  The
// lane's sums are rotated by w_k l at the end (a second, 32-entry table), then reduced over the warp.
// A piece is a whole buffer when it fits a table (32 * steps samples), else one of its chunks of that length: the
// chunk sums, taken with t counted from the chunk's start, go to scratch and direct_combine_kernel rotates each by
// w_k c0 (its own sincos: nothing accumulates along the buffer) and adds them up in order -- so a few very long
// buffers spread over the whole GPU like many short ones.
// KB harmonics per pass over the record (N > KB re-reads it).
// Rotating term by term instead (the first version of this kernel: one complex rotation per sample and harmonic, two
// sincos per 64 samples to stop its drift) spent 7 fp64 operations where this one spends 2: 0.34 TB/s.
// ---------------------------------------------------------------------------------------------------
constexpr int kDirectThreads = 256;

struct DirectParams {
    const double* x;
    long long nbuf, bpc, ld_c, R;
    int N;
    double w0;
    double* qi;
    double* dc;
    int steps;          // table length: pieces of up to 32 * steps samples
    long long cpb;      // pieces (chunks) per buffer; 1: a piece is the buffer, results go straight to qi / dc
    double* part;       // cpb > 1: [nbuf * cpb][2 N + 1] rotated, un-normalised chunk sums and the chunk's plain sum
};

// piece v of the launch: where it starts and how long it is
DFK_D const double* direct_piece(const DirectParams& p, long long v, long long& len) {
    const long long b = v / p.cpb, c = v - b * p.cpb;
    const long long L = 32ll * p.steps;
    len = p.cpb == 1 ? p.R : (p.R - c * L < L ? p.R - c * L : L);
    return p.x + (b / p.bpc) * p.ld_c + (b % p.bpc) * p.R + c * L;
}

DFK_D void direct_build_tables(const DirectParams& p, int k0, int KB, double2* tab, double2* lane_tab, int tid, int nthreads) {
    for (int i = tid; i < p.steps * KB; i += nthreads) {
        const int j = i / KB, kk = i - j * KB;
        const double wk = static_cast<double>(k0 + kk + 1) * p.w0;  // fl((k + 1) * w0), fit.py:59
        double sv, cv;
        sincos(wk * static_cast<double>(32 * j), &sv, &cv);
        tab[i] = make_double2(cv, sv);
    }
    for (int i = tid; i < KB * 32; i += nthreads) {
        const int kk = i >> 5, l = i & 31;
        const double wk = static_cast<double>(k0 + kk + 1) * p.w0;
        double sv, cv;
        sincos(wk * static_cast<double>(l), &sv, &cv);
        lane_tab[i] = make_double2(cv, sv);
    }
}

// lane 0 stores harmonic k0 + kk of piece v: normalised into qi when the piece is the buffer, else raw into scratch
DFK_D void direct_store(const DirectParams& p, long long v, int k, double q, double i, double inv_r) {
    if (p.cpb == 1) {
        p.qi[v * 2 * p.N + k] = q * inv_r;
        p.qi[v * 2 * p.N + p.N + k] = i * inv_r;
    } else {
        p.part[v * (2 * p.N + 1) + k] = q;
        p.part[v * (2 * p.N + 1) + p.N + k] = i;
    }
}
DFK_D void direct_store_sum(const DirectParams& p, long long v, double sum, double inv_r) {
    if (p.cpb == 1) p.dc[v] = sum * inv_r;
    else p.part[v * (2 * p.N + 1) + 2 * p.N] = sum;
}

template <int KB, int THREADS = kDirectThreads>
__global__ void __launch_bounds__(THREADS) demod_direct_kernel(const DirectParams p) {
    extern __shared__ __align__(16) unsigned char direct_smem[];
    double2* tab = reinterpret_cast<double2*>(direct_smem);                  // [steps][KB]: cos, sin of w_k 32 j
    double2* lane_tab = tab + static_cast<size_t>(p.steps) * KB;             // [KB][32]:    cos, sin of w_k l
    const int tid = threadIdx.x, lane = tid & 31;
    const long long warp = (static_cast<long long>(blockIdx.x) * THREADS + tid) >> 5;
    const long long nwarps = (static_cast<long long>(gridDim.x) * THREADS) >> 5;
    const double inv_r = 1.0 / static_cast<double>(p.R);
    const long long npieces = p.nbuf * p.cpb;
    for (int k0 = 0; k0 < p.N; k0 += KB) {
        __syncthreads();  // the previous pass is done with the tables
        direct_build_tables(p, k0, KB, tab, lane_tab, tid, THREADS);
        __syncthreads();
        for (long long v = warp; v < npieces; v += nwarps) {
            long long len;
            const double* src = direct_piece(p, v, len) + lane;
            double sc[KB], ss[KB];
            double asum = 0.0;
#pragma unroll
            for (int kk = 0; kk < KB; ++kk) sc[kk] = ss[kk] = 0.0;
            const int full = static_cast<int>(len >> 5);  // steps with all 32 lanes
            int j = 0;
            for (; j + 4 <= full; j += 4) {  // four loads in flight per lane
                double x4[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) x4[e] = __ldg(src + 32 * (j + e));
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    asum += x4[e];
                    const double2* row = tab + static_cast<size_t>(j + e) * KB;
#pragma unroll
                    for (int kk = 0; kk < KB; ++kk) {
                        const double2 w = row[kk];
                        sc[kk] = fma(x4[e], w.x, sc[kk]);
                        ss[kk] = fma(x4[e], w.y, ss[kk]);
                    }
                }
            }
            const int last = static_cast<int>((len + 31) >> 5);
            for (; j < last; ++j) {  // the remaining whole steps and the ragged one
                const double xv = (lane + 32ll * j < len) ? __ldg(src + 32 * j) : 0.0;
                asum += xv;
                const double2* row = tab + static_cast<size_t>(j) * KB;
#pragma unroll
                for (int kk = 0; kk < KB; ++kk) {
                    const double2 w = row[kk];
                    sc[kk] = fma(xv, w.x, sc[kk]);
                    ss[kk] = fma(xv, w.y, ss[kk]);
                }
            }
            // rotate by w_k lane: cos(a + b) = ca cb - sa sb, sin(a + b) = sa cb + ca sb
#pragma unroll
            for (int kk = 0; kk < KB; ++kk) {
                const double2 w = lane_tab[kk * 32 + lane];
                const double qs = warp_sum(w.x * sc[kk] - w.y * ss[kk]);
                const double is = warp_sum(w.y * sc[kk] + w.x * ss[kk]);
                if (lane == 0 && k0 + kk < p.N) direct_store(p, v, k0 + kk, qs, is, inv_r);
            }
            if (k0 == 0) {
                asum = warp_sum(asum);
                if (lane == 0) direct_store_sum(p, v, asum, inv_r);
            }
        }
    }
}

// Two pieces per warp.  ncu puts the one-piece kernel at 87 % of the LSU data pipe: a broadcast LDS.128 still writes
// 512 B of registers per warp, ten of them per step.  A table entry fetched once here serves both pieces, which halves
// that traffic at twice the accumulators; four steps of both are loaded ahead (with two, the 12 warps per SM the
// registers allow capped the bytes in flight: 2.4 TB/s).  Pieces v and v + 1 are adjacent in the launch's numbering;
// an odd last one goes alone.  Same per-lane order of operations as the one-piece kernel: identical numbers.
template <int KB, int THREADS>
__global__ void __launch_bounds__(THREADS) demod_direct_pair_kernel(const DirectParams p) {
    extern __shared__ __align__(16) unsigned char direct_smem[];
    double2* tab = reinterpret_cast<double2*>(direct_smem);
    double2* lane_tab = tab + static_cast<size_t>(p.steps) * KB;
    const int tid = threadIdx.x, lane = tid & 31;
    const long long warp = (static_cast<long long>(blockIdx.x) * THREADS + tid) >> 5;
    const long long nwarps = (static_cast<long long>(gridDim.x) * THREADS) >> 5;
    const double inv_r = 1.0 / static_cast<double>(p.R);
    const long long npieces = p.nbuf * p.cpb;
    const long long npairs = (npieces + 1) >> 1;
    constexpr int U = 4;
    for (int k0 = 0; k0 < p.N; k0 += KB) {
        __syncthreads();
        direct_build_tables(p, k0, KB, tab, lane_tab, tid, THREADS);
        __syncthreads();
        for (long long pr = warp; pr < npairs; pr += nwarps) {
            const long long v0 = 2 * pr, v1 = (2 * pr + 1 < npieces) ? 2 * pr + 1 : 2 * pr;  // (an odd tail reads itself twice)
            long long len0, len1;
            const double* src0 = direct_piece(p, v0, len0) + lane;
            const double* src1 = direct_piece(p, v1, len1) + lane;
            double sc0[KB], ss0[KB], sc1[KB], ss1[KB];
            double asum0 = 0.0, asum1 = 0.0;
#pragma unroll
            for (int kk = 0; kk < KB; ++kk) sc0[kk] = ss0[kk] = sc1[kk] = ss1[kk] = 0.0;
            const long long lmin = len0 < len1 ? len0 : len1, lmax = len0 < len1 ? len1 : len0;
            const int full = static_cast<int>(lmin >> 5);  // steps whole in both pieces
            int j = 0;
            for (; j + U <= full; j += U) {
                double a[U], b[U];
#pragma unroll
                for (int e = 0; e < U; ++e) {
                    a[e] = __ldg(src0 + 32 * (j + e));
                    b[e] = __ldg(src1 + 32 * (j + e));
                }
#pragma unroll
                for (int e = 0; e < U; ++e) {
                    asum0 += a[e];
                    asum1 += b[e];
                    const double2* row = tab + static_cast<size_t>(j + e) * KB;
#pragma unroll
                    for (int kk = 0; kk < KB; ++kk) {
                        const double2 w = row[kk];
                        sc0[kk] = fma(a[e], w.x, sc0[kk]);
                        ss0[kk] = fma(a[e], w.y, ss0[kk]);
                        sc1[kk] = fma(b[e], w.x, sc1[kk]);
                        ss1[kk] = fma(b[e], w.y, ss1[kk]);
                    }
                }
            }
            const int last = static_cast<int>((lmax + 31) >> 5);
            for (; j < last; ++j) {  // remaining steps: whole, ragged, or past the shorter piece's end
                const double a = (lane + 32ll * j < len0) ? __ldg(src0 + 32 * j) : 0.0;
                const double b = (lane + 32ll * j < len1) ? __ldg(src1 + 32 * j) : 0.0;
                asum0 += a;
                asum1 += b;
                const double2* row = tab + static_cast<size_t>(j) * KB;
#pragma unroll
                for (int kk = 0; kk < KB; ++kk) {
                    const double2 w = row[kk];
                    sc0[kk] = fma(a, w.x, sc0[kk]);
                    ss0[kk] = fma(a, w.y, ss0[kk]);
                    sc1[kk] = fma(b, w.x, sc1[kk]);
                    ss1[kk] = fma(b, w.y, ss1[kk]);
                }
            }
#pragma unroll
            for (int kk = 0; kk < KB; ++kk) {
                const double2 w = lane_tab[kk * 32 + lane];
                const double q0 = warp_sum(w.x * sc0[kk] - w.y * ss0[kk]);
                const double i0 = warp_sum(w.y * sc0[kk] + w.x * ss0[kk]);
                const double q1 = warp_sum(w.x * sc1[kk] - w.y * ss1[kk]);
                const double i1 = warp_sum(w.y * sc1[kk] + w.x * ss1[kk]);
                if (lane == 0 && k0 + kk < p.N) {
                    direct_store(p, v0, k0 + kk, q0, i0, inv_r);
                    if (v1 != v0) direct_store(p, v1, k0 + kk, q1, i1, inv_r);
                }
            }
            if (k0 == 0) {
                asum0 = warp_sum(asum0);
                asum1 = warp_sum(asum1);
                if (lane == 0) {
                    direct_store_sum(p, v0, asum0, inv_r);
                    if (v1 != v0) direct_store_sum(p, v1, asum1, inv_r);
                }
            }
        }
    }
}

// Chunked buffers: harmonic k of buffer b is sum_c exp(i w_k c0_c) S_c with S_c the chunk's sums taken from its own
// start c0_c = c * 32 * steps -- one thread per (buffer, harmonic), the chunks in order; thread k = N sums the means.
__global__ void direct_combine_kernel(const DirectParams p) {
    const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    const int per = p.N + 1;
    if (i >= p.nbuf * per) return;
    const long long b = i / per;
    const int k = static_cast<int>(i - b * per);
    const double inv_r = 1.0 / static_cast<double>(p.R);
    const double* part = p.part + b * p.cpb * (2 * p.N + 1);
    if (k == p.N) {
        double s = 0.0;
        for (long long c = 0; c < p.cpb; ++c) s += part[c * (2 * p.N + 1) + 2 * p.N];
        p.dc[b] = s * inv_r;
        return;
    }
    const double wk = static_cast<double>(k + 1) * p.w0;
    double q = 0.0, iv = 0.0;
    for (long long c = 0; c < p.cpb; ++c) {
        double sa, ca;
        sincos(wk * static_cast<double>(c * 32ll * p.steps), &sa, &ca);
        const double qc = part[c * (2 * p.N + 1) + k], ic = part[c * (2 * p.N + 1) + p.N + k];
        q += ca * qc - sa * ic;
        iv += sa * qc + ca * ic;
    }
    p.qi[b * 2 * p.N + k] = q * inv_r;
    p.qi[b * 2 * p.N + p.N + k] = iv * inv_r;
}

}  // namespace dfk
