// Batched Levenberg-Marquardt kernels around the solver core in dfk_lm_core.cuh.
//
// Stage 1 (lm_first_kernel<G>): G lanes per fit run the first descent (fit.py:331).  A fit that ends
//   below FITOK_THRESHOLD is finished: status 0, normalised, row written.  The others park their
//   (p, ssq, steps) in the row and append their index to a retry list.
//   Cold batches (fits of a warp needing very different numbers of steps) use lm_flat_kernel instead: the same
//   driver as a per-lane state machine with immediate refill.
// Stage 2 (lm_retry_kernel / lm_retry_flat_kernel): the grid-search fallback (51 m candidates) and the second
//   descent (fit.py:336-349) for the parked fits -- a warp per fit for a handful of stragglers, a thread per fit when
//   thousands are parked.  Splitting the stages keeps the 20-40x more expensive fallback from stalling warps whose
//   other fits converged at once.
// Optional (lm_cov_kernel): the covariance of every final row, for callers that ask for uncertainties.
//
// Bessel columns live in shared memory, one column per thread (index k * blockDim.x + threadIdx.x), so
// the Miller recurrence -- evaluated redundantly by the lanes of a group -- never conflicts on banks.
#pragma once
#include "dfk_lm_core.cuh"

namespace dfk {

constexpr int kLmThreads = 128;
constexpr int kRowStride = 8;

// Where fit number f of a launch finds its data: unit u = f * step + offset indexes qi (u * 2N), dc (u) and
// rows (u * 8); the initial guess is val, or ptr[(u / div) * stride .. +3].  With div = buffers per channel
// and ptr = the row table this is "seed every buffer from its channel's buffer 0" (fitters.py:404-417);
// skip_first then leaves units with u % div == 0 (already fitted) alone.
struct GuessSrc {
    const double* ptr;  // nullptr -> val
    long long stride;   // doubles between consecutive guesses
    long long div;      // units sharing one guess (>= 1)
    int skip_first;
    double val[4];
};

struct FitMap {
    long long step, offset;  // unit u = f * step + offset indexes qi and dc
    long long row_mul;       // its result row is rows[u * row_mul]  (1 unless qi is a compacted subset)
};

// The reference's warm-start schedule (fitters.py:370-428).  Buffer 0 of a record is fitted from the user's guess;
// the M buffers after it are cut into k chunks (np.array_split: r chunks of q + 1 buffers, then k - r of q); the first
// buffer of a chunk starts from buffer 0's result, every other buffer from its predecessor's.  k = 1 is also the
// sequential mode (parallel=False).  Unit u of a launch is buffer b0 + u % bpc of channel u / bpc.
struct ChainPlan {
    long long bpc;    // buffers per channel in this launch
    long long b0;     // index within the record of the launch's first buffer (host slabs: buffers already done)
    long long first;  // first chained buffer of a record: 1 (buffer 0 is the cold fit) or 0 (the seed comes from elsewhere)
    long long q, r;   // chunk sizes (q == 0: every buffer is its own chunk)
};

DFK_HD bool chunk_start(const ChainPlan& c, long long record_buffer) {
    const long long i = record_buffer - c.first;
    if (i < 0) return true;  // the cold buffer itself
    if (c.q == 0) return true;
    const long long head = c.r * (c.q + 1);
    return i < head ? (i % (c.q + 1)) == 0 : ((i - head) % c.q) == 0;
}

DFK_D void flush_counts(const LmCounts& c, LmCounts* global, bool leader) {
    // leaders of each group hold the counts; sum over the warp, one atomic per counter per warp
    unsigned long long v[5] = {leader ? c.n_state : 0ull, leader ? c.n_ssq : 0ull, leader ? c.n_solve : 0ull,
                               leader ? c.n_grid : 0ull, leader ? c.n_bessel_steps : 0ull};
#pragma unroll
    for (int i = 0; i < 5; ++i) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v[i] += __shfl_xor_sync(0xffffffffu, v[i], o);
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(&global->n_state, v[0]);
        atomicAdd(&global->n_ssq, v[1]);
        atomicAdd(&global->n_solve, v[2]);
        atomicAdd(&global->n_grid, v[3]);
        atomicAdd(&global->n_bessel_steps, v[4]);
    }
}

// TPB: threads per block.  Large batches use kLmThreads; a handful of fits (the cold seed fits that overlap the
// demodulation) use one-warp blocks so that they spread over all SMs instead of loading a few of them.
template <int G, int MINB, int TPB>
__global__ void __launch_bounds__(TPB, MINB) lm_first_kernel(const double* __restrict__ qi, long long nfit, FitMap map,
                                                              int N, GuessSrc guess, const double* __restrict__ dc,
                                                              LmOpts o, double* rows,
                                                              int* __restrict__ retry_list, int* __restrict__ retry_count,
                                                              LmCounts* __restrict__ counts,
                                                              int* __restrict__ parked_flags) {
    extern __shared__ double bes_smem[];
    constexpr int kFitsPerBlock = TPB / G;
    const int group = threadIdx.x / G;
    const int rank = threadIdx.x & (G - 1);
    double* bes = bes_smem + threadIdx.x;
    LmCounts cnt = {};
    const long long nblocks_work = (nfit + kFitsPerBlock - 1) / kFitsPerBlock;
    for (long long blk = blockIdx.x; blk < nblocks_work; blk += gridDim.x) {
        const long long f = blk * kFitsPerBlock + group;
        // groups past the end still walk the code with fit 0's data so that full-mask shuffles of
        // G == 32 stay convergent; they write nothing.
        const long long u = (f < nfit ? f : 0) * map.step + map.offset;
        const bool live = f < nfit && !(guess.skip_first && (u % guess.div) == 0);
        const double* q = qi + u * 2 * N;
        double p[4];
        if (guess.ptr) {
            const double* g = guess.ptr + (u / guess.div) * guess.stride;
            p[0] = g[0]; p[1] = g[1]; p[2] = g[2]; p[3] = g[3];
        } else {
            p[0] = guess.val[0]; p[1] = guess.val[1]; p[2] = guess.val[2]; p[3] = guess.val[3];
        }
        int steps = 0;
        LmCounts local = {};
        const double ssq = lm_descend<G>(N, q, 1, bes, TPB, o, p, steps, local);
        if (live) {
            cnt.n_state += local.n_state; cnt.n_ssq += local.n_ssq; cnt.n_solve += local.n_solve;
            cnt.n_bessel_steps += local.n_bessel_steps;
        }
        if (live && rank == 0) {
            double* row = rows + u * map.row_mul * kRowStride;
            const bool converged = ssq < o.fitok_threshold;
            // Chain schedule: a descent that converged with a < 0 or m < 0 took a detour the chain, starting next to
            // the solution, does not take -- and the reference's sign normalisation (fit.py:352-357) is not a symmetry
            // of the model (the exact one is (a, -m, phi) = (a, m, -phi)), so the two would report different phi.
            // Such fits are parked too (flag 2) and refitted from their predecessor.
            const bool flipped = parked_flags && (p[0] < 0.0 || p[1] < 0.0);
            const bool done = converged && !flipped;
            if (done) normalise_params(p);
            row[0] = p[0]; row[1] = p[1]; row[2] = p[2]; row[3] = p[3];
            row[4] = dc ? dc[u] : 0.0;
            row[5] = ssq;
            row[6] = done ? 0.0 : -1.0;  // -1: parked for the retry stage
            row[7] = static_cast<double>(steps);
            if (parked_flags) {  // chain schedule: lm_chain_kernel walks the parked runs
                parked_flags[u] = done ? 0 : (converged ? 2 : 1);
            } else if (!done) {
                retry_list[atomicAdd(retry_count, 1)] = static_cast<int>(u);
            }
        }
    }
    flush_counts(cnt, counts, rank == 0);
}

// Second stage of the chain schedule.  The first stage started every buffer from its chunk's seed (buffer 0's
// result); on a stationary record that converges everywhere and this kernel finds nothing to do.  Where the
// parameters drift along the record the first descent of later buffers fails (parked), while the reference, whose
// warm start moves along with the record, keeps converging.  Here a warp takes each maximal run of parked buffers
// inside a chunk and walks it in order, fitting each buffer from its predecessor's final result exactly as
// fitters.py:42-58 does (first descent, grid fallback if that fails, fit.py:322-362).  A parked buffer that opens a
// chunk already had the reference's start (the chunk seed), so it continues with the fallback alone.
// Buffers that converged in the first stage are taken to be where the chain would have put them: the same minimum,
// reached from a different start (the schedules agree to <= 1e-10 on such buffers, DESIGN.md section 2).
__global__ void __launch_bounds__(kLmThreads) lm_chain_kernel(const double* __restrict__ qi, long long nfit, int N,
                                                              LmOpts o, ChainPlan plan, double* rows,
                                                              const int* __restrict__ parked,
                                                              LmCounts* __restrict__ counts) {
    extern __shared__ double bes_smem[];
    double* bes = bes_smem + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const long long warp = (static_cast<long long>(blockIdx.x) * kLmThreads + threadIdx.x) >> 5;
    const long long nwarps = (static_cast<long long>(gridDim.x) * kLmThreads) >> 5;
    LmCounts cnt = {};
    for (long long base = warp * 32; base < nfit; base += nwarps * 32) {
        const long long u = base + lane;
        bool opens = false;
        if (u < nfit && parked[u]) {
            const long long b = u % plan.bpc;
            opens = b == 0 || chunk_start(plan, plan.b0 + b) || !parked[u - 1];
        }
        unsigned todo = __ballot_sync(0xffffffffu, opens);
        while (todo) {
            const int l = __ffs(todo) - 1;
            todo &= todo - 1;
            long long v = base + l;  // first buffer of the run
            double p[4];
            bool have_prev = false;
            while (true) {
                const long long b = v % plan.bpc;
                double* row = rows + v * kRowStride;
                const double* q = qi + v * 2 * N;
                const bool start = chunk_start(plan, plan.b0 + b);
                double ssq;
                int steps, status;
                __syncwarp();
                if (start) {  // the first descent from the chunk seed was stage 1, the reference's own start
                    p[0] = row[0]; p[1] = row[1]; p[2] = row[2]; p[3] = row[3];
                    ssq = row[5];
                    steps = static_cast<int>(row[7]);
                    // flag 2: it converged (with a sign to normalise); flag 1: continue with the fallback
                    status = parked[v] == 2 ? 0 : retry_fit<32>(N, q, 1, bes, kLmThreads, o, p, ssq, steps, cnt);
                    normalise_params(p);
                } else {
                    if (!have_prev) {
                        const double* prev = row - kRowStride;  // final: it converged in stage 1 or belongs to an earlier launch
                        p[0] = prev[0]; p[1] = prev[1]; p[2] = prev[2]; p[3] = prev[3];
                    }
                    status = fit_full<32>(N, q, 1, bes, kLmThreads, o, p, ssq, steps, cnt);
                }
                if (lane == 0) {
                    row[0] = p[0]; row[1] = p[1]; row[2] = p[2]; row[3] = p[3];
                    row[5] = ssq;
                    row[6] = static_cast<double>(status);
                    row[7] = static_cast<double>(steps);
                }
                have_prev = true;
                ++v;
                if (v >= nfit || (v % plan.bpc) == 0 || !parked[v] || chunk_start(plan, plan.b0 + v % plan.bpc)) break;
            }
        }
    }
    flush_counts(cnt, counts, lane == 0);
}

// Bulk variant of stage 1 for one thread per fit: the LM driver of fit.py:208-258 flattened into a per-lane state
// machine.  Every trip of the loop does the same thing for every lane -- solve for the current damping, Miller
// recurrence at the trial m, one model+Jacobian evaluation there, accept / reject bookkeeping -- and a lane whose
// fit has ended takes the next fit at once, so the lanes of a warp stay busy although their fits need different
// numbers of steps (in lm_first_kernel<1> only 21 of 32 lanes are active on average).  An accepted trial point is
// where the reference recomputes coeffs (fit.py:250-251); evaluating the Jacobian with every trial makes that
// second pass unnecessary.  The decisions (first strictly better damping of the fixed ladder, the stopping rule, the
// step cap) are those of the reference, so flags and results agree with lm_first_kernel.
// Normal equations of the current point live in shared memory (12 doubles per thread) to keep registers for the
// evaluation.
constexpr int kNeDoubles = 12;

DFK_D void ne_store(double* s, const NormalEq& n, int stride) {
    s[0 * stride] = n.a00; s[1 * stride] = n.a01; s[2 * stride] = n.a02; s[3 * stride] = n.a11;
    s[4 * stride] = n.a12; s[5 * stride] = n.a22; s[6 * stride] = n.a33; s[7 * stride] = n.g0;
    s[8 * stride] = n.g1; s[9 * stride] = n.g2; s[10 * stride] = n.g3; s[11 * stride] = n.ssq;
}
DFK_D void ne_load(const double* s, NormalEq& n, int stride) {
    n.a00 = s[0 * stride]; n.a01 = s[1 * stride]; n.a02 = s[2 * stride]; n.a11 = s[3 * stride];
    n.a12 = s[4 * stride]; n.a22 = s[5 * stride]; n.a33 = s[6 * stride]; n.g0 = s[7 * stride];
    n.g1 = s[8 * stride]; n.g2 = s[9 * stride]; n.g3 = s[10 * stride]; n.ssq = s[11 * stride];
}

// One trip of the per-lane state machine: returns true when the fit has ended (p, ssq, steps final).
struct FlatState {
    double p[4];
    double ssq;
    int lam;  // -1: evaluate the starting point; 0..7: position in the damping ladder
    int steps;
    double m_held;  // m the Bessel column currently holds (NaN: none): a bit-identical trial m reuses the column
};

DFK_D bool flat_step(int N, const double* q, double* bes, double* nes, const LmOpts& o, FlatState& st, LmCounts& cnt) {
    double dp[4] = {0.0, 0.0, 0.0, 0.0};
    bool skip = false;
    if (st.lam >= 0) {
        NormalEq ne;
        ne_load(nes, ne, kLmThreads);
        damped_solve(ne, lambda_of(st.lam), dp);
        cnt.n_solve++;
        skip = sqrt(dp[0] * dp[0] + dp[1] * dp[1] + dp[2] * dp[2] + dp[3] * dp[3]) < 1e-15;  // fit.py:230
    }
    const double pt[4] = {st.p[0] + dp[0], st.p[1] + dp[1], st.p[2] + dp[2], st.p[3] + dp[3]};
    NormalEq nt;
    if (!skip && !(pt[1] == st.m_held)) {
        cnt.n_bessel_steps += bessel_j_upto(pt[1], N + 1, bes, kLmThreads);
        st.m_held = pt[1];
    }
    eval_state<1>(N, q, 1, bes, kLmThreads, pt, nt);
    if (st.lam < 0) {
        cnt.n_state++;
        ne_store(nes, nt, kLmThreads);
        st.ssq = nt.ssq;
        st.lam = 0;
        return o.max_steps <= 0;
    }
    if (!skip) cnt.n_ssq++;
    if (!skip && nt.ssq < st.ssq) {  // first strictly better damping wins (fit.py:240-243)
        const double moved = sqrt(dp[0] * dp[0] + dp[1] * dp[1] + dp[2] * dp[2] + dp[3] * dp[3]);
        st.p[0] = pt[0]; st.p[1] = pt[1]; st.p[2] = pt[2]; st.p[3] = pt[3];
        ne_store(nes, nt, kLmThreads);
        st.ssq = nt.ssq;
        cnt.n_state++;
        ++st.steps;
        st.lam = 0;
        // fit.py:255 compares the accepted ssq with its own recomputation: 0 < conv_improve unless it is <= 0
        return ((0.0 < o.conv_improve) && moved < o.conv_param) || st.steps >= o.max_steps;
    }
    return ++st.lam == 8;  // no damping improved (fit.py:246)
}

template <int MINB>
__global__ void __launch_bounds__(kLmThreads, MINB) lm_flat_kernel(const double* __restrict__ qi, long long nfit, FitMap map,
                                                                   int N, GuessSrc guess, const double* __restrict__ dc,
                                                                   LmOpts o, double* rows, int* __restrict__ retry_list,
                                                                   int* __restrict__ retry_count,
                                                                   LmCounts* __restrict__ counts) {
    extern __shared__ double lm_smem[];
    double* bes = lm_smem + threadIdx.x;                                   // (N + 2) x kLmThreads
    double* nes = lm_smem + (N + 2) * kLmThreads + threadIdx.x;            // kNeDoubles x kLmThreads
    const long long stride = static_cast<long long>(gridDim.x) * kLmThreads;
    long long f = static_cast<long long>(blockIdx.x) * kLmThreads + threadIdx.x;
    LmCounts cnt = {};
    FlatState st = {{0.0, 0.0, 0.0, 0.0}, 0.0, -1, 0, 0.0};
    const double* q = qi;
    long long u = 0;
    bool active = false;
    // fetch the next fit this lane has to do (skipping units that are already fitted)
    auto fetch = [&]() {
        active = false;
        while (f < nfit) {
            u = f * map.step + map.offset;
            f += stride;
            if (guess.skip_first && (u % guess.div) == 0) continue;
            active = true;
            break;
        }
        if (!active) return;
        q = qi + u * 2 * N;
        if (guess.ptr) {
            const double* g = guess.ptr + (guess.div == 1 ? u : u / guess.div) * guess.stride;
            st.p[0] = g[0]; st.p[1] = g[1]; st.p[2] = g[2]; st.p[3] = g[3];
        } else {
            st.p[0] = guess.val[0]; st.p[1] = guess.val[1]; st.p[2] = guess.val[2]; st.p[3] = guess.val[3];
        }
        st.lam = -1;
        st.steps = 0;
        st.m_held = __longlong_as_double(0x7ff8000000000000ll);  // NaN: column not built yet
    };
    fetch();
    while (active) {
        if (flat_step(N, q, bes, nes, o, st, cnt)) {
            double* row = rows + u * map.row_mul * kRowStride;
            const bool done = st.ssq < o.fitok_threshold;
            if (done) normalise_params(st.p);
            row[0] = st.p[0]; row[1] = st.p[1]; row[2] = st.p[2]; row[3] = st.p[3];
            row[4] = dc ? dc[u] : 0.0;
            row[5] = st.ssq;
            row[6] = done ? 0.0 : -1.0;
            row[7] = static_cast<double>(st.steps);
            if (!done) retry_list[atomicAdd(retry_count, 1)] = static_cast<int>(u);
            fetch();
        }
    }
    flush_counts(cnt, counts, true);
}

// Retry stage for MANY parked fits (a sweep cold-started far from the truth parks most of them): one thread per
// fit.  The warp-per-fit retry kernel below spends 32 lanes on one fit -- right for a handful of stragglers, but
// every lane then repeats the same Miller recurrence, so its cost per fit is that of 32 independent fits.  Here the
// 51-point grid search runs in lock step (the same work for every lane) and the second descent through the per-lane
// state machine; the two kernels split the work by the number of parked fits (kFlatRetryMin).
constexpr int kFlatRetryMin = 4096;

__global__ void __launch_bounds__(kLmThreads) lm_retry_flat_kernel(const double* __restrict__ qi, int N, LmOpts o,
                                                                   long long row_mul, double* __restrict__ rows,
                                                                   const int* __restrict__ retry_list,
                                                                   const int* __restrict__ retry_count,
                                                                   LmCounts* __restrict__ counts) {
    extern __shared__ double lm_smem[];
    double* bes = lm_smem + threadIdx.x;
    double* nes = lm_smem + (N + 2) * kLmThreads + threadIdx.x;
    const int n = *retry_count;
    if (n < kFlatRetryMin) return;
    LmCounts cnt = {};
    for (long long i = static_cast<long long>(blockIdx.x) * kLmThreads + threadIdx.x; i < n;
         i += static_cast<long long>(gridDim.x) * kLmThreads) {
        const long long u = retry_list[i];
        double* row = rows + u * row_mul * kRowStride;
        const double* q = qi + u * 2 * N;
        double p1[4] = {row[0], row[1], row[2], row[3]};
        double ssq1 = row[5];
        int steps1 = static_cast<int>(row[7]);
        FlatState st = {{0.0, 0.0, 0.0, 0.0}, 0.0, -1, 0, __longlong_as_double(0x7ff8000000000000ll)};
        grid_seed<1>(N, q, 1, bes, kLmThreads, o, st.p, cnt);
        cnt.n_grid++;
        if (st.p[0] != 0.0 || st.p[1] != 0.0 || st.p[2] != 0.0 || st.p[3] != 0.0) {  // np.any (NaN counts as true)
            while (!flat_step(N, q, bes, nes, o, st, cnt)) {
            }
            if (st.ssq < ssq1) {  // fit.py:345-347: keep the second descent only if it is better
                p1[0] = st.p[0]; p1[1] = st.p[1]; p1[2] = st.p[2]; p1[3] = st.p[3];
                ssq1 = st.ssq;
                steps1 = st.steps;
            }
        }
        normalise_params(p1);
        row[0] = p1[0]; row[1] = p1[1]; row[2] = p1[2]; row[3] = p1[3];
        row[5] = ssq1;
        row[6] = ssq1 < o.fitok_threshold ? 1.0 : 2.0;
        row[7] = static_cast<double>(steps1);
    }
    flush_counts(cnt, counts, true);
}

// retry_list holds unit indices (into qi and rows alike).
__global__ void __launch_bounds__(kLmThreads) lm_retry_kernel(const double* __restrict__ qi, int N, LmOpts o,
                                                              long long row_mul, double* __restrict__ rows,
                                                              const int* __restrict__ retry_list,
                                                              const int* __restrict__ retry_count,
                                                              LmCounts* __restrict__ counts) {
    extern __shared__ double bes_smem[];
    double* bes = bes_smem + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const int warps_per_block = kLmThreads / 32;
    const int n = *retry_count;
    if (n >= kFlatRetryMin) return;  // lm_retry_flat_kernel's share
    LmCounts cnt = {};
    for (int i = blockIdx.x * warps_per_block + (threadIdx.x >> 5); i < n; i += gridDim.x * warps_per_block) {
        const long long f = retry_list[i];
        double* row = rows + f * row_mul * kRowStride;
        const double* q = qi + f * 2 * N;
        double p[4] = {row[0], row[1], row[2], row[3]};
        double ssq = row[5];
        int steps = static_cast<int>(row[7]);
        __syncwarp();
        const int status = retry_fit<32>(N, q, 1, bes, kLmThreads, o, p, ssq, steps, cnt);
        normalise_params(p);
        if (lane == 0) {
            row[0] = p[0]; row[1] = p[1]; row[2] = p[2]; row[3] = p[3];
            row[5] = ssq;
            row[6] = static_cast<double>(status);
            row[7] = static_cast<double>(steps);
        }
        __syncwarp();
    }
    flush_counts(cnt, counts, lane == 0);
}

// Covariance of every fit's reported parameters (fit_covariance): one thread per fit, its Bessel column in shared
// memory ((N + 2) x kLmThreads doubles, as lm_retry_flat_kernel).  Reads the final rows; touches no LM counter.
__global__ void __launch_bounds__(kLmThreads) lm_cov_kernel(const double* __restrict__ qi, long long nfit, int N,
                                                            const double* __restrict__ rows, double* __restrict__ cov) {
    extern __shared__ double bes_smem[];
    double* bes = bes_smem + threadIdx.x;
    for (long long f = static_cast<long long>(blockIdx.x) * kLmThreads + threadIdx.x; f < nfit;
         f += static_cast<long long>(gridDim.x) * kLmThreads)
        fit_covariance(N, qi + f * 2 * N, 1, bes, kLmThreads, rows + f * kRowStride, cov + f * kCovStride);
}

// J_0..J_nmax of n arguments, one thread each (testing hook behind dfk_bessel_dev).
__global__ void bessel_kernel(const double* __restrict__ x, long long n, int nmax, double* __restrict__ out) {
    const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (i < n) bessel_j_upto(x[i], nmax, out + i * (nmax + 1), 1);
}

// FP64 FMA throughput probe: 8 independent DFMA chains per thread (the denominator bench.py quotes the LM
// kernel's fp64 rate against; MEASURED_PEAKS.json has no fp64 figure).
__global__ void __launch_bounds__(256) fp64_probe_kernel(int iters, double seed, double* __restrict__ sink) {
    double a[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) a[i] = seed + 1e-3 * (threadIdx.x + i);
    const double m = 1.0 - 1e-9, c = 1e-9;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 8; ++i) a[i] = fma(a[i], m, c);
    }
    double t = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) t += a[i];
    if (t == 123.456) sink[0] = t;  // keeps the chains alive without writing in practice
}

}  // namespace dfk
