// C ABI of the B200-native DFMI readout path (declared in include/dfk_b200.h).
// CUDA only: every entry point fails with DFK_ERR_CUDA when no usable device exists.
#include "../../include/dfk_b200.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <mutex>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <new>
#include <thread>
#include <vector>

#include "dfk_demod.cuh"
#include "dfk_ekf_kernels.cuh"
#include "dfk_ekf_smooth.cuh"
#include "dfk_lm_kernels.cuh"
#include "dfk_synth.cuh"
#include "dfk_sweep.cuh"

#include "dfk_host.h"

namespace {

// Development overrides of kernel choice and geometry (benchmarks/tune.py, the kernel A/B tests).  They are set
// by an explicit call, dfk_dev_set("DFK_NO_TILE", 1); the library never reads the environment, so nothing outside
// the calling program can change which kernel runs.
struct DevOverride {
    char name[32];
    int value;
};
DevOverride g_dev[16];
std::atomic<int> g_dev_count{0};
std::mutex g_dev_mutex;

int dev_int(const char* name, int fallback) {
    const int n = g_dev_count.load(std::memory_order_acquire);
    for (int i = 0; i < n; ++i)
        if (std::strcmp(g_dev[i].name, name) == 0) return g_dev[i].value;
    return fallback;
}

dfk::LmOpts to_opts(const dfk_lm_opts* o) {
    dfk_lm_opts d;
    if (!o) {
        dfk_default_lm_opts(&d);
        o = &d;
    }
    dfk::LmOpts r;
    r.max_steps = o->max_lma_steps;
    r.conv_improve = o->conv_improve;
    r.conv_param = o->conv_param;
    r.fitok_threshold = o->fitok_threshold;
    r.grid_min = o->m_grid_min;
    r.grid_max = o->m_grid_max;
    r.grid_step = o->m_grid_step;
    r.bessel_thr = o->bessel_amp_threshold;
    r.sincos_thr = o->sincos_amp_threshold;
    return r;
}

// Every kernel launch of this file but the FP64 probe's: raise the kernel's dynamic shared-memory limit to what this
// launch uses, launch it on st, count it (dfk_launch_count) and report a launch error.
template <class... Params, class... Args>
int launch_kernel(dfk_ctx* ctx, void (*kernel)(Params...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                  const Args&... args) {
    if (smem) DFK_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    kernel<<<grid, block, smem, st>>>(args...);
    ctx->launches++;
    DFK_CUDA(cudaGetLastError());
    return DFK_OK;
}

// The deepest ring of 2..deepest stages whose shared memory, smem_of(stages), fits one CTA less `reserve` bytes:
// its depth, or 0 when not even two stages fit; its size goes to *smem.
template <class SmemOf>
int ring_depth(const dfk_ctx* ctx, int deepest, size_t reserve, SmemOf smem_of, size_t* smem) {
    for (int nst = deepest; nst >= 2; --nst) {
        *smem = smem_of(nst);
        if (*smem <= static_cast<size_t>(ctx->max_smem_optin) - reserve) return nst;
    }
    return 0;
}

// ---- demodulation -------------------------------------------------------------------------------
// Shared memory left free on every SM next to a persistent demod CTA so that one block of the cold seed fits
// (Bessel columns: (N+2) x 128 doubles) can co-reside and overlap with it; given up when it would cost the
// ring too much (many harmonics).
size_t seed_fit_reserve(int N) {
    const size_t need = static_cast<size_t>(N + 2) * dfk::kLmThreads * sizeof(double) + 2048;
    return need <= 24 * 1024 ? need : 0;
}

// The lock-in plan of R-sample buffers; the development override DFK_FOLD_DRIFT forces the drift term on or off.
dfk::DemodPlan demod_plan(int64_t R, double w0, int N) {
    dfk::DemodPlan pl = dfk::make_demod_plan(R, w0, N);
    const int forced = dev_int("DFK_FOLD_DRIFT", -1);
    if (forced >= 0) pl.drift = forced != 0;
    return pl;
}

// The fields of the fold kernels' parameters that do not depend on the launch geometry (pps, nstages).
dfk::FoldParams fold_params(const dfk::DemodPlan& pl, const double* x, int64_t nbuf, int64_t bpc, int64_t ld_c, int64_t R,
                            int64_t P, int N, double* qi, double* dc) {
    dfk::FoldParams p;
    p.x = x;
    p.qi = qi;
    p.dc = dc;
    p.nbuf = nbuf;
    p.bpc = bpc;
    p.ld_c = ld_c;
    p.R = static_cast<int>(R);
    p.P = static_cast<int>(P);
    p.periods = static_cast<int>(pl.periods);
    p.N = N;
    p.kmul = pl.kmul;
    for (int k = 0; k < dfk::kMaxHarmonics; ++k) p.delta[k] = pl.delta[k];
    return p;
}

struct FoldGeometry {
    int pps, nstages;
    size_t smem;
    int ctas_per_sm;
};

bool fold_geometry(const dfk_ctx* ctx, const dfk::DemodPlan& pl, int N, size_t reserve, FoldGeometry* g) {
    const int P = static_cast<int>(pl.P);
    // development overrides (tuning runs only): DFK_FOLD_STAGE_BYTES, DFK_FOLD_NSTAGES, DFK_FOLD_CTAS
    const int env_stage = dev_int("DFK_FOLD_STAGE_BYTES", 0), env_nst = dev_int("DFK_FOLD_NSTAGES", 0),
              env_ctas = dev_int("DFK_FOLD_CTAS", 0);
    int pps = (env_stage > 0 ? env_stage : dfk::kFoldStageBytes) / (P * 8);
    if (pps < 1) pps = 1;
    if (pps > pl.periods) pps = static_cast<int>(pl.periods);
    if (env_nst > 0 || env_ctas > 0) {
        const int ctas = env_ctas > 0 ? env_ctas : 2, nst = env_nst > 0 ? env_nst : 4;
        const dfk::FoldSmem L = dfk::fold_smem_layout(P, pps, nst, N, pl.drift);
        if (L.total <= static_cast<size_t>(ctx->max_smem_optin) &&
            static_cast<size_t>(ctas) * (L.total + 1024) <= static_cast<size_t>(ctx->smem_per_sm)) {
            g->pps = pps;
            g->nstages = nst;
            g->smem = L.total;
            g->ctas_per_sm = ctas;
            return true;
        }
        return false;  // the override does not fit: take the direct kernel rather than mislead a sweep
    }
    // Measured on B200 (profiles/r01_tune_demod_*.jsonl): throughput follows the bytes in flight per SM and
    // prefers few large stages (fewer mbarrier round trips), saturating near 7.3 TB/s from ~130 kB up.
    // Candidates: 1 or 2 resident CTAs, stages of 16..64 kB of whole periods, rings of 2..6 stages; take the
    // most bytes in flight, then the larger stage, then two CTAs (one folds while the other takes harmonics).
    const int stage_targets[] = {65536, 40960, 32768, 24576, 16384};
    size_t best_flight = 0;
    int best_stage = 0;
    bool found = false;
    for (int ctas = 2; ctas >= 1; --ctas) {
        const size_t budget = ctas == 2 ? (static_cast<size_t>(ctx->smem_per_sm) - reserve) / 2 - 1024
                                        : static_cast<size_t>(ctx->max_smem_optin) - reserve;
        for (int target : stage_targets) {
            int q = target / (P * 8);
            if (q < 1) q = 1;
            if (q > pl.periods) q = static_cast<int>(pl.periods);
            for (int nst = 6; nst >= 2; --nst) {
                const dfk::FoldSmem L = dfk::fold_smem_layout(P, q, nst, N, pl.drift);
                if (L.total > budget) continue;
                const int stage_bytes = q * P * 8;
                const size_t flight = static_cast<size_t>(ctas) * nst * stage_bytes;
                if (!found || flight > best_flight || (flight == best_flight && stage_bytes > best_stage)) {
                    found = true;
                    best_flight = flight;
                    best_stage = stage_bytes;
                    g->pps = q;
                    g->nstages = nst;
                    g->smem = L.total;
                    g->ctas_per_sm = ctas;
                }
                break;  // deeper rings of this shape fit less
            }
        }
    }
    return found;
}

// One period per buffer (R == P <= 256, P % 4 == 0, no drift term): the quarter-wave kernel.  Returns 1 if it
// launched, 0 if the geometry does not fit it, < 0 on error.
int try_launch_period(dfk_ctx* ctx, const dfk::DemodPlan& pl, const double* x, int64_t nbuf, int32_t N, double* qi,
                      double* dc, size_t reserve, cudaStream_t st) {
    if (pl.periods != 1 || pl.kmul != 1 || pl.drift || pl.P > dfk::kTileMaxPeriod || (pl.P % 4) != 0) return 0;
    if (reinterpret_cast<uintptr_t>(qi) & 15u) return 0;  // the kernel stores harmonic vectors 128 bits at a time
    const int P = static_cast<int>(pl.P);
    size_t smem = 0;
    // a stage per consumer warp: measured flat from 6 stages up
    const int nst = ring_depth(ctx, dev_int("DFK_PERIOD_NSTAGES", dfk::kPeriodWarps), reserve,
                               [&](int n) { return dfk::period_smem_layout(P, N, n).total; }, &smem);
    if (nst == 0) return 0;
    const dfk::PeriodParams p = {x, qi, dc, nbuf, P, N, nst};
    const int64_t ngroups = (nbuf + dfk::kPeriodNbw - 1) / dfk::kPeriodNbw;
    const int grid = static_cast<int>(std::min<int64_t>(ngroups, ctx->sm_count));
    const int rc =
        launch_kernel(ctx, dfk::demod_period_kernel<dfk::kPeriodWarps>, grid, (dfk::kPeriodWarps + 1) * 32, smem, st, p);
    return rc ? rc : 1;
}

// Short periods (P <= 256) with contiguous buffers: the barrier-free tile kernel.  Returns 1 if it launched,
// 0 if the geometry does not fit it, < 0 on error.
int try_launch_tile(dfk_ctx* ctx, const dfk::DemodPlan& pl, const double* x, int64_t nbuf, int64_t R, int32_t N,
                    double* qi, double* dc, size_t reserve, cudaStream_t st) {
    if (pl.P > dfk::kTileMaxPeriod || dev_int("DFK_NO_TILE", 0)) return 0;
    const int P = static_cast<int>(pl.P), n = static_cast<int>(pl.periods);
    int nbw = 8;
    while (nbw > 1 && static_cast<int64_t>(nbw) * R * 8 > dfk::kTileStageBytes) nbw >>= 1;
    int pps = dfk::kTileStageBytes / (P * 8);
    if (pps < 1) pps = 1;
    if (pps > nbw * n) pps = nbw * n;
    size_t smem = 0;
    const int nst = ring_depth(ctx, dev_int("DFK_TILE_NSTAGES", 12), reserve,
                               [&](int s) { return dfk::tile_smem_layout(P, N, nbw, pps, s, pl.drift).total; }, &smem);
    if (nst == 0) return 0;
    dfk::TileParams p;
    p.x = x;
    p.qi = qi;
    p.dc = dc;
    p.nbuf = nbuf;
    p.R = static_cast<int>(R);
    p.P = P;
    p.periods = n;
    p.N = N;
    p.kmul = pl.kmul;
    p.pps = pps;
    p.cpg = (nbw * n + pps - 1) / pps;
    p.nstages = nst;
    for (int k = 0; k < dfk::kMaxHarmonics; ++k) p.delta[k] = pl.delta[k];
    const int64_t ngroups = (nbuf + nbw - 1) / nbw;
    const int grid = static_cast<int>(std::min<int64_t>(ngroups, ctx->sm_count));
    auto tile = [&](auto kernel) { return launch_kernel(ctx, kernel, grid, dfk::kFoldThreads, smem, st, p); };
    int rc;
    if (pl.drift) {
        switch (nbw) {
            case 8: rc = tile(dfk::demod_tile_kernel<true, 8>); break;
            case 4: rc = tile(dfk::demod_tile_kernel<true, 4>); break;
            case 2: rc = tile(dfk::demod_tile_kernel<true, 2>); break;
            default: rc = tile(dfk::demod_tile_kernel<true, 1>); break;
        }
    } else {
        switch (nbw) {
            case 8: rc = tile(dfk::demod_tile_kernel<false, 8>); break;
            case 4: rc = tile(dfk::demod_tile_kernel<false, 4>); break;
            case 2: rc = tile(dfk::demod_tile_kernel<false, 2>); break;
            default: rc = tile(dfk::demod_tile_kernel<false, 1>); break;
        }
    }
    return rc ? rc : 1;
}

// Fold lengths beyond the register kernel: column chunks of 2048, 32 kB stages (two period slices), as deep a ring as
// one CTA per SM holds.  STORE: the folded arrays go to p.qi and p.dc instead of the harmonics (time-major records).
template <bool STORE>
int launch_fold_long(dfk_ctx* ctx, dfk::FoldParams p, bool drift, size_t reserve, cudaStream_t st) {
    p.pps = std::min(2, p.periods);
    size_t smem = 0;
    p.nstages = ring_depth(ctx, 6, reserve, [&](int n) { return dfk::fold_long_smem_layout(p.pps, n, p.N, drift).total; },
                           &smem);
    if (p.nstages == 0) return fail(DFK_ERR_ARG, "no shared memory for the long-period fold");
    const int grid = static_cast<int>(std::min<int64_t>(p.nbuf, ctx->sm_count));
    return drift ? launch_kernel(ctx, dfk::demod_fold_long_kernel<true, STORE>, grid, dfk::kFoldThreads, smem, st, p)
                 : launch_kernel(ctx, dfk::demod_fold_long_kernel<false, STORE>, grid, dfk::kFoldThreads, smem, st, p);
}

// nbuf buffers in channel records of bpc buffers each, records ld_c samples apart
// leave_room: keep enough shared memory free on each SM for a block of the seed fits that run beside this launch
// Records that do not fold (dfk_demod.cuh, demod_direct_kernel): a warp per piece (two when there are enough), 8 to 16
// harmonics per pass; a piece is the buffer when a CTA's table can hold its steps, else a 16 384-sample chunk of it.
template <int KB, int THREADS>
int launch_direct_one(dfk_ctx* ctx, const dfk::DirectParams& q, size_t smem, int per_sm, cudaStream_t st) {
    const int64_t warps_per_cta = THREADS / 32, npieces = q.nbuf * q.cpb;
    const int grid = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>((npieces + warps_per_cta - 1) / warps_per_cta,
                                                                            static_cast<int64_t>(ctx->sm_count) * per_sm)));
    return launch_kernel(ctx, dfk::demod_direct_kernel<KB, THREADS>, grid, THREADS, smem, st, q);
}

template <int KB, int THREADS>
int launch_direct_pair(dfk_ctx* ctx, const dfk::DirectParams& q, size_t smem, cudaStream_t st) {
    const int64_t warps_per_cta = THREADS / 32, npairs = (q.nbuf * q.cpb + 1) / 2;
    const int grid = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>((npairs + warps_per_cta - 1) / warps_per_cta,
                                                                            static_cast<int64_t>(ctx->sm_count))));
    return launch_kernel(ctx, dfk::demod_direct_pair_kernel<KB, THREADS>, grid, THREADS, smem, st, q);
}

template <int KB>
int launch_direct_t(dfk_ctx* ctx, const dfk::DirectParams& q, cudaStream_t st) {
    const size_t smem = (static_cast<size_t>(q.steps) * KB + static_cast<size_t>(KB) * 32) * sizeof(double2);
    // enough pieces to give every warp of the GPU a pair: two per warp (registers: one CTA of 12 warps per SM)
    if constexpr (KB <= 10) {
        if (q.nbuf * q.cpb >= 2 * 12 * static_cast<int64_t>(ctx->sm_count) && dev_int("DFK_DIRECT_PAIR", 1))
            return launch_direct_pair<KB, 384>(ctx, q, smem, st);
    }
    const int per_sm = static_cast<int>(std::max<size_t>(1, std::min<size_t>(4, static_cast<size_t>(ctx->smem_per_sm) / (smem + 1024))));
    // one CTA per SM (a long table): 512 threads, which the 128 registers of the narrower builds allow
    if constexpr (KB <= 12) {
        if (per_sm == 1) return launch_direct_one<KB, 512>(ctx, q, smem, per_sm, st);
    }
    return launch_direct_one<KB, dfk::kDirectThreads>(ctx, q, smem, per_sm, st);
}

int launch_direct(dfk_ctx* ctx, const double* x, int64_t nbuf, int64_t bpc, int64_t ld_c, int64_t R, int N, double w0,
                  double* qi, double* dc, cudaStream_t st) {
    dfk::DirectParams p = {x, nbuf, bpc, ld_c, R, N, w0, qi, dc, 0, 1, nullptr};
    const int64_t need = (R + 31) / 32;  // steps that cover a buffer
    const size_t budget = static_cast<size_t>(ctx->max_smem_optin) - 2048;
    // harmonics per pass: the narrow builds run twice as fast per pass as the 16-wide one (registers: one CTA of eight
    // warps per SM), so beyond 16 harmonics several passes of 10 or 12 beat fewer of 16
    int kb = N <= 8 ? 8 : (N <= 10 ? 10 : (N <= 12 ? 12 : 16));
    if (N > 16) kb = (N + 11) / 12 < (N + 9) / 10 ? 12 : 10;
    const int64_t fit = static_cast<int64_t>(budget / sizeof(double2) / kb) - 32;
    if (need <= fit) {
        p.steps = static_cast<int>(need);
    } else {  // long buffers: 16 384-sample chunks, their sums combined afterwards
        p.steps = static_cast<int>(std::min<int64_t>(512, fit));
        p.cpb = (need + p.steps - 1) / p.steps;
        const int rc = ensure(ctx, ctx->post[6], static_cast<size_t>(nbuf) * p.cpb * (2 * N + 1) * sizeof(double));
        if (rc) return rc;
        p.part = static_cast<double*>(ctx->post[6].ptr);
    }
    int rc;
    switch (kb) {
        case 8: rc = launch_direct_t<8>(ctx, p, st); break;
        case 10: rc = launch_direct_t<10>(ctx, p, st); break;
        case 12: rc = launch_direct_t<12>(ctx, p, st); break;
        default: rc = launch_direct_t<16>(ctx, p, st); break;
    }
    if (rc || p.cpb == 1) return rc;
    const int64_t n = nbuf * (N + 1);
    return launch_kernel(ctx, dfk::direct_combine_kernel, static_cast<unsigned>((n + 127) / 128), 128, 0, st, p);
}

int launch_demod(dfk_ctx* ctx, const double* x, int64_t nbuf, int64_t bpc, int64_t ld_c, int64_t R, int32_t N, double w0,
                 double* qi, double* dc, cudaStream_t st, bool leave_room = false) {
    if (nbuf == 0) return DFK_OK;
    const dfk::DemodPlan pl = demod_plan(R, w0, N);
    const size_t reserve = leave_room ? seed_fit_reserve(N) : 0;
    const bool fold = pl.folded && (reinterpret_cast<uintptr_t>(x) & 15u) == 0 && (ld_c % 2) == 0;
    if (fold && ld_c == bpc * R) {
        int tiled = try_launch_period(ctx, pl, x, nbuf, N, qi, dc, reserve, st);
        if (tiled == 0) tiled = try_launch_tile(ctx, pl, x, nbuf, R, N, qi, dc, reserve, st);
        if (tiled) return tiled < 0 ? tiled : DFK_OK;
    }
    const bool fold_int = fold && R <= std::numeric_limits<int>::max();
    if (fold_int && pl.P > dfk::kFoldRegisterPeriod && !dev_int("DFK_NO_FOLD_LONG", 0))
        return launch_fold_long<false>(ctx, fold_params(pl, x, nbuf, bpc, ld_c, R, pl.P, N, qi, dc), pl.drift, reserve, st);
    FoldGeometry g;
    if (!(fold_int && pl.P <= dfk::kFoldRegisterPeriod && fold_geometry(ctx, pl, N, reserve, &g)))
        return launch_direct(ctx, x, nbuf, bpc, ld_c, R, N, w0, qi, dc, st);
    dfk::FoldParams p = fold_params(pl, x, nbuf, bpc, ld_c, R, pl.P, N, qi, dc);
    p.pps = g.pps;
    p.nstages = g.nstages;
    const int grid = static_cast<int>(std::min<int64_t>(nbuf, static_cast<int64_t>(ctx->sm_count) * g.ctas_per_sm));
    const int slots = (p.P / 2 + dfk::kFoldConsumers - 1) / dfk::kFoldConsumers;
    auto fold_t = [&](auto kernel) { return launch_kernel(ctx, kernel, grid, dfk::kFoldThreads, g.smem, st, p); };
    if (pl.drift) {
        switch (slots) {
            case 1: return fold_t(dfk::demod_fold_kernel<true, 1>);
            case 2: return fold_t(dfk::demod_fold_kernel<true, 2>);
            case 3: return fold_t(dfk::demod_fold_kernel<true, 3>);
            default: return fold_t(dfk::demod_fold_kernel<true, 4>);
        }
    }
    switch (slots) {
        case 1: return fold_t(dfk::demod_fold_kernel<false, 1>);
        case 2: return fold_t(dfk::demod_fold_kernel<false, 2>);
        case 3: return fold_t(dfk::demod_fold_kernel<false, 3>);
        default: return fold_t(dfk::demod_fold_kernel<false, 4>);
    }
}

// ---- LM -------------------------------------------------------------------------------------------
// Lock-in of a time-major record x[t * C + c]: nbuf_t buffers of R time steps, all C channels; harmonic vectors and
// means of unit u = c * nbuf_t + b.  The interleaved buffer folds like one channel of period P C (column-chunked fold
// kernel in STORE mode: every sample read once), then the per-channel harmonics are taken from the folded arrays.
// Returns DFK_ERR_ARG for geometries that cannot fold (the caller then transposes and takes the channel-major path).
int launch_demod_tm(dfk_ctx* ctx, const double* x, int64_t nbuf_t, int64_t C, int64_t R, int32_t N, double w0, double* qi,
                    double* dc, cudaStream_t st) {
    if (nbuf_t == 0 || C == 0) return DFK_OK;
    const dfk::DemodPlan pl = demod_plan(R, w0, N);
    const int64_t Pc = pl.P * C, Rc = R * C;
    if (!pl.folded || (Pc & 1) || Pc > dfk::kMaxFoldPeriod || Rc > std::numeric_limits<int>::max() ||
        (reinterpret_cast<uintptr_t>(x) & 15u) != 0)
        return fail(DFK_ERR_ARG, "time-major record does not fold (period %lld x %lld channels)", (long long)pl.P, (long long)C);
    const size_t fold_doubles = static_cast<size_t>(nbuf_t) * static_cast<size_t>(Pc);
    int rc = ensure(ctx, ctx->post[6], fold_doubles * sizeof(double) * (pl.drift ? 2 : 1));
    if (!rc) rc = ensure(ctx, ctx->post[7], sizeof(double) * dfk::kMaxHarmonics);
    if (rc) return rc;
    double* fs = static_cast<double*>(ctx->post[6].ptr);
    double* ft = pl.drift ? fs + fold_doubles : fs;
    double* delta_dev = static_cast<double*>(ctx->post[7].ptr);
    DFK_CUDA(cudaMemcpyAsync(delta_dev, pl.delta, sizeof(double) * dfk::kMaxHarmonics, cudaMemcpyHostToDevice, st));
    rc = launch_fold_long<true>(ctx, fold_params(pl, x, nbuf_t, nbuf_t, 0, Rc, Pc, N, fs, ft), pl.drift, 0, st);
    if (rc) return rc;
    const unsigned pgrid = static_cast<unsigned>((nbuf_t * C + 127) / 128);
    return launch_kernel(ctx, pl.drift ? dfk::project_interleaved_kernel<true> : dfk::project_interleaved_kernel<false>, pgrid,
                         128, 0, st, fs, ft, nbuf_t, static_cast<int>(C), static_cast<int>(pl.P), static_cast<int>(R), N,
                         pl.kmul, delta_dev, qi, dc);
}

int pick_lanes(const dfk_ctx* ctx, int64_t nfit, int N, int requested) {
    if (requested == 1 || requested == 2 || requested == 4 || requested == 8 || requested == 16 || requested == 32)
        return requested;
    // enough groups to give every SM ~1024 resident threads; never more lanes than harmonics can use
    const int64_t threads_wanted = static_cast<int64_t>(ctx->sm_count) * 1024;
    int g = 32;
    while (g > 1 && nfit * g > threads_wanted) g >>= 1;
    while (g > 1 && g > N) g >>= 1;
    if (g < 1) g = 1;
    return g;
}

template <int G, int MINB, int TPB>
int launch_first_b(dfk_ctx* ctx, const double* qi, int64_t nfit, dfk::FitMap map, int N, const dfk::GuessSrc& gs, const double* dc,
                   const dfk::LmOpts& o, double* rows, int* list, int* count, dfk::LmCounts* counters, cudaStream_t st,
                   int* flags) {
    const size_t smem = static_cast<size_t>(N + 2) * TPB * sizeof(double);
    // keep the SM's L1/shared split at "all shared": a block of this kernel may share an SM with a demod CTA that
    // needs > 200 kB, and an SM only changes its carve-out when it is idle
    // (only the one-warp-block variant, which is the one that overlaps a demod launch: the bulk variant wants its L1)
    if (TPB == 32)
        DFK_CUDA(cudaFuncSetAttribute(dfk::lm_first_kernel<G, MINB, TPB>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                      cudaSharedmemCarveoutMaxShared));
    const int64_t fits_per_block = TPB / G;
    const int64_t blocks = (nfit + fits_per_block - 1) / fits_per_block;
    const int grid = static_cast<int>(std::min<int64_t>(blocks, static_cast<int64_t>(ctx->sm_count) * 16));
    return launch_kernel(ctx, dfk::lm_first_kernel<G, MINB, TPB>, grid, TPB, smem, st, qi, nfit, map, N, gs, dc, o, rows, list,
                         count, counters, flags);
}

// The per-lane state machine: its one build, four 128-thread blocks per SM
int launch_flat(dfk_ctx* ctx, const double* qi, int64_t nfit, dfk::FitMap map, int N, const dfk::GuessSrc& gs, const double* dc,
                const dfk::LmOpts& o, double* rows, int* list, int* count, dfk::LmCounts* counters, cudaStream_t st) {
    const size_t smem = static_cast<size_t>(N + 2 + dfk::kNeDoubles) * dfk::kLmThreads * sizeof(double);
    const int64_t blocks = (nfit + dfk::kLmThreads - 1) / dfk::kLmThreads;
    const int grid = static_cast<int>(std::min<int64_t>(blocks, static_cast<int64_t>(ctx->sm_count) * 4));
    return launch_kernel(ctx, dfk::lm_flat_kernel<4>, grid, dfk::kLmThreads, smem, st, qi, nfit, map, N, gs, dc, o, rows, list,
                         count, counters);
}

template <int G>
int launch_first(dfk_ctx* ctx, const double* qi, int64_t nfit, dfk::FitMap map, int N, const dfk::GuessSrc& gs, const double* dc,
                 const dfk::LmOpts& o, double* rows, int* list, int* count, dfk::LmCounts* counters, cudaStream_t st,
                 int* flags) {
    // 128 registers give 4 resident blocks per SM; the 96-register build (5 per SM, a few spills) is ~10 % slower
    // per fit but wins when it saves a whole wave of a small batch (cfg 2: 1407 blocks = 3 waves of 592 or 2 of 740)
    const int64_t blocks = (nfit + (dfk::kLmThreads / G) - 1) / (dfk::kLmThreads / G);
    const int64_t w4 = (blocks + 4 * ctx->sm_count - 1) / (4 * ctx->sm_count);
    const int64_t w5 = (blocks + 5 * ctx->sm_count - 1) / (5 * ctx->sm_count);
    const int minb = dev_int("DFK_LM_MINB", (w5 < w4 && w5 <= 3) ? 5 : 4);
    switch (minb) {
        case 5: return launch_first_b<G, 5, dfk::kLmThreads>(ctx, qi, nfit, map, N, gs, dc, o, rows, list, count, counters, st, flags);
        default: return launch_first_b<G, 4, dfk::kLmThreads>(ctx, qi, nfit, map, N, gs, dc, o, rows, list, count, counters, st, flags);
    }
}

int ensure_counters(dfk_ctx* ctx) {
    if (ctx->counters.ptr) return DFK_OK;
    const int rc = ensure(ctx, ctx->counters, sizeof(dfk::LmCounts));
    if (rc) return rc;
    DFK_CUDA(cudaMemsetAsync(ctx->counters.ptr, 0, sizeof(dfk::LmCounts), ctx->stream()));
    return DFK_OK;
}

// first descent for every fit + retry stage for those that stayed above the threshold.
// max_unit: largest unit index + 1 the launch can touch (sizes the retry list).
// cold: the guesses are not expected to be near the solutions, so the fits of a warp will need very different
// numbers of steps -- measured, the per-lane state machine (lm_flat_kernel) is 1.56x faster than the lock-step
// kernel on 4e6 cold N = 15 fits, but 0.84x on warm ones, hence the switch.  (DFK_LM_FLAT = 0 puts cold fits on the
// lock-step kernel, for tests.)
int launch_lm(dfk_ctx* ctx, const double* qi, int64_t nfit, dfk::FitMap map, int N, const dfk::GuessSrc& gs,
              const double* dc, const dfk_lm_opts* opts, double* rows, cudaStream_t st, bool cold = false,
              const dfk::ChainPlan* chain = nullptr) {
    if (nfit == 0) return DFK_OK;
    const int64_t max_unit = (nfit - 1) * map.step + map.offset + 1;
    if (max_unit > std::numeric_limits<int>::max()) return fail(DFK_ERR_ARG, "more than 2^31-1 fit units in one call");
    const dfk::LmOpts o = to_opts(opts);
    int rc = ensure_counters(ctx);
    if (rc) return rc;
    rc = ensure(ctx, ctx->retry, (static_cast<size_t>(nfit) + 4) * sizeof(int));
    if (rc) return rc;
    int* count = static_cast<int*>(ctx->retry.ptr);
    int* list = count + 4;
    int* flags = nullptr;
    if (chain) {  // the chain schedule marks parked units in place of the retry list (units the launch skips stay 0)
        flags = list;
        DFK_CUDA(cudaMemsetAsync(flags, 0, static_cast<size_t>(nfit) * sizeof(int), st));
    }
    auto* counters = static_cast<dfk::LmCounts*>(ctx->counters.ptr);
    DFK_CUDA(cudaMemsetAsync(count, 0, sizeof(int), st));
    const int requested = opts ? opts->lanes_per_fit : 0;
    const int G = pick_lanes(ctx, nfit, N, requested);
    if (requested == 0 && nfit <= 2 * static_cast<int64_t>(ctx->sm_count)) {
        // a handful of fits: one warp per fit in one-warp blocks, spread over all SMs
        rc = launch_first_b<32, 4, 32>(ctx, qi, nfit, map, N, gs, dc, o, rows, list, count, counters, st, flags);
    } else if (G == 1 && !chain && cold && dev_int("DFK_LM_FLAT", 1) != 0) {
        rc = launch_flat(ctx, qi, nfit, map, N, gs, dc, o, rows, list, count, counters, st);
    } else
    switch (G) {
        case 1: rc = launch_first<1>(ctx, qi, nfit, map, N, gs, dc, o, rows, list, count, counters, st, flags); break;
        case 2: rc = launch_first<2>(ctx, qi, nfit, map, N, gs, dc, o, rows, list, count, counters, st, flags); break;
        case 4: rc = launch_first<4>(ctx, qi, nfit, map, N, gs, dc, o, rows, list, count, counters, st, flags); break;
        case 8: rc = launch_first<8>(ctx, qi, nfit, map, N, gs, dc, o, rows, list, count, counters, st, flags); break;
        case 16: rc = launch_first<16>(ctx, qi, nfit, map, N, gs, dc, o, rows, list, count, counters, st, flags); break;
        default: rc = launch_first<32>(ctx, qi, nfit, map, N, gs, dc, o, rows, list, count, counters, st, flags); break;
    }
    if (rc) return rc;
    const size_t smem = static_cast<size_t>(N + 2) * dfk::kLmThreads * sizeof(double);
    const int64_t warps = dfk::kLmThreads / 32;
    if (chain) {
        if (map.step != 1 || map.offset != 0 || map.row_mul != 1) return fail(DFK_ERR_ARG, "chain schedule needs contiguous units");
        DFK_CUDA(cudaFuncSetAttribute(dfk::lm_chain_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                      cudaSharedmemCarveoutMaxShared));
        const int64_t spans = (nfit + 31) / 32;  // a warp scans 32 units at a time
        const int grid = static_cast<int>(std::min<int64_t>((spans + warps - 1) / warps, static_cast<int64_t>(ctx->sm_count) * 8));
        return launch_kernel(ctx, dfk::lm_chain_kernel, grid, dfk::kLmThreads, smem, st, qi, nfit, N, o, *chain, rows, flags,
                             counters);
    }
    DFK_CUDA(cudaFuncSetAttribute(dfk::lm_retry_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                  cudaSharedmemCarveoutMaxShared));
    const int grid = static_cast<int>(std::min<int64_t>((nfit + warps - 1) / warps, static_cast<int64_t>(ctx->sm_count) * 8));
    rc = launch_kernel(ctx, dfk::lm_retry_kernel, grid, dfk::kLmThreads, smem, st, qi, N, o, map.row_mul, rows, list, count,
                       counters);
    if (rc || nfit < dfk::kFlatRetryMin) return rc;
    // enough fits that many may be parked: the thread-per-fit retry kernel stands by
    const size_t fsmem = static_cast<size_t>(N + 2 + dfk::kNeDoubles) * dfk::kLmThreads * sizeof(double);
    const int fgrid = static_cast<int>(std::min<int64_t>((nfit + dfk::kLmThreads - 1) / dfk::kLmThreads,
                                                         static_cast<int64_t>(ctx->sm_count) * 3));
    return launch_kernel(ctx, dfk::lm_retry_flat_kernel, fgrid, dfk::kLmThreads, fsmem, st, qi, N, o, map.row_mul, rows, list,
                         count, counters);
}

// Covariance rows (dfk::fit_covariance) of nfit final result rows on their harmonic vectors: a thread per fit.
int launch_cov(dfk_ctx* ctx, const double* qi, int64_t nfit, int N, const double* rows, double* cov, cudaStream_t st) {
    if (nfit == 0) return DFK_OK;
    const size_t smem = static_cast<size_t>(N + 2) * dfk::kLmThreads * sizeof(double);
    const int grid = static_cast<int>(std::min<int64_t>((nfit + dfk::kLmThreads - 1) / dfk::kLmThreads,
                                                        static_cast<int64_t>(ctx->sm_count) * 8));
    return launch_kernel(ctx, dfk::lm_cov_kernel, grid, dfk::kLmThreads, smem, st, qi, static_cast<long long>(nfit), N, rows,
                         cov);
}

int check_nls_args(int64_t nbuf, int64_t R, int32_t N, double w0) {
    if (nbuf < 0 || R <= 0) return fail(DFK_ERR_ARG, "bad geometry: nbuf=%lld R=%lld", (long long)nbuf, (long long)R);
    if (N < 1 || N > DFK_MAX_HARMONICS) return fail(DFK_ERR_ARG, "harmonic count %d outside 1..%d", N, DFK_MAX_HARMONICS);
    if (!(w0 > 0.0) || !std::isfinite(w0)) return fail(DFK_ERR_ARG, "w0 must be positive and finite");
    return DFK_OK;
}

dfk::GuessSrc guess_value(const double v[4]) {
    dfk::GuessSrc g;
    g.ptr = nullptr;
    g.stride = 0;
    g.div = 1;
    g.skip_first = 0;
    for (int i = 0; i < 4; ++i) g.val[i] = v[i];
    return g;
}

dfk::GuessSrc guess_rows(const double* ptr, int64_t stride, int64_t div, bool skip_first) {
    dfk::GuessSrc g;
    g.ptr = ptr;
    g.stride = stride;
    g.div = div < 1 ? 1 : div;
    g.skip_first = skip_first ? 1 : 0;
    for (int i = 0; i < 4; ++i) g.val[i] = 0.0;
    return g;
}

// How the warm starts of a record are scheduled (fitters.py:370-428).
struct Schedule {
    int64_t chunks = -1;         // 0: every buffer an independent start from init (workers.py:167-173);
                                 // k >= 1: buffer 0 cold, the rest in k chained chunks (k = 1: the sequential chain);
                                 // -1: every buffer its own chunk (the pool schedule at n_cores >= nbuf - 1)
    int64_t b0 = 0;              // buffers of the record that earlier calls have done (host slabs)
    int64_t record_buffers = 0;  // buffers of the whole record (0: the launch is the record)
    bool external_seed = false;  // init is the result of a buffer 0 that lives elsewhere (another GPU's slab)
};

dfk::ChainPlan chain_plan(const Schedule& sc, int64_t bpc) {
    dfk::ChainPlan c;
    c.bpc = bpc;
    c.b0 = sc.b0;
    c.first = sc.external_seed ? 0 : 1;
    const int64_t M = std::max<int64_t>((sc.record_buffers ? sc.record_buffers : bpc) - c.first, 0);
    const int64_t k = std::max<int64_t>(1, std::min<int64_t>(sc.chunks, std::max<int64_t>(M, 1)));
    c.q = M / k;
    c.r = M % k;
    return c;
}

// demod + fits of C device-resident channel records of bpc buffers each (records ld_c samples apart).
//   init_dev == nullptr: every cold start uses init[4]; else channel c starts from init_dev[c * init_stride ..+3].
//   seed_row (single-channel continuation slabs only): the row that already holds buffer 0's result.
//   cov (may be NULL): receives the covariance row of every buffer, from the whole record's harmonic vectors.
int nls_on_device(dfk_ctx* ctx, const double* x, int64_t C, int64_t bpc, int64_t ld_c, int64_t R, int32_t N, double w0,
                  const double init[4], const double* init_dev, int64_t init_stride, const Schedule& sc,
                  const double* seed_row, const dfk_lm_opts* opts, double* rows, double* cov, cudaStream_t st,
                  bool time_major = false) {
    const int64_t nbuf = C * bpc;
    if (nbuf == 0) return DFK_OK;
    int rc = ensure(ctx, ctx->qi, static_cast<size_t>(nbuf) * 2 * N * sizeof(double));
    if (rc) return rc;
    rc = ensure(ctx, ctx->dc, static_cast<size_t>(nbuf) * sizeof(double));
    if (rc) return rc;
    rc = ensure(ctx, ctx->retry, (static_cast<size_t>(nbuf) + 4) * sizeof(int));
    if (rc) return rc;
    rc = ensure_counters(ctx);
    if (rc) return rc;
    double* qi = static_cast<double*>(ctx->qi.ptr);
    double* dc = static_cast<double*>(ctx->dc.ptr);
    const bool seeded = sc.chunks != 0 && !sc.external_seed;
    const dfk::GuessSrc cold = init_dev ? guess_rows(init_dev, init_stride, bpc, false) : guess_value(init);
    const dfk::ChainPlan plan = chain_plan(sc, bpc);
    const dfk::ChainPlan* chain = sc.chunks >= 1 ? &plan : nullptr;
    const bool two_stage = seeded && !seed_row && bpc > 1;
    if (two_stage) {
        // fitters.py:404-405: buffer 0 of every channel is fitted cold before anything else.  Those C fits are a
        // short, latency-bound chain, so they run on a side stream -- their own demodulation of the C first
        // buffers, then the cold fits -- while the main stream demodulates the whole record.
        rc = ensure(ctx, ctx->qi_seed, static_cast<size_t>(C) * 2 * N * sizeof(double));
        if (rc) return rc;
        rc = ensure(ctx, ctx->dc_seed, static_cast<size_t>(C) * sizeof(double));
        if (rc) return rc;
        double* qs = static_cast<double*>(ctx->qi_seed.ptr);
        double* ds = static_cast<double*>(ctx->dc_seed.ptr);
        cudaStream_t aux = ctx->aux_stream;
        // The seed demodulation (C buffers: microseconds) goes first on the MAIN stream: it is itself a persistent
        // shared-memory-filling launch, and queued beside the record's demodulation it would wait for that one to end
        // whenever the GPU is already busy at enqueue time (back-to-back calls: measured +1.2 ms on the cfg-3 wave).
        // Only the cold fits -- one-warp blocks that fit beside a demodulation CTA -- run on the side stream.
        rc = time_major ? launch_demod_tm(ctx, x, 1, C, R, N, w0, qs, ds, st) : launch_demod(ctx, x, C, 1, ld_c, R, N, w0, qs, ds, st);
        if (rc) return rc;
        DFK_CUDA(cudaEventRecord(ctx->fork, st));
        DFK_CUDA(cudaStreamWaitEvent(aux, ctx->fork, 0));
        {
            ProfScope ps(ctx, 2, aux);
            const dfk::GuessSrc cold_c = init_dev ? guess_rows(init_dev, init_stride, 1, false) : guess_value(init);
            rc = launch_lm(ctx, qs, C, {1, 0, bpc}, N, cold_c, ds, opts, rows, aux);
            if (rc) return rc;
        }
        DFK_CUDA(cudaEventRecord(ctx->join, aux));
    }
    {
        ProfScope ps(ctx, 0, st);
        rc = time_major ? launch_demod_tm(ctx, x, bpc, C, R, N, w0, qi, dc, st)
                        : launch_demod(ctx, x, nbuf, bpc, ld_c, R, N, w0, qi, dc, st, two_stage);
    }
    if (rc) return rc;
    if (two_stage) DFK_CUDA(cudaStreamWaitEvent(st, ctx->join, 0));  // before the LM timing scope opens
    ProfScope ps(ctx, 1, st);
    auto fit = [&]() {
        if (sc.external_seed)  // a slab of a record whose buffer 0 lives elsewhere: init is that buffer's result
            return launch_lm(ctx, qi, nbuf, {1, 0, 1}, N, cold, dc, opts, rows, st, false, chain);
        if (!seeded || (bpc == 1 && !seed_row)) return launch_lm(ctx, qi, nbuf, {1, 0, 1}, N, cold, dc, opts, rows, st, true);
        if (seed_row)  // continuation slab of a single record: chunk seeds come from the stored row of buffer 0
            return launch_lm(ctx, qi, nbuf, {1, 0, 1}, N, guess_rows(seed_row, 0, nbuf, false), dc, opts, rows, st, false,
                             chain);
        // fitters.py:407-417: every chunk starts from its channel's buffer-0 result
        return launch_lm(ctx, qi, nbuf, {1, 0, 1}, N, guess_rows(rows, bpc * DFK_ROW_STRIDE, bpc, true), dc, opts, rows, st,
                         false, chain);
    };
    rc = fit();
    // after the last LM launch, so it sees the final rows; buffer 0 of a two-stage record was fitted on qi_seed, but its
    // covariance, like every other buffer's, comes from the whole record's harmonic vectors
    if (rc || !cov) return rc;
    return launch_cov(ctx, qi, nbuf, N, rows, cov, st);
}

Schedule schedule_of(int32_t seeded) {
    Schedule sc;
    sc.chunks = seeded;
    return sc;
}

// Channels per one-warp block of the EKF kernels: the fewest that still leave every warp a scheduler (sub-partition)
// of its own; the development setting DFK_EKF_CPW forces a power of two <= 32.
int ekf_channels_per_warp(const dfk_ctx* ctx, int64_t C) {
    const int64_t schedulers = static_cast<int64_t>(ctx->sm_count) * 4;
    int cpw = 1;
    while (cpw < 32 && (C + cpw - 1) / cpw > schedulers) cpw <<= 1;
    const int forced = dev_int("DFK_EKF_CPW", 0);
    if (forced == 1 || forced == 2 || forced == 4 || forced == 8 || forced == 16 || forced == 32) cpw = forced;
    return cpw;
}

// Per-channel mean and variance of a device record (either layout); see dfk_ekf_kernels.cuh.
int launch_channel_stats(dfk_ctx* ctx, const double* z, int64_t T, int64_t C, int64_t ld_t, int64_t ld_c, double* stats,
                         double* acc, cudaStream_t st) {
    if (ld_c == 1 && C > 1) {  // time-major: coalesced rows, time split over warps and blocks
        const int64_t groups = (C + 31) / 32;
        int nsplit = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>(64, (4ll * ctx->sm_count) / groups)));
        nsplit = static_cast<int>(std::min<int64_t>(nsplit, std::max<int64_t>(1, T / 256)));
        int rc = ensure(ctx, ctx->stats_part, static_cast<size_t>(2) * nsplit * C * sizeof(double));
        if (rc) return rc;
        double* sums = static_cast<double*>(ctx->stats_part.ptr);
        double* sq = sums + static_cast<size_t>(nsplit) * C;
        const dim3 grid(static_cast<unsigned>(groups), static_cast<unsigned>(nsplit));
        rc = launch_kernel(ctx, dfk::stats_tm_kernel, grid, dfk::kStatsThreads, 0, st, z, T, C, ld_t, 0, nullptr, 0, sums);
        if (!rc) rc = launch_kernel(ctx, dfk::stats_tm_kernel, grid, dfk::kStatsThreads, 0, st, z, T, C, ld_t, 1, sums, nsplit, sq);
        if (rc) return rc;
        return launch_kernel(ctx, dfk::stats_tm_finish_kernel, static_cast<int>((C + 127) / 128), 128, 0, st, sums, sq, nsplit,
                             T, C, stats, acc);
    }
    const int sgrid = static_cast<int>(std::min<int64_t>(C, static_cast<int64_t>(ctx->sm_count) * 8));
    return launch_kernel(ctx, dfk::channel_stats_kernel, sgrid, dfk::kStatsThreads, 0, st, z, T, C, ld_t, ld_c, stats, acc);
}

}  // namespace

// ==================================================================================================
extern "C" {

int dfk_abi_version(void) { return DFK_ABI_VERSION; }

const char* dfk_last_error(void) { return g_err; }

int dfk_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

void dfk_default_lm_opts(dfk_lm_opts* o) {
    if (!o) return;
    o->max_lma_steps = 100;
    o->lanes_per_fit = 0;
    o->conv_improve = 1e-9;
    o->conv_param = 1e-9;
    o->fitok_threshold = 1e-3;
    o->m_grid_min = 5.0;
    o->m_grid_max = 30.0;
    o->m_grid_step = 0.5;
    o->bessel_amp_threshold = 0.05;
    o->sincos_amp_threshold = 0.1;
}

void dfk_default_ekf_opts(dfk_ekf_opts* o) {
    if (!o) return;
    const double init[4] = {1.6, 6.0, 0.0, 0.0};
    const double q[5] = {1e-8, 1e-8, 1e-6, 1e-6, 1e-8};
    for (int i = 0; i < 4; ++i) o->init[i] = init[i];
    for (int i = 0; i < 5; ++i) {
        o->p0_diag[i] = 1.0;
        o->q_diag[i] = q[i];
    }
    o->r_val = std::numeric_limits<double>::quiet_NaN();
    o->init_dc = std::numeric_limits<double>::quiet_NaN();
}

int dfk_create(int device, dfk_ctx** out) {
    if (!out) return fail(DFK_ERR_ARG, "null output pointer");
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
        cudaGetLastError();
        return fail(DFK_ERR_CUDA, "no CUDA device available (this library has no CPU path)");
    }
    if (device < 0 || device >= n) return fail(DFK_ERR_ARG, "device %d out of range (0..%d)", device, n - 1);
    cudaDeviceProp prop;
    DFK_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return fail(DFK_ERR_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major,
                    prop.minor);
    dfk_ctx* ctx = new (std::nothrow) dfk_ctx();
    if (!ctx) return fail(DFK_ERR_NOMEM, "out of host memory");
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    ctx->max_smem_optin = static_cast<int>(prop.sharedMemPerBlockOptin);
    ctx->smem_per_sm = static_cast<int>(prop.sharedMemPerMultiprocessor);
    Guard g(ctx);
    if (!g.ok) {
        delete ctx;
        return fail(DFK_ERR_CUDA, "cudaSetDevice(%d) failed", device);
    }
    cudaError_t e = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) {
        // the side stream carries the short cold-seed chain that must start beside a persistent demodulation launch
        // queued at the same moment: highest priority, so that its few one-warp blocks are placed first
        int lo = 0, hi = 0;
        e = cudaDeviceGetStreamPriorityRange(&lo, &hi);
        if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&ctx->aux_stream, cudaStreamNonBlocking, hi);
    }
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->fork, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->join, cudaEventDisableTiming);
    for (int i = 0; i < 2 && e == cudaSuccess; ++i) {
        e = cudaEventCreateWithFlags(&ctx->copied[i], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->consumed[i], cudaEventDisableTiming);
    }
    if (e != cudaSuccess) {
        dfk_destroy(ctx);
        return fail(DFK_ERR_CUDA, "stream/event creation failed: %s", cudaGetErrorString(e));
    }
    *out = ctx;
    return DFK_OK;
}

int dfk_destroy(dfk_ctx* ctx) {
    if (!ctx) return DFK_OK;
    Guard g(ctx);
    if (ctx->own_stream) cudaStreamSynchronize(ctx->own_stream);
    if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
    if (ctx->aux_stream) cudaStreamSynchronize(ctx->aux_stream);
    DevBuf* bufs[] = {&ctx->qi, &ctx->dc, &ctx->retry, &ctx->counters, &ctx->slab[0], &ctx->slab[1],
                      &ctx->rows, &ctx->stats, &ctx->stats_part, &ctx->misc, &ctx->qi_seed, &ctx->dc_seed, &ctx->cov, &ctx->smooth};
    for (DevBuf* b : bufs)
        if (b->ptr) cudaFree(b->ptr);
    for (DevBuf& b : ctx->post)
        if (b.ptr) cudaFree(b.ptr);
    for (auto& kind : ctx->prof_ev)
        for (auto& pair : kind)
            for (cudaEvent_t ev : pair)
                if (ev) cudaEventDestroy(ev);
    for (int i = 0; i < 2; ++i) {
        if (ctx->copied[i]) cudaEventDestroy(ctx->copied[i]);
        if (ctx->consumed[i]) cudaEventDestroy(ctx->consumed[i]);
    }
    for (int i = 0; i < dfk_ctx::kStagers; ++i) {
        if (ctx->stager[i]) cudaFreeHost(ctx->stager[i]);
        if (ctx->stager_free[i]) cudaEventDestroy(ctx->stager_free[i]);
    }
    if (ctx->fork) cudaEventDestroy(ctx->fork);
    if (ctx->join) cudaEventDestroy(ctx->join);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->aux_stream) cudaStreamDestroy(ctx->aux_stream);
    delete ctx;
    return DFK_OK;
}

int dfk_set_stream(dfk_ctx* ctx, void* cuda_stream) {
    if (!ctx) return fail(DFK_ERR_ARG, "null context");
    ctx->user_stream = static_cast<cudaStream_t>(cuda_stream);
    ctx->use_user = cuda_stream != nullptr;
    return DFK_OK;
}

int dfk_use_legacy_default_stream(dfk_ctx* ctx, int on) {
    if (!ctx) return fail(DFK_ERR_ARG, "null context");
    ctx->user_stream = nullptr;  // the legacy default stream is the null handle
    ctx->use_user = on != 0;
    return DFK_OK;
}

int dfk_synchronize(dfk_ctx* ctx) {
    DFK_ENTER(ctx);
    DFK_CUDA(cudaStreamSynchronize(ctx->stream()));
    return DFK_OK;
}

int dfk_demod(dfk_ctx* ctx, const double* x_dev, int64_t nbuf, int64_t R, int32_t N, double w0, double* qi_dev,
              double* dc_dev) {
    DFK_ENTER(ctx);
    const int rc = check_nls_args(nbuf, R, N, w0);
    if (rc) return rc;
    if (nbuf > 0 && (!x_dev || !qi_dev || !dc_dev)) return fail(DFK_ERR_ARG, "null device pointer");
    return launch_demod(ctx, x_dev, nbuf, nbuf, nbuf * R, R, N, w0, qi_dev, dc_dev, ctx->stream());
}

int dfk_lm_fit(dfk_ctx* ctx, const double* qi_dev, int64_t nbuf, int32_t N, const double* guess_dev,
               int64_t guess_stride, const double* dc_dev, const dfk_lm_opts* opts, double* rows_dev) {
    DFK_ENTER(ctx);
    if (nbuf < 0) return fail(DFK_ERR_ARG, "negative fit count");
    if (N < 1 || N > DFK_MAX_HARMONICS) return fail(DFK_ERR_ARG, "harmonic count %d outside 1..%d", N, DFK_MAX_HARMONICS);
    if (nbuf > 0 && (!qi_dev || !guess_dev || !rows_dev)) return fail(DFK_ERR_ARG, "null device pointer");
    if (guess_stride != 0 && guess_stride < 4) return fail(DFK_ERR_ARG, "guess_stride must be 0 or >= 4");
    const dfk::GuessSrc gs = guess_stride == 0 ? guess_rows(guess_dev, 0, nbuf, false) : guess_rows(guess_dev, guess_stride, 1, false);
    return launch_lm(ctx, qi_dev, nbuf, {1, 0, 1}, N, gs, dc_dev, opts, rows_dev, ctx->stream(), guess_stride != 0);
}

// The record entries below and their _cov variants share one body; cov == NULL launches exactly what the plain
// entry always launched.
static int nls_fit_dev_impl(dfk_ctx* ctx, const double* x_dev, int64_t nbuf, int64_t R, int32_t N, double w0,
                            const double init[4], int32_t seeded, const dfk_lm_opts* opts, double* rows_dev, double* cov_dev) {
    DFK_ENTER(ctx);
    const int rc = check_nls_args(nbuf, R, N, w0);
    if (rc) return rc;
    if (!init) return fail(DFK_ERR_ARG, "null init");
    if (nbuf > 0 && (!x_dev || !rows_dev)) return fail(DFK_ERR_ARG, "null device pointer");
    return nls_on_device(ctx, x_dev, 1, nbuf, nbuf * R, R, N, w0, init, nullptr, 0, schedule_of(seeded), nullptr, opts,
                         rows_dev, cov_dev, ctx->stream());
}

// The _cov entries need somewhere to put the covariance rows.
static int check_cov(const double* cov, int64_t n) {
    return (n > 0 && !cov) ? fail(DFK_ERR_ARG, "null covariance pointer") : DFK_OK;
}

int dfk_lm_cov(dfk_ctx* ctx, const double* qi_dev, int64_t nbuf, int32_t N, const double* rows_dev, double* cov_dev) {
    DFK_ENTER(ctx);
    if (nbuf < 0) return fail(DFK_ERR_ARG, "negative fit count");
    if (N < 1 || N > DFK_MAX_HARMONICS) return fail(DFK_ERR_ARG, "harmonic count %d outside 1..%d", N, DFK_MAX_HARMONICS);
    if (nbuf > 0 && (!qi_dev || !rows_dev || !cov_dev)) return fail(DFK_ERR_ARG, "null device pointer");
    return launch_cov(ctx, qi_dev, nbuf, N, rows_dev, cov_dev, ctx->stream());
}

int dfk_nls_fit_dev(dfk_ctx* ctx, const double* x_dev, int64_t nbuf, int64_t R, int32_t N, double w0,
                    const double init[4], int32_t seeded, const dfk_lm_opts* opts, double* rows_dev) {
    return nls_fit_dev_impl(ctx, x_dev, nbuf, R, N, w0, init, seeded, opts, rows_dev, nullptr);
}

int dfk_nls_fit_cov_dev(dfk_ctx* ctx, const double* x_dev, int64_t nbuf, int64_t R, int32_t N, double w0,
                        const double init[4], int32_t seeded, const dfk_lm_opts* opts, double* rows_dev, double* cov_dev) {
    return check_cov(cov_dev, nbuf) ? DFK_ERR_ARG
                                    : nls_fit_dev_impl(ctx, x_dev, nbuf, R, N, w0, init, seeded, opts, rows_dev, cov_dev);
}

int dfk_nls_fit_seeded_dev(dfk_ctx* ctx, const double* x_dev, int64_t nbuf, int64_t R, int32_t N, double w0,
                           const double seed[4], int32_t chunks, const dfk_lm_opts* opts, double* rows_dev) {
    DFK_ENTER(ctx);
    const int rc = check_nls_args(nbuf, R, N, w0);
    if (rc) return rc;
    if (!seed) return fail(DFK_ERR_ARG, "null seed");
    if (chunks == 0) return fail(DFK_ERR_ARG, "a seeded slab has at least one chunk (or DFK_SCHED_EACH)");
    if (nbuf > 0 && (!x_dev || !rows_dev)) return fail(DFK_ERR_ARG, "null device pointer");
    Schedule sc;
    sc.chunks = chunks;
    sc.external_seed = true;
    return nls_on_device(ctx, x_dev, 1, nbuf, nbuf * R, R, N, w0, seed, nullptr, 0, sc, nullptr, opts, rows_dev, nullptr,
                         ctx->stream());
}

static int nls_fit_batch_impl(dfk_ctx* ctx, const double* x_dev, int64_t C, int64_t bufs_per_channel, int64_t ld_c,
                              int64_t R, int32_t N, double w0, const double init[4], const double* init_dev,
                              int64_t init_stride, int32_t seeded, const dfk_lm_opts* opts, double* rows_dev, double* cov_dev) {
    DFK_ENTER(ctx);
    if (C < 0 || bufs_per_channel < 0) return fail(DFK_ERR_ARG, "negative channel or buffer count");
    const int rc = check_nls_args(C * bufs_per_channel, R, N, w0);
    if (rc) return rc;
    if (ld_c < bufs_per_channel * R) return fail(DFK_ERR_ARG, "channel stride shorter than the channel record");
    if (!init && !init_dev) return fail(DFK_ERR_ARG, "no initial guess");
    if (init_dev && init_stride < 4) return fail(DFK_ERR_ARG, "init_stride must be >= 4");
    if (C * bufs_per_channel > 0 && (!x_dev || !rows_dev)) return fail(DFK_ERR_ARG, "null device pointer");
    const double zero[4] = {0, 0, 0, 0};
    return nls_on_device(ctx, x_dev, C, bufs_per_channel, ld_c, R, N, w0, init ? init : zero, init_dev, init_stride,
                         schedule_of(seeded), nullptr, opts, rows_dev, cov_dev, ctx->stream());
}

int dfk_nls_fit_batch_dev(dfk_ctx* ctx, const double* x_dev, int64_t C, int64_t bufs_per_channel, int64_t ld_c,
                          int64_t R, int32_t N, double w0, const double init[4], const double* init_dev,
                          int64_t init_stride, int32_t seeded, const dfk_lm_opts* opts, double* rows_dev) {
    return nls_fit_batch_impl(ctx, x_dev, C, bufs_per_channel, ld_c, R, N, w0, init, init_dev, init_stride, seeded, opts,
                              rows_dev, nullptr);
}

int dfk_nls_fit_batch_cov_dev(dfk_ctx* ctx, const double* x_dev, int64_t C, int64_t bufs_per_channel, int64_t ld_c,
                              int64_t R, int32_t N, double w0, const double init[4], const double* init_dev,
                              int64_t init_stride, int32_t seeded, const dfk_lm_opts* opts, double* rows_dev, double* cov_dev) {
    return check_cov(cov_dev, C * bufs_per_channel) ? DFK_ERR_ARG
                                                    : nls_fit_batch_impl(ctx, x_dev, C, bufs_per_channel, ld_c, R, N, w0, init,
                                                                         init_dev, init_stride, seeded, opts, rows_dev, cov_dev);
}

int dfk_demod_tm_dev(dfk_ctx* ctx, const double* x_dev, int64_t bufs_per_channel, int64_t C, int64_t R, int32_t N, double w0,
                     double* qi_dev, double* dc_dev) {
    DFK_ENTER(ctx);
    if (C < 0 || bufs_per_channel < 0) return fail(DFK_ERR_ARG, "negative channel or buffer count");
    const int rc = check_nls_args(C * bufs_per_channel, R, N, w0);
    if (rc) return rc;
    if (C * bufs_per_channel > 0 && (!x_dev || !qi_dev || !dc_dev)) return fail(DFK_ERR_ARG, "null device pointer");
    ProfScope ps(ctx, 0, ctx->stream());
    return launch_demod_tm(ctx, x_dev, bufs_per_channel, C, R, N, w0, qi_dev, dc_dev, ctx->stream());
}

static int nls_fit_batch_tm_impl(dfk_ctx* ctx, const double* x_dev, int64_t C, int64_t bufs_per_channel, int64_t R,
                                 int32_t N, double w0, const double init[4], const double* init_dev, int64_t init_stride,
                                 int32_t seeded, const dfk_lm_opts* opts, double* rows_dev, double* cov_dev) {
    DFK_ENTER(ctx);
    if (C < 0 || bufs_per_channel < 0) return fail(DFK_ERR_ARG, "negative channel or buffer count");
    const int rc = check_nls_args(C * bufs_per_channel, R, N, w0);
    if (rc) return rc;
    if (!init && !init_dev) return fail(DFK_ERR_ARG, "no initial guess");
    if (init_dev && init_stride < 4) return fail(DFK_ERR_ARG, "init_stride must be >= 4");
    if (C * bufs_per_channel > 0 && (!x_dev || !rows_dev)) return fail(DFK_ERR_ARG, "null device pointer");
    const double zero[4] = {0, 0, 0, 0};
    return nls_on_device(ctx, x_dev, C, bufs_per_channel, 0, R, N, w0, init ? init : zero, init_dev, init_stride,
                         schedule_of(seeded), nullptr, opts, rows_dev, cov_dev, ctx->stream(), true);
}

int dfk_nls_fit_batch_tm_dev(dfk_ctx* ctx, const double* x_dev, int64_t C, int64_t bufs_per_channel, int64_t R, int32_t N,
                             double w0, const double init[4], const double* init_dev, int64_t init_stride, int32_t seeded,
                             const dfk_lm_opts* opts, double* rows_dev) {
    return nls_fit_batch_tm_impl(ctx, x_dev, C, bufs_per_channel, R, N, w0, init, init_dev, init_stride, seeded, opts, rows_dev,
                                 nullptr);
}

int dfk_nls_fit_batch_tm_cov_dev(dfk_ctx* ctx, const double* x_dev, int64_t C, int64_t bufs_per_channel, int64_t R, int32_t N,
                                 double w0, const double init[4], const double* init_dev, int64_t init_stride, int32_t seeded,
                                 const dfk_lm_opts* opts, double* rows_dev, double* cov_dev) {
    return check_cov(cov_dev, C * bufs_per_channel) ? DFK_ERR_ARG
                                                    : nls_fit_batch_tm_impl(ctx, x_dev, C, bufs_per_channel, R, N, w0, init,
                                                                            init_dev, init_stride, seeded, opts, rows_dev, cov_dev);
}


static int nls_host_impl(dfk_ctx* ctx, const double* x_host, int64_t nsamp, int64_t R, int32_t N, double w0,
                         const double init[4], Schedule sc, const dfk_lm_opts* opts, double* rows_host, double* cov_host);

int dfk_nls_fit_host(dfk_ctx* ctx, const double* x_host, int64_t nsamp, int64_t R, int32_t N, double w0,
                     const double init[4], int32_t seeded, const dfk_lm_opts* opts, double* rows_host) {
    return nls_host_impl(ctx, x_host, nsamp, R, N, w0, init, schedule_of(seeded), opts, rows_host, nullptr);
}

int dfk_nls_fit_cov_host(dfk_ctx* ctx, const double* x_host, int64_t nsamp, int64_t R, int32_t N, double w0,
                         const double init[4], int32_t seeded, const dfk_lm_opts* opts, double* rows_host, double* cov_host) {
    return check_cov(cov_host, R > 0 ? nsamp / R : 0)
               ? DFK_ERR_ARG
               : nls_host_impl(ctx, x_host, nsamp, R, N, w0, init, schedule_of(seeded), opts, rows_host, cov_host);
}

int dfk_nls_fit_seeded_host(dfk_ctx* ctx, const double* x_host, int64_t nsamp, int64_t R, int32_t N, double w0,
                            const double seed[4], int32_t chunks, const dfk_lm_opts* opts, double* rows_host) {
    if (chunks == 0) return fail(DFK_ERR_ARG, "a seeded slab has at least one chunk (or DFK_SCHED_EACH)");
    Schedule sc;
    sc.chunks = chunks;
    sc.external_seed = true;
    return nls_host_impl(ctx, x_host, nsamp, R, N, w0, seed, sc, opts, rows_host, nullptr);
}

static int nls_host_impl(dfk_ctx* ctx, const double* x_host, int64_t nsamp, int64_t R, int32_t N, double w0,
                         const double init[4], Schedule sc, const dfk_lm_opts* opts, double* rows_host, double* cov_host) {
    DFK_ENTER(ctx);
    if (nsamp < 0) return fail(DFK_ERR_ARG, "negative sample count");
    const int64_t nbuf = R > 0 ? nsamp / R : 0;
    int rc = check_nls_args(nbuf, R, N, w0);
    if (rc) return rc;
    if (!init) return fail(DFK_ERR_ARG, "null init");
    if (nbuf == 0) return DFK_OK;
    if (!x_host || !rows_host) return fail(DFK_ERR_ARG, "null host pointer");
    // slabs of whole buffers, ~128 MiB each, double buffered: the copy of slab i+1 overlaps the
    // kernels of slab i.  (A record that fits one slab is a single copy.)
    const int64_t slab_target = ctx->host_slab_bytes ? static_cast<int64_t>(ctx->host_slab_bytes) : (128ll << 20);
    const int64_t slab_buffers = std::max<int64_t>(1, std::min<int64_t>(nbuf, slab_target / (R * 8)));
    const size_t slab_bytes = static_cast<size_t>(slab_buffers) * R * 8;
    const int nslab_bufs = nbuf > slab_buffers ? 2 : 1;
    for (int i = 0; i < nslab_bufs; ++i) {
        rc = ensure(ctx, ctx->slab[i], slab_bytes);
        if (rc) return rc;
    }
    rc = ensure(ctx, ctx->rows, static_cast<size_t>(nbuf) * DFK_ROW_STRIDE * sizeof(double));
    if (rc) return rc;
    if (cov_host) {
        rc = ensure(ctx, ctx->cov, static_cast<size_t>(nbuf) * DFK_COV_STRIDE * sizeof(double));
        if (rc) return rc;
    }
    // scratch for one slab, sized up front so that no reallocation happens mid-pipeline
    rc = ensure(ctx, ctx->qi, static_cast<size_t>(slab_buffers) * 2 * N * sizeof(double));
    if (rc) return rc;
    rc = ensure(ctx, ctx->dc, static_cast<size_t>(slab_buffers) * sizeof(double));
    if (rc) return rc;
    rc = ensure(ctx, ctx->retry, (static_cast<size_t>(slab_buffers) + 4) * sizeof(int));
    if (rc) return rc;
    double* rows = static_cast<double*>(ctx->rows.ptr);
    double* cov = cov_host ? static_cast<double*>(ctx->cov.ptr) : nullptr;
    cudaStream_t st = ctx->stream();
    const bool pageable = is_pageable(x_host);
    HostCallGuard quiesce(ctx);
    sc.record_buffers = nbuf;
    const bool seeded = sc.chunks != 0 && !sc.external_seed;
    int64_t done = 0;
    for (int64_t i = 0; done < nbuf; ++i) {
        const int sl = static_cast<int>(i & 1);
        const int64_t nb = std::min(slab_buffers, nbuf - done);
        double* dst = static_cast<double*>(ctx->slab[sl].ptr);
        if (i >= 2) DFK_CUDA(cudaStreamWaitEvent(ctx->copy_stream, ctx->consumed[sl], 0));
        rc = copy_slab_to_device(ctx, dst, x_host + done * R, static_cast<size_t>(nb) * R * 8, pageable);
        if (rc) return rc;
        DFK_CUDA(cudaEventRecord(ctx->copied[sl], ctx->copy_stream));
        DFK_CUDA(cudaStreamWaitEvent(st, ctx->copied[sl], 0));
        sc.b0 = done;
        // the covariance of a slab comes from that slab's harmonic vectors, before the next slab overwrites them
        rc = nls_on_device(ctx, dst, 1, nb, nb * R, R, N, w0, init, nullptr, 0, sc,
                           (seeded && done > 0) ? rows : nullptr, opts, rows + done * DFK_ROW_STRIDE,
                           cov ? cov + done * DFK_COV_STRIDE : nullptr, st);
        if (rc) return rc;
        DFK_CUDA(cudaEventRecord(ctx->consumed[sl], st));
        done += nb;
    }
    DFK_CUDA(cudaMemcpyAsync(rows_host, rows, static_cast<size_t>(nbuf) * DFK_ROW_STRIDE * sizeof(double),
                             cudaMemcpyDeviceToHost, st));
    if (cov)
        DFK_CUDA(cudaMemcpyAsync(cov_host, cov, static_cast<size_t>(nbuf) * DFK_COV_STRIDE * sizeof(double),
                                 cudaMemcpyDeviceToHost, st));
    DFK_CUDA(cudaStreamSynchronize(st));
    quiesce.done();
    return DFK_OK;
}

int dfk_set_host_slab_bytes(dfk_ctx* ctx, int64_t bytes) {
    if (!ctx) return fail(DFK_ERR_ARG, "null context");
    if (bytes < 0) return fail(DFK_ERR_ARG, "negative slab size");
    ctx->host_slab_bytes = static_cast<size_t>(bytes);
    return DFK_OK;
}

int dfk_ekf_dev(dfk_ctx* ctx, const double* z_dev, int64_t T, int64_t C, int64_t ld_t, int64_t ld_c, int64_t R,
                double f_samp, double f_mod, const dfk_ekf_opts* opts, double* rows_dev) {
    return dfk_ekf_stream_dev(ctx, z_dev, T, C, ld_t, ld_c, R, f_samp, f_mod, opts, 0, nullptr, rows_dev);
}

int dfk_ekf_stream_dev(dfk_ctx* ctx, const double* z_dev, int64_t T, int64_t C, int64_t ld_t, int64_t ld_c, int64_t R,
                       double f_samp, double f_mod, const dfk_ekf_opts* opts, int64_t k0, double* state_dev,
                       double* rows_dev) {
    DFK_ENTER(ctx);
    if (k0 < 0 || (R > 0 && k0 % R != 0)) return fail(DFK_ERR_ARG, "k0 must be a non-negative multiple of R");
    if (k0 > 0 && !state_dev) return fail(DFK_ERR_ARG, "a continuation slab needs the carried state");
    if (T < 0 || C < 0 || R <= 0) return fail(DFK_ERR_ARG, "bad geometry: T=%lld C=%lld R=%lld", (long long)T, (long long)C, (long long)R);
    if (!(f_samp > 0.0) || !(f_mod > 0.0)) return fail(DFK_ERR_ARG, "f_samp and f_mod must be positive");
    if (T == 0 || C == 0) return DFK_OK;
    if (!z_dev || !rows_dev) return fail(DFK_ERR_ARG, "null device pointer");
    dfk_ekf_opts d;
    if (!opts) {
        dfk_default_ekf_opts(&d);
        opts = &d;
    }
    int rc = ensure(ctx, ctx->stats, static_cast<size_t>(C) * 2 * sizeof(double));
    if (rc) return rc;
    cudaStream_t st = ctx->stream();
    double* stats = static_cast<double*>(ctx->stats.ptr);
    const bool need_stats = std::isnan(opts->init_dc) || std::isnan(opts->r_val);
    if (k0 == 0 && need_stats && !ctx->stats_ready) {
        // initial dc and default measurement variance come from the first (or only) slab, unless the caller
        // prepared whole-record moments (dfk_ekf_host on a streamed record)
        rc = launch_channel_stats(ctx, z_dev, T, C, ld_t, ld_c, stats, nullptr, st);
        if (rc) return rc;
    }
    dfk::EkfLaunch a;
    a.k0 = k0;
    a.state = state_dev;
    for (int i = 0; i < 4; ++i) a.init[i] = opts->init[i];
    a.init_dc = opts->init_dc;
    for (int i = 0; i < 5; ++i) {
        a.p0[i] = opts->p0_diag[i];
        a.q[i] = opts->q_diag[i];
    }
    a.r_val = opts->r_val;
    a.w_m = 2 * dfk::kPi * f_mod;  // fitters.py:262
    a.f_samp = f_samp;
    const int cpw = ekf_channels_per_warp(ctx, C);
    a.cpw = cpw;
    const int64_t grid = (C + cpw - 1) / cpw;
    if (grid > std::numeric_limits<int>::max()) return fail(DFK_ERR_ARG, "too many channels");
    ProfScope ps(ctx, 3, st);
    return launch_kernel(ctx, dfk::ekf_kernel, static_cast<int>(grid), 32, 0, st, z_dev, T, C, ld_t, ld_c, R, a, stats, rows_dev);
}

int dfk_ekf_smooth_dev(dfk_ctx* ctx, const double* z_dev, int64_t T, int64_t C, int64_t ld_t, int64_t ld_c, int64_t R,
                       double f_samp, double f_mod, const dfk_ekf_opts* opts, int64_t k0, const double* state_dev,
                       int64_t block, double* rows_dev, double* var_dev, double* filt_rows_dev, double* filt_var_dev) {
    DFK_ENTER(ctx);
    if (k0 < 0 || (R > 0 && k0 % R != 0)) return fail(DFK_ERR_ARG, "k0 must be a non-negative multiple of R");
    if (k0 > 0 && !state_dev) return fail(DFK_ERR_ARG, "a window that starts at k0 > 0 needs the carried state");
    if (T < 0 || C < 0 || R <= 0) return fail(DFK_ERR_ARG, "bad geometry: T=%lld C=%lld R=%lld", (long long)T, (long long)C, (long long)R);
    if (!(f_samp > 0.0) || !(f_mod > 0.0)) return fail(DFK_ERR_ARG, "f_samp and f_mod must be positive");
    if (block < 0 || block % dfk::kEkfTile != 0)
        return fail(DFK_ERR_ARG, "block must be 0 (library's choice) or a positive multiple of %d", dfk::kEkfTile);
    if (T / R == 0 || C == 0) return DFK_OK;
    if (!z_dev || !rows_dev) return fail(DFK_ERR_ARG, "null device pointer");
    dfk_ekf_opts d;
    if (!opts) {
        dfk_default_ekf_opts(&d);
        opts = &d;
    }
    const int64_t t_round = (T + dfk::kEkfTile - 1) / dfk::kEkfTile * dfk::kEkfTile;
    const int64_t B = std::min<int64_t>(block ? block : dfk::kSmoothBlockDefault, t_round);
    const int64_t nblk = (T + B - 1) / B;
    // C (nblk + B) 20 doubles; C < 2^31 * 32 and nblk + B <= T + 32, so the product is formed in 128 bits
    const unsigned __int128 want = static_cast<unsigned __int128>(C) * static_cast<unsigned __int128>(nblk + B) *
                                   dfk::kSmoothDoubles * sizeof(double);
    size_t free_b = 0, total_b = 0;
    DFK_CUDA(cudaMemGetInfo(&free_b, &total_b));
    if (want > static_cast<unsigned __int128>(free_b) + ctx->smooth.bytes)
        return fail(DFK_ERR_NOMEM, "smoother scratch of %.0f bytes (checkpoints every %lld samples and a block store) does "
                    "not fit the device's %zu free bytes", static_cast<double>(want), (long long)B, free_b + ctx->smooth.bytes);
    int rc = ensure(ctx, ctx->smooth, static_cast<size_t>(want));
    if (rc) return rc;
    rc = ensure(ctx, ctx->stats, static_cast<size_t>(C) * 2 * sizeof(double));
    if (rc) return rc;
    cudaStream_t st = ctx->stream();
    double* stats = static_cast<double*>(ctx->stats.ptr);
    if (!state_dev && (std::isnan(opts->init_dc) || std::isnan(opts->r_val))) {
        rc = launch_channel_stats(ctx, z_dev, T, C, ld_t, ld_c, stats, nullptr, st);
        if (rc) return rc;
    }
    dfk::SmoothLaunch a;
    a.f.k0 = k0;
    a.f.state = const_cast<double*>(state_dev);  // read only: the smoother never writes the carried state
    for (int i = 0; i < 4; ++i) a.f.init[i] = opts->init[i];
    a.f.init_dc = opts->init_dc;
    for (int i = 0; i < 5; ++i) {
        a.f.p0[i] = opts->p0_diag[i];
        a.f.q[i] = opts->q_diag[i];
    }
    a.f.r_val = opts->r_val;
    a.f.w_m = 2 * dfk::kPi * f_mod;
    a.f.f_samp = f_samp;
    const int cpw = ekf_channels_per_warp(ctx, C);
    a.f.cpw = cpw;
    const int64_t grid = (C + cpw - 1) / cpw;
    if (grid > std::numeric_limits<int>::max()) return fail(DFK_ERR_ARG, "too many channels");
    a.B = B;
    a.ckpt = static_cast<double*>(ctx->smooth.ptr);
    a.store = a.ckpt + static_cast<size_t>(C) * nblk * dfk::kSmoothDoubles;
    a.rows = rows_dev;
    a.var = var_dev;
    a.filt_rows = filt_rows_dev;
    a.filt_var = filt_var_dev;
    rc = launch_kernel(ctx, dfk::ekf_smooth_forward_kernel, static_cast<int>(grid), 32, 0, st, z_dev, T, C, ld_t, ld_c, R,
                       a, stats);
    if (rc) return rc;
    return launch_kernel(ctx, dfk::ekf_smooth_backward_kernel, static_cast<int>(grid), 32, 0, st, z_dev, T, C, ld_t, ld_c,
                         R, a, stats);
}

// EKFFitter.fit on host records [C][T].  A record that fits the device goes up whole.  A longer one (cfg 4 is 655 GB)
// is streamed in slabs of whole buffers, twice when the filter needs the whole-record mean / variance first
// (fitters.py:253,256 take them over the full record): pass 1 merges per-slab moments, pass 2 runs the filter
// with its state carried from slab to slab.
int dfk_ekf_host(dfk_ctx* ctx, const double* z_host, int64_t T, int64_t C, int64_t R, double f_samp, double f_mod,
                 const dfk_ekf_opts* opts, double* rows_host) {
    DFK_ENTER(ctx);
    if (T < 0 || C < 0 || R <= 0) return fail(DFK_ERR_ARG, "bad geometry");
    const int64_t nbuf = T / R;
    if (T == 0 || C == 0) return DFK_OK;
    if (!z_host || (nbuf > 0 && !rows_host)) return fail(DFK_ERR_ARG, "null host pointer");
    dfk_ekf_opts d;
    if (!opts) {
        dfk_default_ekf_opts(&d);
        opts = &d;
    }
    size_t free_b = 0, total_b = 0;
    DFK_CUDA(cudaMemGetInfo(&free_b, &total_b));
    const size_t rec_bytes = static_cast<size_t>(T) * C * 8;
    size_t budget = ctx->host_slab_bytes ? 2 * ctx->host_slab_bytes : (free_b + ctx->slab[0].bytes + ctx->slab[1].bytes) / 2;
    cudaStream_t st = ctx->stream();
    int rc = ensure(ctx, ctx->rows, std::max<size_t>(8, static_cast<size_t>(nbuf) * C * DFK_ROW_STRIDE * 8));
    if (rc) return rc;
    double* rows = static_cast<double*>(ctx->rows.ptr);
    const bool pageable = is_pageable(z_host);
    HostCallGuard quiesce(ctx);
    if (rec_bytes <= budget || nbuf <= 1) {
        rc = ensure(ctx, ctx->slab[0], rec_bytes);
        if (rc) return rc;
        rc = copy_slab_to_device(ctx, ctx->slab[0].ptr, z_host, rec_bytes, pageable);
        if (rc) return rc;
        DFK_CUDA(cudaEventRecord(ctx->copied[0], ctx->copy_stream));
        DFK_CUDA(cudaStreamWaitEvent(st, ctx->copied[0], 0));
        rc = dfk_ekf_dev(ctx, static_cast<const double*>(ctx->slab[0].ptr), T, C, 1, T, R, f_samp, f_mod, opts, rows);
        if (rc) return rc;
    } else {
        // slab = bps buffers of every channel, device layout [C][bps * R]; two slabs alternate
        int64_t bps = static_cast<int64_t>(budget / 2 / (static_cast<size_t>(C) * R * 8));
        if (bps < 1) return fail(DFK_ERR_NOMEM, "one buffer of all %lld channels does not fit the device", (long long)C);
        bps = std::min(bps, nbuf);
        const int64_t Ts = bps * R;
        for (int i = 0; i < 2; ++i) {
            rc = ensure(ctx, ctx->slab[i], static_cast<size_t>(C) * Ts * 8);
            if (rc) return rc;
        }
        rc = ensure(ctx, ctx->misc, static_cast<size_t>(C) * (3 + dfk::kEkfStateStride) * 8 + 256);
        if (rc) return rc;
        rc = ensure(ctx, ctx->stats, static_cast<size_t>(C) * 2 * sizeof(double));
        if (rc) return rc;
        double* acc = static_cast<double*>(ctx->misc.ptr);
        double* state = acc + 3 * C;
        double* slab_rows = nullptr;
        rc = ensure(ctx, ctx->qi, static_cast<size_t>(C) * bps * DFK_ROW_STRIDE * 8);  // rows of one slab, [C][bps]
        if (rc) return rc;
        slab_rows = static_cast<double*>(ctx->qi.ptr);
        const bool need_stats = std::isnan(opts->init_dc) || std::isnan(opts->r_val);
        int64_t slab_no = 0;
        for (int pass = need_stats ? 0 : 1; pass < 2; ++pass) {
            if (pass == 0) DFK_CUDA(cudaMemsetAsync(acc, 0, static_cast<size_t>(C) * 3 * 8, st));
            // the tail of the record past the last whole buffer only matters to the moments (pass 0)
            const int64_t t_end = pass == 0 ? T : nbuf * R;
            for (int64_t t0 = 0; t0 < t_end; t0 += Ts, ++slab_no) {
                const int sl = static_cast<int>(slab_no & 1);
                const int64_t tn = std::min(Ts, t_end - t0);
                double* dst = static_cast<double*>(ctx->slab[sl].ptr);
                if (slab_no >= 2) DFK_CUDA(cudaStreamWaitEvent(ctx->copy_stream, ctx->consumed[sl], 0));
                // channel c's piece of the slab is contiguous on the host: one strided copy
                DFK_CUDA(cudaMemcpy2DAsync(dst, static_cast<size_t>(tn) * 8, z_host + t0, static_cast<size_t>(T) * 8,
                                           static_cast<size_t>(tn) * 8, static_cast<size_t>(C), cudaMemcpyHostToDevice,
                                           ctx->copy_stream));
                DFK_CUDA(cudaEventRecord(ctx->copied[sl], ctx->copy_stream));
                DFK_CUDA(cudaStreamWaitEvent(st, ctx->copied[sl], 0));
                if (pass == 0) {
                    rc = launch_channel_stats(ctx, dst, tn, C, 1, tn, nullptr, acc, st);
                    if (rc) return rc;
                } else {
                    const int64_t nb = tn / R;
                    ctx->stats_ready = need_stats;
                    rc = dfk_ekf_stream_dev(ctx, dst, nb * R, C, 1, tn, R, f_samp, f_mod, opts, t0, state, slab_rows);
                    ctx->stats_ready = false;
                    if (rc) return rc;
                    // rows of this slab [C][nb] -> their place in the [C][nbuf] table
                    DFK_CUDA(cudaMemcpy2DAsync(rows + (t0 / R) * DFK_ROW_STRIDE, static_cast<size_t>(nbuf) * DFK_ROW_STRIDE * 8,
                                               slab_rows, static_cast<size_t>(nb) * DFK_ROW_STRIDE * 8,
                                               static_cast<size_t>(nb) * DFK_ROW_STRIDE * 8, static_cast<size_t>(C),
                                               cudaMemcpyDeviceToDevice, st));
                }
                DFK_CUDA(cudaEventRecord(ctx->consumed[sl], st));
            }
            if (pass == 0) {
                rc = launch_kernel(ctx, dfk::stats_finish_kernel, static_cast<int>((C + 127) / 128), 128, 0, st, acc, C,
                                   static_cast<double*>(ctx->stats.ptr));
                if (rc) return rc;
            }
        }
    }
    if (nbuf > 0)
        DFK_CUDA(cudaMemcpyAsync(rows_host, rows, static_cast<size_t>(nbuf) * C * DFK_ROW_STRIDE * 8,
                                 cudaMemcpyDeviceToHost, st));
    DFK_CUDA(cudaStreamSynchronize(st));
    quiesce.done();
    return DFK_OK;
}

int dfk_synth_snr_dev(dfk_ctx* ctx, double* x_dev, int64_t T, int64_t C, double f_samp, double f_mod, double m,
                      double amp, double visibility, double phi0, double dphi, double psi0, double snr_db,
                      uint64_t seed) {
    return dfk_synth_snr_slab_dev(ctx, x_dev, T, C, T, 0, f_samp, f_mod, m, amp, visibility, phi0, dphi, psi0, snr_db,
                                  seed);
}

int dfk_synth_snr_slab_dev(dfk_ctx* ctx, double* x_dev, int64_t T, int64_t C, int64_t ld_c, int64_t t0, double f_samp,
                           double f_mod, double m, double amp, double visibility, double phi0, double dphi,
                           double psi0, double snr_db, uint64_t seed) {
    DFK_ENTER(ctx);
    if (T < 0 || C < 0) return fail(DFK_ERR_ARG, "bad geometry");
    if (t0 < 0) return fail(DFK_ERR_ARG, "t0 must be non-negative");
    if (ld_c < T) return fail(DFK_ERR_ARG, "channel stride shorter than the slab");
    if (!(f_samp > 0.0) || !(f_mod > 0.0)) return fail(DFK_ERR_ARG, "f_samp and f_mod must be positive");
    if (T == 0 || C == 0) return DFK_OK;
    if (!x_dev) return fail(DFK_ERR_ARG, "null device pointer");
    dfk::SynthParams p;
    p.x = x_dev;
    p.T = T;
    p.C = C;
    p.t0 = t0;
    p.ld_c = ld_c;
    const double per = f_samp / f_mod;
    p.P = (per == std::floor(per) && per >= 1.0 && per < 9e15) ? static_cast<long long>(per) : 0;
    p.f_ratio = f_mod / f_samp;
    p.m = m;
    p.amp = amp;
    p.vis = visibility;
    p.phi0 = phi0;
    p.dphi = dphi;
    p.psi0 = psi0;
    p.sigma_scale = std::pow(10.0, -snr_db / 20.0);
    p.seed = seed;
    // one tabulated clean period per block when the period is a whole number of samples and the table pays for
    // itself: all channels share it (dphi == 0), or every channel's slab is several periods long
    const bool shared_tab = dphi == 0.0 || C == 1;
    const int table = (p.P > 0 && p.P <= dfk::kSynthMaxTable && (shared_tab || T >= 8 * p.P)) ? 1 : 0;
    const int64_t nq = ((t0 + T + 3) >> 2) - (t0 >> 2);
    int64_t ch_per_block = 1;
    if (shared_tab || !table) {  // short records: several channels per block so that a block has ~64k samples
        ch_per_block = std::max<int64_t>(1, std::min<int64_t>(C, 65536 / std::max<int64_t>(T, 1)));
    }
    const int64_t gy = (C + ch_per_block - 1) / ch_per_block;
    int64_t gx = std::max<int64_t>(1, std::min<int64_t>((nq + dfk::kSynthThreads - 1) / dfk::kSynthThreads,
                                                       (static_cast<int64_t>(ctx->sm_count) * 16 + gy - 1) / gy));
    if (gy > 65535) {  // grid.y limit: fold the excess into more channels per block
        ch_per_block = (C + 65534) / 65535;
    }
    const dim3 grid(static_cast<unsigned>(gx), static_cast<unsigned>((C + ch_per_block - 1) / ch_per_block));
    const size_t smem = table ? static_cast<size_t>(p.P) * sizeof(double) : 0;
    return launch_kernel(ctx, dfk::synth_snr_kernel, grid, dfk::kSynthThreads, smem, ctx->stream(), p, table, ch_per_block);
}

int dfk_sweep_demod_dev(dfk_ctx* ctx, int64_t nbuf, int64_t c0, int64_t R, int32_t N, double f_samp, double f_mod, double m,
                        double amp, double visibility, double phi0, double psi0, double snr_db, uint64_t seed,
                        double* qi_dev, double* dc_dev) {
    DFK_ENTER(ctx);
    if (nbuf < 0 || c0 < 0 || R <= 0) return fail(DFK_ERR_ARG, "bad geometry: nbuf=%lld R=%lld", (long long)nbuf, (long long)R);
    if (N < 1 || N > DFK_MAX_HARMONICS) return fail(DFK_ERR_ARG, "harmonic count %d outside 1..%d", N, DFK_MAX_HARMONICS);
    if (!(f_samp > 0.0) || !(f_mod > 0.0)) return fail(DFK_ERR_ARG, "f_samp and f_mod must be positive");
    if (nbuf == 0) return DFK_OK;
    if (!qi_dev || !dc_dev) return fail(DFK_ERR_ARG, "null pointer");
    cudaStream_t st = ctx->stream();
    const double per = f_samp / f_mod;
    const bool whole = per == std::floor(per) && per >= 1.0;
    const int64_t P = whole ? static_cast<int64_t>(per) : 0;
    // fused path: one whole period per record, the geometry of the quarter-wave kernel, tables that fit the SM
    if (whole && R == P && P <= dfk::kTileMaxPeriod && (P % 4) == 0 && (reinterpret_cast<uintptr_t>(qi_dev) & 15u) == 0 &&
        !dev_int("DFK_NO_SWEEP_FUSE", 0)) {
        dfk::SweepParams sp = {};
        sp.synth.T = P;
        sp.synth.C = nbuf;
        sp.synth.P = P;
        sp.synth.f_ratio = f_mod / f_samp;
        sp.synth.m = m;
        sp.synth.amp = amp;
        sp.synth.vis = visibility;
        sp.synth.phi0 = phi0;
        sp.synth.psi0 = psi0;
        sp.synth.sigma_scale = std::pow(10.0, -snr_db / 20.0);
        sp.synth.seed = seed;
        sp.phi = phi0;
        sp.qi = qi_dev;
        sp.dc = dc_dev;
        sp.nbuf = nbuf;
        sp.c0 = c0;
        sp.N = N;
        const int64_t ngroups = (nbuf + dfk::kPeriodNbw - 1) / dfk::kPeriodNbw;
        const int grid = static_cast<int>(std::min<int64_t>(ngroups, ctx->sm_count));
        // 6 consumer and 10 generator warps around a ring of 10 stages; many harmonics: 5 and 11 around a ring of 6
        size_t smem = dfk::sweep_smem_layout(static_cast<int>(P), N, 6, 10).total;
        if (smem <= static_cast<size_t>(ctx->max_smem_optin)) {
            ProfScope ps(ctx, 0, st);
            return launch_kernel(ctx, dfk::sweep_period_kernel<6, 10, 10>, grid, (6 + 10) * 32, smem, st, sp);
        }
        smem = dfk::sweep_smem_layout(static_cast<int>(P), N, 5, 6).total;
        if (smem <= static_cast<size_t>(ctx->max_smem_optin)) {
            ProfScope ps(ctx, 0, st);
            return launch_kernel(ctx, dfk::sweep_period_kernel<5, 11, 6>, grid, (5 + 11) * 32, smem, st, sp);
        }
    }
    // any other geometry: records generated into scratch in waves, then the ordinary lock-in
    const double w0 = 2.0 * dfk::kPi * f_mod / f_samp;
    const int64_t per_wave = std::max<int64_t>(1, std::min<int64_t>(nbuf, (static_cast<int64_t>(256) << 20) / (R * 8)));
    int rc = ensure(ctx, ctx->slab[0], static_cast<size_t>(per_wave) * R * 8);
    if (rc) return rc;
    double* x = static_cast<double*>(ctx->slab[0].ptr);
    for (int64_t done = 0; done < nbuf; done += per_wave) {
        const int64_t nw = std::min(per_wave, nbuf - done);
        rc = dfk_synth_snr_slab_dev(ctx, x, R, nw, R, 0, f_samp, f_mod, m, amp, visibility, phi0, 0.0, psi0, snr_db,
                                    seed + static_cast<uint64_t>(c0 + done));
        if (rc) return rc;
        ProfScope ps(ctx, 0, st);
        rc = launch_demod(ctx, x, nw, 1, R, R, N, w0, qi_dev + done * 2 * N, dc_dev + done, st);
        if (rc) return rc;
    }
    return DFK_OK;
}

static int nls_sweep_impl(dfk_ctx* ctx, const double* m_values, int32_t nm, int64_t ntrials, int64_t trial0,
                          int64_t seed_stride, int64_t R, int32_t N, double f_samp, double f_mod, double amp, double visibility,
                          double phi0, double psi0, double snr_db, uint64_t seed, double init_a, double init_m,
                          const dfk_lm_opts* opts, double* rows_dev, double* cov_dev) {
    DFK_ENTER(ctx);
    if (nm < 0 || ntrials < 0 || trial0 < 0) return fail(DFK_ERR_ARG, "bad sweep size");
    if (nm == 0 || ntrials == 0) return DFK_OK;
    if (!m_values || !rows_dev) return fail(DFK_ERR_ARG, "null pointer");
    const int64_t nfit = static_cast<int64_t>(nm) * ntrials;
    int rc = ensure(ctx, ctx->qi, static_cast<size_t>(nfit) * 2 * N * sizeof(double));
    if (!rc) rc = ensure(ctx, ctx->dc, static_cast<size_t>(nfit) * sizeof(double));
    if (!rc) rc = ensure(ctx, ctx->qi_seed, static_cast<size_t>(nm) * 4 * sizeof(double));
    if (rc) return rc;
    double* qi = static_cast<double*>(ctx->qi.ptr);
    double* dc = static_cast<double*>(ctx->dc.ptr);
    cudaStream_t st = ctx->stream();
    std::vector<double> guess(static_cast<size_t>(nm) * 4, 0.0);
    for (int i = 0; i < nm; ++i) {
        guess[4 * i] = init_a;
        guess[4 * i + 1] = std::isnan(init_m) ? m_values[i] : init_m;  // workers.py:167-173: init_m = m_true
        guess[4 * i + 3] = 0.0;
    }
    DFK_CUDA(cudaMemcpyAsync(ctx->qi_seed.ptr, guess.data(), guess.size() * sizeof(double), cudaMemcpyHostToDevice, st));
    DFK_CUDA(cudaStreamSynchronize(st));  // `guess` leaves scope; the copy is 600 bytes
    for (int i = 0; i < nm; ++i) {
        rc = dfk_sweep_demod_dev(ctx, ntrials, trial0, R, N, f_samp, f_mod, m_values[i], amp, visibility, phi0, psi0, snr_db,
                                 seed + static_cast<uint64_t>(i) * static_cast<uint64_t>(seed_stride),
                                 qi + static_cast<int64_t>(i) * ntrials * 2 * N, dc + static_cast<int64_t>(i) * ntrials);
        if (rc) return rc;
    }
    ProfScope ps(ctx, 1, st);
    rc = launch_lm(ctx, qi, nfit, {1, 0, 1}, N, guess_rows(static_cast<const double*>(ctx->qi_seed.ptr), 4, ntrials, false), dc,
                   opts, rows_dev, st, true);
    if (rc || !cov_dev) return rc;
    return launch_cov(ctx, qi, nfit, N, rows_dev, cov_dev, st);
}

int dfk_nls_sweep_dev(dfk_ctx* ctx, const double* m_values, int32_t nm, int64_t ntrials, int64_t trial0, int64_t seed_stride,
                      int64_t R, int32_t N, double f_samp, double f_mod, double amp, double visibility, double phi0,
                      double psi0, double snr_db, uint64_t seed, double init_a, double init_m, const dfk_lm_opts* opts,
                      double* rows_dev) {
    return nls_sweep_impl(ctx, m_values, nm, ntrials, trial0, seed_stride, R, N, f_samp, f_mod, amp, visibility, phi0, psi0,
                          snr_db, seed, init_a, init_m, opts, rows_dev, nullptr);
}

int dfk_nls_sweep_cov_dev(dfk_ctx* ctx, const double* m_values, int32_t nm, int64_t ntrials, int64_t trial0,
                          int64_t seed_stride, int64_t R, int32_t N, double f_samp, double f_mod, double amp, double visibility,
                          double phi0, double psi0, double snr_db, uint64_t seed, double init_a, double init_m,
                          const dfk_lm_opts* opts, double* rows_dev, double* cov_dev) {
    return check_cov(cov_dev, static_cast<int64_t>(nm) * ntrials)
               ? DFK_ERR_ARG
               : nls_sweep_impl(ctx, m_values, nm, ntrials, trial0, seed_stride, R, N, f_samp, f_mod, amp, visibility, phi0,
                                psi0, snr_db, seed, init_a, init_m, opts, rows_dev, cov_dev);
}

int dfk_lm_counters_read(dfk_ctx* ctx, dfk_lm_counters* out, int32_t reset) {
    DFK_ENTER(ctx);
    if (!out) return fail(DFK_ERR_ARG, "null output pointer");
    const int rc = ensure_counters(ctx);
    if (rc) return rc;
    static_assert(sizeof(dfk_lm_counters) == sizeof(dfk::LmCounts), "counter layouts must agree");
    DFK_CUDA(cudaMemcpyAsync(out, ctx->counters.ptr, sizeof(dfk_lm_counters), cudaMemcpyDeviceToHost, ctx->stream()));
    if (reset) DFK_CUDA(cudaMemsetAsync(ctx->counters.ptr, 0, sizeof(dfk::LmCounts), ctx->stream()));
    DFK_CUDA(cudaStreamSynchronize(ctx->stream()));
    return DFK_OK;
}

int dfk_profile_enable(dfk_ctx* ctx, int32_t on) {
    DFK_ENTER(ctx);
    if (!on) {
        const int rc = prof_drain(ctx);
        if (rc) return rc;
    }
    ctx->profiling = on != 0;
    return DFK_OK;
}

int dfk_profile_read(dfk_ctx* ctx, double ms_total[DFK_PROFILE_KINDS], int64_t launches[DFK_PROFILE_KINDS], int32_t reset) {
    DFK_ENTER(ctx);
    if (!ms_total || !launches) return fail(DFK_ERR_ARG, "null output pointer");
    const int rc = prof_drain(ctx);
    if (rc) return rc;
    for (int k = 0; k < DFK_PROFILE_KINDS; ++k) {
        ms_total[k] = ctx->prof_ms[k];
        launches[k] = ctx->prof_n[k];
        if (reset) {
            ctx->prof_ms[k] = 0.0;
            ctx->prof_n[k] = 0;
        }
    }
    return DFK_OK;
}

int dfk_probe_fp64(dfk_ctx* ctx, double* tflops_out) {
    DFK_ENTER(ctx);
    if (!tflops_out) return fail(DFK_ERR_ARG, "null output pointer");
    int rc = ensure(ctx, ctx->misc, 256);
    if (rc) return rc;
    cudaStream_t st = ctx->stream();
    cudaEvent_t e0, e1;
    DFK_CUDA(cudaEventCreate(&e0));
    DFK_CUDA(cudaEventCreate(&e1));
    const int iters = 4096, blocks = ctx->sm_count * 8;
    double best_ms = 1e30;
    for (int rep = 0; rep < 4; ++rep) {  // first repetition warms up
        DFK_CUDA(cudaEventRecord(e0, st));
        dfk::fp64_probe_kernel<<<blocks, 256, 0, st>>>(iters, 0.5, static_cast<double*>(ctx->misc.ptr));
        DFK_CUDA(cudaEventRecord(e1, st));
        DFK_CUDA(cudaEventSynchronize(e1));
        float ms = 0.f;
        DFK_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        if (rep > 0 && ms < best_ms) best_ms = ms;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    DFK_CUDA(cudaGetLastError());
    const double flops = 2.0 * 8.0 * iters * 256.0 * blocks;
    *tflops_out = flops / (best_ms * 1e-3) / 1e12;
    return DFK_OK;
}

int dfk_dev_set(const char* name, int32_t value) {
    if (!name || !*name || std::strlen(name) >= sizeof(g_dev[0].name)) return fail(DFK_ERR_ARG, "bad override name");
    std::lock_guard<std::mutex> lock(g_dev_mutex);
    // geometry of the staged host copies (dfk_host.h), shared by every translation unit
    if (std::strcmp(name, "DFK_STAGE_KB") == 0) {
        if (value < 64 || static_cast<size_t>(value) * 1024 > dfk_ctx::kStageBytes) return fail(DFK_ERR_ARG, "stage size out of range");
        host_copy_tuning().stage_bytes = static_cast<size_t>(value) * 1024;
        return DFK_OK;
    }
    if (std::strcmp(name, "DFK_STAGERS") == 0) {
        if (value < 2 || value > dfk_ctx::kStagers) return fail(DFK_ERR_ARG, "stager count out of range");
        host_copy_tuning().stagers = value;
        return DFK_OK;
    }
    if (std::strcmp(name, "DFK_COPY_NT") == 0) {
        host_copy_tuning().nt = value != 0;
        return DFK_OK;
    }
    if (std::strcmp(name, "DFK_COPY_THREADS") == 0) {
        host_copy_tuning().threads = std::max(1, static_cast<int>(value));
        return DFK_OK;
    }
    const int n = g_dev_count.load(std::memory_order_relaxed);
    for (int i = 0; i < n; ++i)
        if (std::strcmp(g_dev[i].name, name) == 0) {
            g_dev[i].value = value;
            return DFK_OK;
        }
    if (n == static_cast<int>(sizeof(g_dev) / sizeof(g_dev[0]))) return fail(DFK_ERR_ARG, "override table full");
    std::strcpy(g_dev[n].name, name);
    g_dev[n].value = value;
    g_dev_count.store(n + 1, std::memory_order_release);
    return DFK_OK;
}

void dfk_dev_clear(void) {
    std::lock_guard<std::mutex> lock(g_dev_mutex);
    g_dev_count.store(0, std::memory_order_release);
    host_copy_tuning() = HostCopyTuning();
}

int64_t dfk_launch_count(dfk_ctx* ctx) { return ctx ? ctx->launches : 0; }

int dfk_demod_path(int64_t R, double w0) {
    const dfk::DemodPlan pl = dfk::make_demod_plan(R, w0, 1);
    return pl.folded ? 1 : 0;
}

int dfk_bessel_dev(dfk_ctx* ctx, const double* x_dev, int64_t n, int32_t nmax, double* out_dev) {
    DFK_ENTER(ctx);
    if (n < 0 || nmax < 0 || nmax > DFK_MAX_HARMONICS + 1) return fail(DFK_ERR_ARG, "bad arguments");
    if (n == 0) return DFK_OK;
    if (!x_dev || !out_dev) return fail(DFK_ERR_ARG, "null device pointer");
    return launch_kernel(ctx, dfk::bessel_kernel, static_cast<int>((n + 127) / 128), 128, 0, ctx->stream(), x_dev, n, nmax,
                         out_dev);
}

}  // extern "C"
