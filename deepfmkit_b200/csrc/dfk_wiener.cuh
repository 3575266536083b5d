// Time-domain witness subtraction: least-squares multi-input FIR (Wiener) filters and the cleaned target series.
//
// Witnesses x_a (a = 0..Cx-1), targets y_t (t = 0..Cy-1), N samples each, L taps, lead k0 in [0, L-1] (k0 = 0 is
// causal, (L-1)/2 a centred two-sided filter), ridge rho >= 0.
//  1. Means: every series loses its mean over all N samples (x~, y~); the means are fp64 reductions in a fixed order,
//     and the kernels subtract them on load, so the inputs are never rewritten.
//  2. Rows n in [n0, n0 + M), n0 = L-1-k0, M = N-L+1: exactly the rows on which every tap is inside the record.
//  3. Model: yhat_t[n] = sum_a sum_{k<L} h[t,a,k] x~_a[n + k0 - k]; tap k looks offsets[k] = k0 - k samples away.
//  4. Normal equations, n_u = Cx L unknowns per target, one matrix for all targets:
//       G[(a,k),(b,l)] = sum_n x~_a[n+k0-k] x~_b[n+k0-l],   p[(a,k),t] = sum_n x~_a[n+k0-k] y~_t[n],
//       (G + lambda I) h_t = p_t,  lambda = rho trace(G) / n_u  (loading relative to the mean diagonal).
//  5. Residual e_t[i] = y~_t[n0+i] - yhat_t[n0+i] (i < M); var_y = (1/M) sum y~_t^2 and var_res = (1/M) sum e_t^2 over
//     the same rows.
//  6. A Cholesky pivot not above kWienerPivotTol times its loaded diagonal entry (a duplicated or linearly dependent
//     witness with rho = 0) sets a device flag; h, the residual and var_res are then NaN, var_y stays finite.
//  7. 1 <= Cx <= 64, Cy >= 1, Cx + Cy <= 65535, L >= 1, Cx L <= 1024, M >= Cx L.
//
// With q = n + k0 - k every sum runs over q in [L-1-k, N-1-k]:
//       G[(a,k),(b,l)] = sum_q x~_a[q] x~_b[q + k - l],   p[(a,k),t] = sum_q x~_a[q] y~_t[q + k - k0].
// The core q in [L-1, N-L] depends only on (a, b, d = k - l) or (a, t, k - k0): wiener_lag_kernel forms these lag sums
// (the O(N) work); wiener_assemble_kernel adds each entry's own k head and L-1-k tail products (L-1 per entry, so the
// edge work is O(Cx^2 L^3) and independent of N).
//
// Kernels and launches of one call (nb = ceil(n_u / kCholBlock)):
//   wiener_means_kernel      1   a CTA per series: mean over N, and var_y over the M rows for targets
//   wiener_lag_kernel        1   (entry tile, time slice) CTAs; slice partials to scratch, no atomics
//   wiener_assemble_kernel   1   G (lower triangle) and p from the slice partials (fixed order) plus edge terms
//   wiener_load_kernel       1   trace(G), lambda, the loaded diagonal, flag reset
//   chol_panel_kernel        nb  diagonal tile factored in shared memory (every CTA), panel solve below it
//   chol_update_kernel       nb - 1   trailing lower-triangle update, a CTA per 64 x 64 tile
//   wiener_solve_kernel      1   a CTA per target: L z = p, L^T h = z (NaN if flagged)
//   wiener_apply_kernel      1   (time tile, 4 targets) CTAs: residual and per-tile sums of e^2   [res or var_res]
//   wiener_var_kernel        1   var_res from the tile sums in a fixed order                     [var_res]
// so 2 nb + 4 launches, plus 1 with a residual or var_res, plus 1 more with var_res: 2 nb + 6 for everything.
// Every sum has a fixed order (bit-identical results from run to run); products may be contracted (FMA).
#pragma once
#include "dfk_common.cuh"

namespace dfk {

constexpr int kWienerMaxWitnesses = 64;
constexpr int kWienerMaxUnknowns = 1024;
constexpr double kWienerPivotTol = 1e-10;

struct WienerSeries {         // sample q of series u: (u < cx ? x[u ldx + q stride] : y[(u-cx) ldy + q stride]) - mean[u]
    const double* x;
    const double* y;
    long long ldx, ldy, stride;
    long long cx, cy, N;
    const double* mean;       // [cx + cy]

    DFK_D double raw(long long u, long long q) const {
        return u < cx ? x[u * ldx + q * stride] : y[(u - cx) * ldy + q * stride];
    }
    DFK_D double at(long long u, long long q) const { return raw(u, q) - mean[u]; }
};

// ---------------------------------------------------------------------------------------------------------------
// Means (and var_y): a CTA per series, strided partial sums (four independent loads in flight per thread), a fixed
// tree.
// ---------------------------------------------------------------------------------------------------------------
constexpr int kWMeanThreads = 1024;

template <int kThreads>
DFK_D double block_sum_fixed(double v, double* red) {  // red: kThreads doubles; result valid in every thread
    red[threadIdx.x] = v;
    __syncthreads();
#pragma unroll
    for (int w = kThreads / 2; w > 0; w >>= 1) {
        if (threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
        __syncthreads();
    }
    const double s = red[0];
    __syncthreads();
    return s;
}

__global__ void __launch_bounds__(kWMeanThreads) wiener_means_kernel(WienerSeries S, long long n0, long long M,
                                                                     double* __restrict__ mean, double* __restrict__ var_y) {
    __shared__ double red[kWMeanThreads];
    const long long u = blockIdx.x;
    constexpr long long kStep = 4ll * kWMeanThreads;
    double s[4] = {0.0, 0.0, 0.0, 0.0};
    long long q = threadIdx.x;
    for (; q + 3 * kWMeanThreads < S.N; q += kStep)
#pragma unroll
        for (int i = 0; i < 4; ++i) s[i] += S.raw(u, q + i * kWMeanThreads);
    for (; q < S.N; q += kWMeanThreads) s[0] += S.raw(u, q);
    const double m = block_sum_fixed<kWMeanThreads>((s[0] + s[1]) + (s[2] + s[3]), red) / static_cast<double>(S.N);
    if (threadIdx.x == 0) mean[u] = m;
    if (u < S.cx) return;
    double v[4] = {0.0, 0.0, 0.0, 0.0};
    q = n0 + threadIdx.x;
    for (; q + 3 * kWMeanThreads < n0 + M; q += kStep)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const double d = S.raw(u, q + i * kWMeanThreads) - m;
            v[i] = fma(d, d, v[i]);
        }
    for (; q < n0 + M; q += kWMeanThreads) {
        const double d = S.raw(u, q) - m;
        v[0] = fma(d, d, v[0]);
    }
    const double t = block_sum_fixed<kWMeanThreads>((v[0] + v[1]) + (v[2] + v[3]), red);
    if (threadIdx.x == 0) var_y[u - S.cx] = t / static_cast<double>(M);
}

// ---------------------------------------------------------------------------------------------------------------
// Lag sums over the core q in [L-1, N-L].  Columns c enumerate (series, lag): witness b has the 2L-1 lags
// d = -(L-1)..L-1 (columns b (2L-1) + d + L-1), then target t the L lags e = k - k0 (columns Cx (2L-1) + t L + k).
// Row a, column c holds sum_q x~_a[q] s~_c[q + lag_c].  A CTA takes kLagRows witnesses x kLagCols consecutive
// columns and one time slice; it walks the slice in chunks of T samples, staging the witness rows [kLagRows][T] and,
// for every series its columns touch, that series' samples at q + lag over the chunk (T - 1 + its columns in the tile)
// in shared memory.  Warp w sums the samples w, w + 4, ... of each chunk into a register tile of kLagRows x 8 columns
// (lane + 32 i); the four warp partials are combined ((w0 + w1) + (w2 + w3)) into the slice partial
// part[slice][tile][r][col].  Tiles whose series all precede the first witness row are skipped (pairs a <= b only).
// ---------------------------------------------------------------------------------------------------------------
constexpr int kLagThreads = 128;
constexpr int kLagRows = 4;
constexpr int kLagCols = 256;
constexpr int kLagPerThread = kLagCols / 32;
constexpr int kLagTileEntries = kLagRows * kLagCols;

struct LagParams {
    WienerSeries S;
    long long L, k0;
    long long ncols, ncx;      // ncx = cx (2L - 1): the witness columns
    long long col_tiles;       // tiles: (row tile, column tile), row-major
    long long q_begin, q_end;  // core range [L-1, N-L + 1)
    long long slice;           // samples per slice (a multiple of T)
    int T;                     // samples per chunk
    double* part;              // [nslices][tiles][kLagTileEntries]
    long long part_stride;     // tiles * kLagTileEntries
};

DFK_HD long long lag_col_series(long long c, long long cx, long long ncx, long long L) {
    return c < ncx ? c / (2 * L - 1) : cx + (c - ncx) / L;
}
DFK_HD long long lag_col_start(long long s, long long cx, long long ncx, long long L) {
    return s < cx ? s * (2 * L - 1) : ncx + (s - cx) * L;
}
DFK_HD long long lag_col_lag(long long c, long long ncx, long long L, long long k0) {
    return c < ncx ? c % (2 * L - 1) - (L - 1) : (c - ncx) % L - k0;
}

__global__ void __launch_bounds__(kLagThreads) wiener_lag_kernel(const LagParams P) {
    extern __shared__ double sm[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long tile = blockIdx.x;
    const long long a0 = (tile / P.col_tiles) * kLagRows, c0 = (tile % P.col_tiles) * kLagCols;
    const long long cx = P.S.cx, L = P.L;
    const long long c_last = min(c0 + kLagCols, P.ncols) - 1;
    const long long s_first = lag_col_series(c0, cx, P.ncx, L), s_last = lag_col_series(c_last, cx, P.ncx, L);
    if (s_last < a0) return;  // every pair of this tile has b < a
    const int T = P.T;
    double* xs = sm;                   // [kLagRows][T]
    double* ss = sm + kLagRows * T;    // per series of the tile: T - 1 + its columns
    int off[kLagPerThread];
#pragma unroll
    for (int i = 0; i < kLagPerThread; ++i) {
        const long long c = c0 + lane + 32 * i;
        off[i] = c <= c_last ? static_cast<int>((lag_col_series(c, cx, P.ncx, L) - s_first) * (T - 1) + (c - c0)) : 0;
    }
    double acc[kLagRows][kLagPerThread];
#pragma unroll
    for (int r = 0; r < kLagRows; ++r)
#pragma unroll
        for (int i = 0; i < kLagPerThread; ++i) acc[r][i] = 0.0;
    const long long qs = P.q_begin + blockIdx.y * P.slice;
    const long long qe = min(qs + P.slice, P.q_end);
    for (long long q0 = qs; q0 < qe; q0 += T) {
        const int tc = static_cast<int>(min(static_cast<long long>(T), qe - q0));
        __syncthreads();  // the previous chunk's reads are done
        for (int i = tid; i < kLagRows * T; i += kLagThreads) {
            const int r = i / T, q = i % T;
            xs[i] = (a0 + r < cx && q < tc) ? P.S.at(a0 + r, q0 + q) : 0.0;
        }
        for (long long s = s_first; s <= s_last; ++s) {
            const long long cs = max(c0, lag_col_start(s, cx, P.ncx, L));
            const long long ce = min(c_last + 1, lag_col_start(s + 1, cx, P.ncx, L));
            const int n = static_cast<int>(T - 1 + ce - cs);
            double* dst = ss + (s - s_first) * (T - 1) + (cs - c0);
            const long long src0 = q0 + lag_col_lag(cs, P.ncx, L, P.k0);
            for (int u = tid; u < n; u += kLagThreads) {
                const long long q = src0 + u;
                dst[u] = q < P.S.N ? P.S.at(s, q) : 0.0;  // past the chunk's last sample the witness row is 0
            }
        }
        __syncthreads();
#pragma unroll 2
        for (int q = warp; q < tc; q += kLagThreads / 32) {
            double xa[kLagRows];
#pragma unroll
            for (int r = 0; r < kLagRows; ++r) xa[r] = xs[r * T + q];
#pragma unroll
            for (int i = 0; i < kLagPerThread; ++i) {
                const double v = ss[off[i] + q];
#pragma unroll
                for (int r = 0; r < kLagRows; ++r) acc[r][i] = fma(xa[r], v, acc[r][i]);
            }
        }
    }
    __syncthreads();  // staging reads done: the area now holds the warp partials [4][kLagTileEntries]
#pragma unroll
    for (int r = 0; r < kLagRows; ++r)
#pragma unroll
        for (int i = 0; i < kLagPerThread; ++i) sm[warp * kLagTileEntries + r * kLagCols + lane + 32 * i] = acc[r][i];
    __syncthreads();
    double* out = P.part + blockIdx.y * P.part_stride + tile * kLagTileEntries;
    for (int e = tid; e < kLagTileEntries; e += kLagThreads)
        out[e] = (sm[e] + sm[kLagTileEntries + e]) + (sm[2 * kLagTileEntries + e] + sm[3 * kLagTileEntries + e]);
}

// ---------------------------------------------------------------------------------------------------------------
// Assembly: G lower triangle (row-major, ld n_u) and p [cy][n_u].  Entry = core sum (slice partials added in slice
// order) + head products (q = L-1-k .. L-2) + tail products (q = N-L+1 .. N-1-k), in that order.
// ---------------------------------------------------------------------------------------------------------------
constexpr int kAssembleThreads = 256;

struct AssembleParams {
    LagParams P;
    long long nslices, nu;
    double* G;                 // [nu][nu]
    double* rhs;               // [cy][nu]
};

DFK_D double lag_core(const AssembleParams& A, long long a, long long c, long long nslices) {
    const long long tile = (a / kLagRows) * A.P.col_tiles + c / kLagCols;
    const double* p = A.P.part + tile * kLagTileEntries + (a % kLagRows) * kLagCols + c % kLagCols;
    double s = 0.0;
    for (long long i = 0; i < nslices; ++i) s += p[i * A.P.part_stride];
    return s;
}

__global__ void __launch_bounds__(kAssembleThreads) wiener_assemble_kernel(const AssembleParams A) {
    const long long nu = A.nu, L = A.P.L, N = A.P.S.N, width = nu + A.P.S.cy;
    const long long e = static_cast<long long>(blockIdx.x) * kAssembleThreads + threadIdx.x;
    if (e >= nu * width) return;
    const long long i = e / width, j = e % width;
    if (j < nu && j > i) return;
    long long a = i / L, k = i % L, b, shift;  // sum over q of x~_a[q] s~_b[q + shift], q in [L-1-k, N-1-k]
    long long c;
    if (j < nu) {
        b = j / L;
        long long l = j % L;
        if (a > b) {  // use the symmetric entry, whose first witness is the smaller
            const long long t = a; a = b; b = t;
            const long long u = k; k = l; l = u;
        }
        shift = k - l;
        c = lag_col_start(b, A.P.S.cx, A.P.ncx, L) + shift + L - 1;
    } else {
        b = A.P.S.cx + (j - nu);
        shift = k - A.P.k0;
        c = A.P.ncx + (j - nu) * L + k;
    }
    double s = lag_core(A, a, c, A.nslices);
    for (long long q = L - 1 - k; q < L - 1; ++q) s = fma(A.P.S.at(a, q), A.P.S.at(b, q + shift), s);
    for (long long q = N - L + 1; q < N - k; ++q) s = fma(A.P.S.at(a, q), A.P.S.at(b, q + shift), s);
    if (j < nu) A.G[i * nu + j] = s;
    else A.rhs[(j - nu) * nu + i] = s;
}

// trace(G) in a fixed order, lambda = rho trace / n_u, G_ii += lambda, diag0 = loaded diagonal, flag = 0
__global__ void __launch_bounds__(kWMeanThreads) wiener_load_kernel(double* __restrict__ G, long long nu, double rho,
                                                                   double* __restrict__ diag0, int* __restrict__ flag) {
    __shared__ double red[kWMeanThreads];
    double s = 0.0;
    for (long long i = threadIdx.x; i < nu; i += kWMeanThreads) s += G[i * nu + i];
    const double lambda = rho * block_sum_fixed<kWMeanThreads>(s, red) / static_cast<double>(nu);
    for (long long i = threadIdx.x; i < nu; i += kWMeanThreads) {
        const double d = G[i * nu + i] + lambda;
        G[i * nu + i] = d;
        diag0[i] = d;
    }
    if (threadIdx.x == 0) *flag = 0;
}

// ---------------------------------------------------------------------------------------------------------------
// Blocked right-looking Cholesky G = L L^T in place (lower triangle, row-major, ld n_u), tiles of kCholBlock.
// Step k: chol_panel_kernel (1 + row tiles below CTAs) factors the diagonal tile in shared memory in every CTA (the
// same arithmetic, so the same bits); CTA 0 raises the flag on a failed pivot, CTA r solves X L_kk^T = A for row tile
// r below it.  Every CTA reads A_kk from G, and the CTAs of one grid need not run at the same time, so no CTA of the
// panel launch may overwrite it: CTA 0 stores L_kk in the scratch tile Lkk, and chol_update_kernel (the next launch,
// which reads only the panel below) copies it into G while it subtracts L_I L_J^T from each trailing tile J <= I.  The
// last step has no panel below and no update; its panel launch is one CTA, which writes L_kk into G itself.
// ---------------------------------------------------------------------------------------------------------------
constexpr int kCholBlock = 64;
constexpr int kCholThreads = 256;
constexpr int kCholLd = kCholBlock + 1;
constexpr int kCholPanelSmem = 2 * kCholBlock * kCholLd * 8;

__global__ void __launch_bounds__(kCholThreads) chol_panel_kernel(double* __restrict__ G, long long nu, long long k0,
                                                                  const double* __restrict__ diag0, int* __restrict__ flag,
                                                                  double* __restrict__ Lkk) {
    extern __shared__ double cs[];
    double* D = cs;                          // diagonal tile [kCholBlock][kCholLd]
    double* X = cs + kCholBlock * kCholLd;   // panel row tile
    const int tid = threadIdx.x;
    const int bk = static_cast<int>(min(static_cast<long long>(kCholBlock), nu - k0));
    for (int e = tid; e < bk * bk; e += kCholThreads) {
        const int r = e / bk, c = e % bk;
        if (c <= r) D[r * kCholLd + c] = G[(k0 + r) * nu + k0 + c];
    }
    const long long r0 = k0 + bk + static_cast<long long>(blockIdx.x - 1) * kCholBlock;
    const int rows = blockIdx.x == 0 ? 0 : static_cast<int>(min(static_cast<long long>(kCholBlock), nu - r0));
    for (int e = tid; e < rows * bk; e += kCholThreads) {
        const int r = e / bk, c = e % bk;
        X[r * kCholLd + c] = G[(r0 + r) * nu + k0 + c];
    }
    __syncthreads();
    bool bad = false;
    for (int j = 0; j < bk; ++j) {
        const double d = D[j * kCholLd + j];
        bad |= !(d > kWienerPivotTol * diag0[k0 + j]);  // also NaN
        const double l = sqrt(d);
        __syncthreads();  // every thread has read d
        for (int i = j + 1 + tid; i < bk; i += kCholThreads) D[i * kCholLd + j] /= l;
        if (tid == 0) D[j * kCholLd + j] = l;
        __syncthreads();
        const int m = bk - j - 1;
        for (int e = tid; e < m * m; e += kCholThreads) {
            const int r = j + 1 + e / m, c = j + 1 + e % m;
            if (c <= r) D[r * kCholLd + c] = fma(-D[r * kCholLd + j], D[c * kCholLd + j], D[r * kCholLd + c]);
        }
        __syncthreads();
    }
    if (blockIdx.x == 0) {
        const bool alone = gridDim.x == 1;  // no other CTA reads A_kk: write L_kk in place
        for (int e = tid; e < bk * bk; e += kCholThreads) {
            const int r = e / bk, c = e % bk;
            if (c > r) continue;
            if (alone) G[(k0 + r) * nu + k0 + c] = D[r * kCholLd + c];
            else Lkk[r * kCholBlock + c] = D[r * kCholLd + c];
        }
        if (tid == 0 && bad) *flag = 1;
        return;
    }
    // X L^T = A, column by column: X[:, j] = A[:, j] / L_jj, then A[:, c] -= X[:, j] L_cj for c > j
    for (int j = 0; j < bk; ++j) {
        for (int r = tid; r < rows; r += kCholThreads) X[r * kCholLd + j] /= D[j * kCholLd + j];
        __syncthreads();
        const int m = bk - j - 1;
        for (int e = tid; e < rows * m; e += kCholThreads) {
            const int r = e / m, c = j + 1 + e % m;
            X[r * kCholLd + c] = fma(-X[r * kCholLd + j], D[c * kCholLd + j], X[r * kCholLd + c]);
        }
        __syncthreads();
    }
    for (int e = tid; e < rows * bk; e += kCholThreads) {
        const int r = e / bk, c = e % bk;
        G[(r0 + r) * nu + k0 + c] = X[r * kCholLd + c];
    }
}

constexpr int kCholChunk = 32;

__global__ void __launch_bounds__(kCholThreads) chol_update_kernel(double* __restrict__ G, long long nu, long long k0,
                                                                   const double* __restrict__ Lkk) {
    __shared__ double Li[kCholBlock][kCholChunk + 1], Lj[kCholBlock][kCholChunk + 1];
    const int tid = threadIdx.x, tx = tid % 16, ty = tid / 16;
    const int bk = static_cast<int>(min(static_cast<long long>(kCholBlock), nu - k0));
    if (blockIdx.x == 0) {  // the panel launch's factor of the diagonal tile; no CTA of this launch reads that tile
        for (int e = tid; e < bk * bk; e += kCholThreads) {
            const int r = e / bk, c = e % bk;
            if (c <= r) G[(k0 + r) * nu + k0 + c] = Lkk[r * kCholBlock + c];
        }
    }
    long long I = static_cast<long long>((sqrt(8.0 * blockIdx.x + 1.0) - 1.0) * 0.5);
    while (I * (I + 1) / 2 > blockIdx.x) --I;
    while ((I + 1) * (I + 2) / 2 <= blockIdx.x) ++I;
    const long long J = blockIdx.x - I * (I + 1) / 2;
    const long long ri = k0 + bk + I * kCholBlock, rj = k0 + bk + J * kCholBlock;
    const int ni = static_cast<int>(min(static_cast<long long>(kCholBlock), nu - ri));
    const int nj = static_cast<int>(min(static_cast<long long>(kCholBlock), nu - rj));
    double acc[4][4];
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < 4; ++v) acc[u][v] = 0.0;
    for (int m0 = 0; m0 < bk; m0 += kCholChunk) {
        __syncthreads();
        for (int e = tid; e < kCholBlock * kCholChunk; e += kCholThreads) {
            const int r = e / kCholChunk, m = e % kCholChunk;
            const bool in = m0 + m < bk;
            Li[r][m] = (in && r < ni) ? G[(ri + r) * nu + k0 + m0 + m] : 0.0;
            Lj[r][m] = (in && r < nj) ? G[(rj + r) * nu + k0 + m0 + m] : 0.0;
        }
        __syncthreads();
#pragma unroll 4
        for (int m = 0; m < kCholChunk; ++m) {
            double a[4], b[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) a[u] = Li[ty + 16 * u][m];
#pragma unroll
            for (int v = 0; v < 4; ++v) b[v] = Lj[tx + 16 * v][m];
#pragma unroll
            for (int u = 0; u < 4; ++u)
#pragma unroll
                for (int v = 0; v < 4; ++v) acc[u][v] = fma(a[u], b[v], acc[u][v]);
        }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < 4; ++v) {
            const int r = ty + 16 * u, c = tx + 16 * v;
            if (r < ni && c < nj && ri + r >= rj + c) G[(ri + r) * nu + rj + c] -= acc[u][v];
        }
}

// ---------------------------------------------------------------------------------------------------------------
// Solves, a CTA per target, in blocks of 32: the diagonal block by warp 0 with shuffles, the rest of the vector by
// the whole CTA.  rhs [cy][nu] holds p on entry and h on exit (NaN if the flag is set).
// ---------------------------------------------------------------------------------------------------------------
constexpr int kSolveThreads = 256;

__global__ void __launch_bounds__(kSolveThreads) wiener_solve_kernel(const double* __restrict__ G, long long nu,
                                                                     double* __restrict__ rhs, const int* __restrict__ flag) {
    __shared__ double z[kWienerMaxUnknowns];
    const int tid = threadIdx.x, lane = tid & 31;
    double* h = rhs + static_cast<long long>(blockIdx.x) * nu;
    if (*flag) {
        for (long long i = tid; i < nu; i += kSolveThreads) h[i] = __longlong_as_double(0x7ff8000000000000ll);
        return;
    }
    for (long long i = tid; i < nu; i += kSolveThreads) z[i] = h[i];
    __syncthreads();
    for (long long kb = 0; kb < nu; kb += 32) {  // L z = p
        const int bw = static_cast<int>(min(32ll, nu - kb));
        if (tid < 32) {
            double zl = lane < bw ? z[kb + lane] : 0.0;
            for (int c = 0; c < bw; ++c) {
                const double zc = __shfl_sync(0xffffffffu, zl, c) / G[(kb + c) * nu + kb + c];
                if (lane == c) zl = zc;
                if (lane > c && lane < bw) zl = fma(-G[(kb + lane) * nu + kb + c], zc, zl);
            }
            if (lane < bw) z[kb + lane] = zl;
        }
        __syncthreads();
        for (long long i = kb + bw + tid; i < nu; i += kSolveThreads) {
            double s = z[i];
            const double* row = G + i * nu + kb;
            for (int c = 0; c < bw; ++c) s = fma(-row[c], z[kb + c], s);
            z[i] = s;
        }
        __syncthreads();
    }
    for (long long kb = ((nu - 1) / 32) * 32; kb >= 0; kb -= 32) {  // L^T h = z
        const int bw = static_cast<int>(min(32ll, nu - kb));
        if (tid < 32) {
            double zl = lane < bw ? z[kb + lane] : 0.0;
            for (int c = bw - 1; c >= 0; --c) {
                const double hc = __shfl_sync(0xffffffffu, zl, c) / G[(kb + c) * nu + kb + c];
                if (lane == c) zl = hc;
                if (lane < c) zl = fma(-G[(kb + c) * nu + kb + lane], hc, zl);
            }
            if (lane < bw) z[kb + lane] = zl;
        }
        __syncthreads();
        for (long long i = tid; i < kb; i += kSolveThreads) {
            double s = z[i];
            for (int c = 0; c < bw; ++c) s = fma(-G[(kb + c) * nu + i], z[kb + c], s);
            z[i] = s;
        }
        __syncthreads();
    }
    for (long long i = tid; i < nu; i += kSolveThreads) h[i] = z[i];
}

// ---------------------------------------------------------------------------------------------------------------
// Apply: a CTA per (tile of kApplyTile outputs, group of kApplyTargets targets).  The group's filters sit in shared
// memory; the witnesses are staged kApplyChunk at a time over the tile plus its L-1 halo.  Thread p forms outputs p
// and p + 128 for the four targets, sum over a then k in order; e = y~ - yhat.  Per target the CTA's sum of e^2 goes
// to vpart[t][tile] (warp shuffle tree, then warps in order).
// ---------------------------------------------------------------------------------------------------------------
constexpr int kApplyThreads = 128;
constexpr int kApplyTile = 2 * kApplyThreads;
constexpr int kApplyTargets = 4;
constexpr int kApplyStageDoubles = 8192;   // 64 KB of witness staging

struct ApplyParams {
    WienerSeries S;
    long long L, nu, n0, M;
    int chunk;                 // witnesses staged at once
    const double* h;           // [cy][nu]
    const int* flag;
    double* res;               // [cy][ld_res] or null
    long long ld_res;
    double* vpart;             // [cy][tiles] or null
    long long tiles;
};

__global__ void __launch_bounds__(kApplyThreads) wiener_apply_kernel(const ApplyParams A) {
    extern __shared__ double sh[];
    double* hs = sh;                                  // [kApplyTargets][nu]
    double* xs = sh + kApplyTargets * A.nu;           // [chunk][kApplyTile + L - 1]
    __shared__ double red[kApplyThreads / 32][kApplyTargets];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long i0 = static_cast<long long>(blockIdx.x) * kApplyTile;
    const long long t0 = static_cast<long long>(blockIdx.y) * kApplyTargets;
    const long long L = A.L, nu = A.nu, cx = A.S.cx, cy = A.S.cy, N = A.S.N;
    const long long span = kApplyTile + L - 1;
    for (long long e = tid; e < kApplyTargets * nu; e += kApplyThreads) {
        const long long g = e / nu;
        hs[e] = t0 + g < cy ? A.h[(t0 + g) * nu + e % nu] : 0.0;
    }
    double acc[kApplyTargets][2];
#pragma unroll
    for (int g = 0; g < kApplyTargets; ++g) acc[g][0] = acc[g][1] = 0.0;
    for (long long a0 = 0; a0 < cx; a0 += A.chunk) {
        const int na = static_cast<int>(min(static_cast<long long>(A.chunk), cx - a0));
        __syncthreads();
        for (long long e = tid; e < na * span; e += kApplyThreads) {
            const long long a = e / span, u = e % span, q = i0 + u;  // x~_a[n0 + i + k0 - k] = xs[a][i - i0 + L-1-k]
            xs[e] = q < N ? A.S.at(a0 + a, q) : 0.0;
        }
        __syncthreads();
        for (int a = 0; a < na; ++a) {
            const double* xa = xs + a * span + tid + L - 1;
            const double* ha = hs + (a0 + a) * L;
            for (long long k = 0; k < L; ++k) {
                const double x0 = xa[-k], x1 = xa[kApplyThreads - k];
#pragma unroll
                for (int g = 0; g < kApplyTargets; ++g) {
                    const double hv = ha[g * nu + k];
                    acc[g][0] = fma(hv, x0, acc[g][0]);
                    acc[g][1] = fma(hv, x1, acc[g][1]);
                }
            }
        }
    }
    const bool bad = *A.flag != 0;
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    double ss[kApplyTargets];
#pragma unroll
    for (int g = 0; g < kApplyTargets; ++g) {
        ss[g] = 0.0;
        const long long t = t0 + g;
#pragma unroll
        for (int v = 0; v < 2; ++v) {
            const long long i = i0 + tid + v * kApplyThreads;
            if (t < cy && i < A.M) {
                const double e = bad ? nan : A.S.at(cx + t, A.n0 + i) - acc[g][v];
                if (A.res) A.res[t * A.ld_res + i] = e;
                ss[g] = fma(e, e, ss[g]);
            }
        }
    }
    if (!A.vpart) return;
#pragma unroll
    for (int g = 0; g < kApplyTargets; ++g) {
        double v = ss[g];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
        if (lane == 0) red[warp][g] = v;
    }
    __syncthreads();
    if (tid < kApplyTargets && t0 + tid < cy)
        A.vpart[(t0 + tid) * A.tiles + blockIdx.x] = (red[0][tid] + red[1][tid]) + (red[2][tid] + red[3][tid]);
}

__global__ void __launch_bounds__(128) wiener_var_kernel(const double* __restrict__ vpart, long long tiles, long long cy,
                                                         long long M, double* __restrict__ var_res) {
    const long long t = static_cast<long long>(blockIdx.x) * 128 + threadIdx.x;
    if (t >= cy) return;
    double s = 0.0;
    for (long long i = 0; i < tiles; ++i) s += vpart[t * tiles + i];
    var_res[t] = s / static_cast<double>(M);
}

}  // namespace dfk
