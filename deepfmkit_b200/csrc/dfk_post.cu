// Post-fit entries of the C ABI (include/dfk_b200.h, "post-fit step"): block means, log-frequency spectra,
// time-domain witness subtraction and time-domain stability.
#include "dfk_host.h"

#include <cmath>
#include <vector>

#include "dfk_spectra.cuh"
#include "dfk_stability.cuh"
#include "dfk_wiener.cuh"

namespace {

double kaiser_alpha(double psll) {
    const double x = psll / 100.0;
    return ((0.0889732 * x - 0.493285) * x + 4.71469) * x - 0.0821377;
}

double kaiser_rov(double alpha) {
    const double x = alpha;
    return (100.0 - 1.0 / (((4.42204e-05 * x - 0.000925946) * x + 0.00912223) * x + 0.0061076)) / 100.0;
}

double host_i0(double x) {
    const double q = 0.25 * x * x;
    double term = 1.0, sum = 1.0;
    for (int k = 1; k < 500; ++k) {
        term *= q / (static_cast<double>(k) * static_cast<double>(k));
        sum += term;
        if (term < 1e-17 * sum) break;
    }
    return sum;
}

struct PlanRow {
    double f, r, m;
    int64_t L, K;
};

double resolve_olap(const dfk_lpsd_opts& o) {
    if (o.olap >= 0.0) return o.olap;
    return o.window == 0 ? kaiser_rov(kaiser_alpha(o.psll)) : 0.5;
}

// The LTPDA scheduler (ltf_plan): log-spaced frequencies whose resolution follows the frequency until the desired
// number of averages can no longer be met, then a geometric compromise, never finer than fs / N.
int make_plan(int64_t N, double fs, const dfk_lpsd_opts& o, std::vector<PlanRow>& rows) {
    if (N < 2) return fail(DFK_ERR_ARG, "LPSD needs at least 2 samples");
    if (!(fs > 0.0)) return fail(DFK_ERR_ARG, "fs must be positive");
    if (o.jdes < 1 || o.kdes < 1 || !(o.bmin > 0.0)) return fail(DFK_ERR_ARG, "Jdes, Kdes and bmin must be positive");
    if (o.order < -1 || o.order > 2) return fail(DFK_ERR_ARG, "detrend order %d outside -1..2", o.order);
    if (o.window != 0 && o.window != 1) return fail(DFK_ERR_ARG, "unknown window %d", o.window);
    const double olap = resolve_olap(o);
    if (!(olap < 1.0)) return fail(DFK_ERR_ARG, "overlap must be below 1");
    const double xov = 1.0 - olap;
    const double nd = static_cast<double>(N);
    const double fmin = fs / nd * o.bmin, fmax = fs / 2.0, fresmin = fs / nd;
    const double freslim = fresmin * (1.0 + xov * (o.kdes - 1));
    const double logfact = std::pow(nd / 2.0, 1.0 / o.jdes) - 1.0;
    rows.clear();
    double fi = fmin;
    while (fi < fmax) {
        double fres = fi * logfact;
        if (fres <= freslim) fres = std::sqrt(fres * freslim);
        if (fres < fresmin) fres = fresmin;
        double fbin = fi / fres;
        if (fbin < o.bmin) {
            fbin = o.bmin;
            fres = fi / fbin;
        }
        int64_t dftlen = static_cast<int64_t>(std::floor(fs / fres + 0.5));
        if (dftlen > N) dftlen = N;
        if (dftlen < o.lmin) dftlen = o.lmin;
        if (dftlen < 1) dftlen = 1;
        int64_t nseg = static_cast<int64_t>(std::floor(static_cast<double>(N - dftlen) / (xov * dftlen) + 1.0 + 0.5));
        if (nseg <= 1) {
            nseg = 1;
            dftlen = N;
        }
        fres = fs / static_cast<double>(dftlen);
        fbin = fi / fres;
        rows.push_back({fi, fres, fbin, dftlen, nseg});
        fi += fres;
        if (rows.size() > (1u << 22)) return fail(DFK_ERR_ARG, "LPSD plan does not terminate");
    }
    return DFK_OK;
}

// The device plan of one LPSD / LCSD call, built in one place so that both estimates use the same segments.
struct DevicePlan {
    std::vector<PlanRow> rows;          // make_plan's rows, K trimmed as below
    std::vector<dfk::LpsdFreq> freq;
    long long tiles = 0, groups = 0;    // per series
};

int make_device_plan(int64_t N, double fs, const dfk_lpsd_opts& o, DevicePlan& dp) {
    const int rc = make_plan(N, fs, o, dp.rows);
    if (rc) return rc;
    const int nf = static_cast<int>(dp.rows.size());
    dp.freq.resize(nf);
    dp.tiles = dp.groups = 0;
    for (int j = 0; j < nf; ++j) {
        dfk::LpsdFreq& F = dp.freq[j];
        PlanRow& row = dp.rows[j];
        F.L = row.L;
        F.K = row.K;
        F.p = 2.0 * dfk::kPi * row.m / static_cast<double>(row.L);
        double shift = F.K == 1 ? 1.0 : static_cast<double>(N - F.L) / static_cast<double>(F.K - 1);
        if (shift < 1.0) shift = 1.0;
        F.shift = shift;
        // the last segment must stay inside the record whatever the rounding of the plan
        while (F.K > 1 && static_cast<long long>(std::floor((F.K - 1) * shift + 0.5)) + F.L > N) F.K--;
        row.K = F.K;
        const long long ng = (F.K + dfk::kLpsdGroup - 1) / dfk::kLpsdGroup;
        F.tile0 = dp.tiles;
        F.group0 = dp.groups;
        dp.tiles += F.L >= dfk::kLpsdCtaMin ? ng : (ng + dfk::kLpsdThreads / 32 - 1) / (dfk::kLpsdThreads / 32);
        dp.groups += ng;
    }
    return DFK_OK;
}

// Kernel parameters of a plan already copied to plan_dev; the caller sets the series and the scratch.
dfk::LpsdParams lpsd_params(const DevicePlan& dp, const void* plan_dev, int64_t N, int64_t stride,
                            const dfk_lpsd_opts& o) {
    dfk::LpsdParams P;
    P.x = nullptr;
    P.N = N;
    P.stride = stride;
    P.ld_c = 0;
    P.plan = static_cast<const dfk::LpsdFreq*>(plan_dev);
    P.nf = static_cast<int>(dp.freq.size());
    P.ntiles = dp.tiles;
    P.ngroups = dp.groups;
    P.order = o.order;
    P.window = o.window;
    P.beta = dfk::kPi * kaiser_alpha(o.psll);
    P.inv_i0_beta = 1.0 / host_i0(P.beta);
    P.group_sum = nullptr;
    return P;
}

void copy_plan_out(const DevicePlan& dp, double* f_host, int64_t* navs_host) {
    for (size_t j = 0; j < dp.rows.size(); ++j) {
        if (f_host) f_host[j] = dp.rows[j].f;
        if (navs_host) navs_host[j] = dp.rows[j].K;
    }
}

}  // namespace

extern "C" {

void dfk_default_lpsd_opts(dfk_lpsd_opts* o) {
    if (!o) return;
    o->olap = -1.0;  // "default": the window's recommended overlap (data.py:150)
    o->bmin = 1.0;
    o->lmin = 0;
    o->jdes = 500;
    o->kdes = 100;
    o->order = 0;
    o->window = 0;
    o->psll = 200.0;
}

int dfk_lpsd_plan(int64_t N, double fs, const dfk_lpsd_opts* opts, int32_t cap, int32_t* nf, double* f, double* r,
                  double* m, int64_t* L, int64_t* K) {
    dfk_lpsd_opts d;
    if (!opts) {
        dfk_default_lpsd_opts(&d);
        opts = &d;
    }
    if (!nf) return fail(DFK_ERR_ARG, "null output pointer");
    std::vector<PlanRow> rows;
    const int rc = make_plan(N, fs, *opts, rows);
    if (rc) return rc;
    *nf = static_cast<int32_t>(rows.size());
    for (int32_t j = 0; j < *nf && j < cap; ++j) {
        if (f) f[j] = rows[j].f;
        if (r) r[j] = rows[j].r;
        if (m) m[j] = rows[j].m;
        if (L) L[j] = rows[j].L;
        if (K) K[j] = rows[j].K;
    }
    return DFK_OK;
}

int dfk_lpsd_dev(dfk_ctx* ctx, const double* x_dev, int64_t N, int64_t stride, int64_t C, int64_t ld_c, double fs,
                 const dfk_lpsd_opts* opts, int32_t cap, int32_t* nf_out, double* f_host, double* ps_host, double* psd_host,
                 double* enbw_host, int64_t* navs_host) {
    DFK_ENTER(ctx);
    dfk_lpsd_opts d;
    if (!opts) {
        dfk_default_lpsd_opts(&d);
        opts = &d;
    }
    if (!x_dev || !nf_out) return fail(DFK_ERR_ARG, "null pointer");
    if (C < 1 || stride < 1) return fail(DFK_ERR_ARG, "bad geometry: C=%lld stride=%lld", (long long)C, (long long)stride);
    DevicePlan dp;
    int rc = make_device_plan(N, fs, *opts, dp);
    if (rc) return rc;
    const int nf = static_cast<int>(dp.rows.size());
    *nf_out = nf;
    if (nf > cap) return fail(DFK_ERR_ARG, "plan has %d frequencies, outputs hold %d (call dfk_lpsd_plan first)", nf, cap);
    if (nf == 0) return DFK_OK;
    const long long tiles = dp.tiles, groups = dp.groups;
    if (tiles > 0x7fffffffll || C > 65535) return fail(DFK_ERR_ARG, "LPSD problem too large for one launch");
    DevBuf& plan_dev = ctx->post[0];
    DevBuf& group_dev = ctx->post[1];
    DevBuf& out_dev = ctx->post[2];
    rc = ensure(ctx, plan_dev, sizeof(dfk::LpsdFreq) * nf);
    if (!rc) rc = ensure(ctx, group_dev, sizeof(double) * groups * C);
    if (!rc) rc = ensure(ctx, out_dev, sizeof(double) * (2 * C + 1) * nf);
    if (rc) return rc;
    cudaStream_t st = ctx->stream();
    DFK_CUDA(cudaMemcpyAsync(plan_dev.ptr, dp.freq.data(), sizeof(dfk::LpsdFreq) * nf, cudaMemcpyHostToDevice, st));
    dfk::LpsdParams P = lpsd_params(dp, plan_dev.ptr, N, stride, *opts);
    P.x = x_dev;
    P.ld_c = ld_c;
    P.group_sum = static_cast<double*>(group_dev.ptr);
    double* ps_dev = static_cast<double*>(out_dev.ptr);
    double* psd_dev = ps_dev + C * nf;
    double* enbw_dev = psd_dev + C * nf;
    const dim3 grid(static_cast<unsigned>(tiles), static_cast<unsigned>(C));
    dfk::lpsd_segment_kernel<<<grid, dfk::kLpsdThreads, 0, st>>>(P);
    DFK_CUDA(cudaGetLastError());
    dfk::lpsd_finish_kernel<<<nf, 128, 0, st>>>(P, C, fs, ps_dev, psd_dev, enbw_dev);
    DFK_CUDA(cudaGetLastError());
    ctx->launches += 2;
    if (ps_host) DFK_CUDA(cudaMemcpyAsync(ps_host, ps_dev, sizeof(double) * C * nf, cudaMemcpyDeviceToHost, st));
    if (psd_host) DFK_CUDA(cudaMemcpyAsync(psd_host, psd_dev, sizeof(double) * C * nf, cudaMemcpyDeviceToHost, st));
    if (enbw_host) DFK_CUDA(cudaMemcpyAsync(enbw_host, enbw_dev, sizeof(double) * nf, cudaMemcpyDeviceToHost, st));
    DFK_CUDA(cudaStreamSynchronize(st));
    copy_plan_out(dp, f_host, navs_host);
    return DFK_OK;
}

int dfk_lcsd_dev(dfk_ctx* ctx, const double* x_dev, int64_t Cx, int64_t ldx, const double* y_dev, int64_t Cy,
                 int64_t ldy, int64_t N, int64_t stride, double fs, const dfk_lpsd_opts* opts, int32_t cap,
                 int32_t* nf_out, double* f_host, double* sxx_host, double* syy_host, double* sxy_host,
                 double* enbw_host, int64_t* navs_host) {
    DFK_ENTER(ctx);
    dfk_lpsd_opts d;
    if (!opts) {
        dfk_default_lpsd_opts(&d);
        opts = &d;
    }
    if (!x_dev || !y_dev || !nf_out) return fail(DFK_ERR_ARG, "null pointer");
    if (Cx < 1 || Cy < 1 || stride < 1)
        return fail(DFK_ERR_ARG, "bad geometry: Cx=%lld Cy=%lld stride=%lld", (long long)Cx, (long long)Cy,
                    (long long)stride);
    if (Cx + Cy > 65535) return fail(DFK_ERR_ARG, "LCSD takes at most 65535 series in all (Cx + Cy)");
    DevicePlan dp;
    int rc = make_device_plan(N, fs, *opts, dp);
    if (rc) return rc;
    const int nf = static_cast<int>(dp.rows.size());
    *nf_out = nf;
    if (nf > cap) return fail(DFK_ERR_ARG, "plan has %d frequencies, outputs hold %d (call dfk_lpsd_plan first)", nf, cap);
    if (nf == 0) return DFK_OK;
    if (dp.tiles > 0x7fffffffll) return fail(DFK_ERR_ARG, "LCSD problem too large for one launch");
    const long long ns = Cx + Cy, npair = Cx * Cy;
    const long long nslots = dp.groups * dfk::kLpsdGroup;
    DevBuf& plan_dev = ctx->post[0];
    DevBuf& seg_dev = ctx->post[1];
    DevBuf& out_dev = ctx->post[2];
    // per-segment projections: 16 B per slot and series; outputs: auto densities, cross densities (re, im), ENBW
    rc = ensure(ctx, plan_dev, sizeof(dfk::LpsdFreq) * nf);
    if (!rc) rc = ensure(ctx, seg_dev, sizeof(double2) * static_cast<size_t>(nslots) * static_cast<size_t>(ns));
    if (!rc) rc = ensure(ctx, out_dev, sizeof(double) * static_cast<size_t>(ns + 2 * npair + 1) * static_cast<size_t>(nf));
    if (rc) return rc;
    cudaStream_t st = ctx->stream();
    DFK_CUDA(cudaMemcpyAsync(plan_dev.ptr, dp.freq.data(), sizeof(dfk::LpsdFreq) * nf, cudaMemcpyHostToDevice, st));
    dfk::LcsdParams Q;
    Q.P = lpsd_params(dp, plan_dev.ptr, N, stride, *opts);
    Q.P.x = x_dev;
    Q.P.ld_c = ldx;
    Q.y = y_dev;
    Q.ld_y = ldy;
    Q.cx = Cx;
    Q.cy = Cy;
    Q.seg = static_cast<double2*>(seg_dev.ptr);
    Q.nslots = nslots;
    double* psd_dev = static_cast<double*>(out_dev.ptr);  // [Cx + Cy][nf]: x series, then y
    double* sxy_dev = psd_dev + ns * nf;                    // [Cx][Cy][nf][2]
    double* enbw_dev = sxy_dev + 2 * npair * nf;
    const dim3 grid(static_cast<unsigned>(dp.tiles), static_cast<unsigned>(ns));
    dfk::lcsd_segment_kernel<<<grid, dfk::kLpsdThreads, 0, st>>>(Q);
    DFK_CUDA(cudaGetLastError());
    dfk::lcsd_finish_kernel<<<nf, dfk::kLcsdFinishThreads, 0, st>>>(Q, fs, psd_dev, sxy_dev, enbw_dev);
    DFK_CUDA(cudaGetLastError());
    ctx->launches += 2;
    if (sxx_host) DFK_CUDA(cudaMemcpyAsync(sxx_host, psd_dev, sizeof(double) * Cx * nf, cudaMemcpyDeviceToHost, st));
    if (syy_host)
        DFK_CUDA(cudaMemcpyAsync(syy_host, psd_dev + Cx * nf, sizeof(double) * Cy * nf, cudaMemcpyDeviceToHost, st));
    if (sxy_host) DFK_CUDA(cudaMemcpyAsync(sxy_host, sxy_dev, sizeof(double) * 2 * npair * nf, cudaMemcpyDeviceToHost, st));
    if (enbw_host) DFK_CUDA(cudaMemcpyAsync(enbw_host, enbw_dev, sizeof(double) * nf, cudaMemcpyDeviceToHost, st));
    DFK_CUDA(cudaStreamSynchronize(st));
    copy_plan_out(dp, f_host, navs_host);
    return DFK_OK;
}

int dfk_lcsd_cond_dev(dfk_ctx* ctx, const double* x_dev, int64_t Cx, int64_t ldx, const double* y_dev, int64_t Cy,
                      int64_t ldy, int64_t N, int64_t stride, double fs, const dfk_lpsd_opts* opts, int32_t cap,
                      int32_t* nf_out, double* f_host, double* sxx_host, double* syy_host, double* sxy_host,
                      double* h_host, double* sres_host, double* mcoh_host, double* enbw_host, int64_t* navs_host) {
    DFK_ENTER(ctx);
    dfk_lpsd_opts d;
    if (!opts) {
        dfk_default_lpsd_opts(&d);
        opts = &d;
    }
    if (!x_dev || !y_dev || !nf_out) return fail(DFK_ERR_ARG, "null pointer");
    if (Cx < 1 || Cx > dfk::kCondMaxWitnesses || Cy < 1 || stride < 1)
        return fail(DFK_ERR_ARG, "bad geometry: Cx=%lld (1..%d) Cy=%lld stride=%lld", (long long)Cx,
                    dfk::kCondMaxWitnesses, (long long)Cy, (long long)stride);
    if (Cx + Cy > 65535) return fail(DFK_ERR_ARG, "conditioned spectra take at most 65535 series in all (Cx + Cy)");
    DevicePlan dp;
    int rc = make_device_plan(N, fs, *opts, dp);
    if (rc) return rc;
    const int nf = static_cast<int>(dp.rows.size());
    *nf_out = nf;
    if (nf > cap) return fail(DFK_ERR_ARG, "plan has %d frequencies, outputs hold %d (call dfk_lpsd_plan first)", nf, cap);
    if (nf == 0) return DFK_OK;
    const long long ns = Cx + Cy, npair = Cx * Cy;
    const long long row_tiles = (Cx + dfk::kGramRows - 1) / dfk::kGramRows;
    const long long col_tiles = (ns + dfk::kGramCols - 1) / dfk::kGramCols;
    const long long gram_tiles = row_tiles * col_tiles + (Cy + dfk::kGramCols - 1) / dfk::kGramCols;
    if (dp.tiles > 0x7fffffffll || gram_tiles > 0x7fffffffll)
        return fail(DFK_ERR_ARG, "conditioned-spectra problem too large for one launch");
    const long long nslots = dp.groups * dfk::kLpsdGroup;
    DevBuf& plan_dev = ctx->post[0];
    DevBuf& seg_dev = ctx->post[1];
    DevBuf& out_dev = ctx->post[2];
    // outputs: Sxx (re, im), Syy, Sxy (re, im), H (re, im), Sres, mcoh, ENBW
    const size_t out_doubles = static_cast<size_t>(2 * Cx * Cx + 3 * Cy + 4 * npair + 1) * static_cast<size_t>(nf);
    rc = ensure(ctx, plan_dev, sizeof(dfk::LpsdFreq) * nf);
    if (!rc) rc = ensure(ctx, seg_dev, sizeof(double2) * static_cast<size_t>(nslots) * static_cast<size_t>(ns));
    if (!rc) rc = ensure(ctx, out_dev, sizeof(double) * out_doubles);
    if (rc) return rc;
    cudaStream_t st = ctx->stream();
    DFK_CUDA(cudaMemcpyAsync(plan_dev.ptr, dp.freq.data(), sizeof(dfk::LpsdFreq) * nf, cudaMemcpyHostToDevice, st));
    dfk::LcsdParams Q;
    Q.P = lpsd_params(dp, plan_dev.ptr, N, stride, *opts);
    Q.P.x = x_dev;
    Q.P.ld_c = ldx;
    Q.y = y_dev;
    Q.ld_y = ldy;
    Q.cx = Cx;
    Q.cy = Cy;
    Q.seg = static_cast<double2*>(seg_dev.ptr);
    Q.nslots = nslots;
    double* sxx_dev = static_cast<double*>(out_dev.ptr);  // [Cx][Cx][nf][2]
    double* syy_dev = sxx_dev + 2 * Cx * Cx * nf;          // [Cy][nf]
    double* sxy_dev = syy_dev + Cy * nf;                   // [Cx][Cy][nf][2]
    double* h_dev = sxy_dev + 2 * npair * nf;              // [Cx][Cy][nf][2]
    double* sres_dev = h_dev + 2 * npair * nf;             // [Cy][nf]
    double* mcoh_dev = sres_dev + Cy * nf;                 // [Cy][nf]
    double* enbw_dev = mcoh_dev + Cy * nf;
    dfk::GramParams G;
    G.seg = Q.seg;
    G.nslots = nslots;
    G.plan = Q.P.plan;
    G.nf = nf;
    G.cx = Cx;
    G.cy = Cy;
    G.row_tiles = row_tiles;
    G.col_tiles = col_tiles;
    G.sxx = sxx_dev;
    G.syy = syy_dev;
    G.sxy = sxy_dev;
    dfk::CondParams C;
    C.P = Q.P;
    C.cx = Cx;
    C.cy = Cy;
    C.fs = fs;
    C.sxx = sxx_dev;
    C.syy = syy_dev;
    C.sxy = sxy_dev;
    C.h = h_dev;
    C.sres = sres_dev;
    C.mcoh = mcoh_dev;
    C.enbw = enbw_dev;
    const size_t cond_smem = sizeof(double2) * static_cast<size_t>(Cx) * static_cast<size_t>(Cx + 1);
    DFK_CUDA(cudaFuncSetAttribute(dfk::lcsd_cond_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  static_cast<int>(cond_smem)));
    const dim3 seg_grid(static_cast<unsigned>(dp.tiles), static_cast<unsigned>(ns));
    dfk::lcsd_segment_kernel<<<seg_grid, dfk::kLpsdThreads, 0, st>>>(Q);
    DFK_CUDA(cudaGetLastError());
    const dim3 gram_grid(static_cast<unsigned>(gram_tiles), static_cast<unsigned>(std::min(nf, 65535)));
    dfk::lcsd_gram_kernel<<<gram_grid, dfk::kGramThreads, 0, st>>>(G);
    DFK_CUDA(cudaGetLastError());
    dfk::lcsd_cond_kernel<<<nf, dfk::kCondThreads, cond_smem, st>>>(C);
    DFK_CUDA(cudaGetLastError());
    ctx->launches += 3;
    auto out = [&](double* host, const double* dev, long long n) -> int {
        if (host) DFK_CUDA(cudaMemcpyAsync(host, dev, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
        return DFK_OK;
    };
    rc = out(sxx_host, sxx_dev, 2 * Cx * Cx * nf);
    if (!rc) rc = out(syy_host, syy_dev, Cy * nf);
    if (!rc) rc = out(sxy_host, sxy_dev, 2 * npair * nf);
    if (!rc) rc = out(h_host, h_dev, 2 * npair * nf);
    if (!rc) rc = out(sres_host, sres_dev, Cy * nf);
    if (!rc) rc = out(mcoh_host, mcoh_dev, Cy * nf);
    if (!rc) rc = out(enbw_host, enbw_dev, nf);
    if (rc) return rc;
    DFK_CUDA(cudaStreamSynchronize(st));
    copy_plan_out(dp, f_host, navs_host);
    return DFK_OK;
}

int dfk_wiener_dev(dfk_ctx* ctx, const double* x_dev, int64_t Cx, int64_t ldx, const double* y_dev, int64_t Cy,
                   int64_t ldy, int64_t N, int64_t stride, int64_t L, int64_t lead, double ridge, double* res_dev,
                   int64_t ld_res, double* h_host, double* var_y_host, double* var_res_host, int32_t* singular_out) {
    DFK_ENTER(ctx);
    if (!x_dev || !y_dev) return fail(DFK_ERR_ARG, "null pointer");
    if (Cx < 1 || Cx > dfk::kWienerMaxWitnesses || Cy < 1 || Cx + Cy > 65535 || stride < 1)
        return fail(DFK_ERR_ARG, "bad geometry: Cx=%lld (1..%d) Cy=%lld (Cx + Cy <= 65535) stride=%lld", (long long)Cx,
                    dfk::kWienerMaxWitnesses, (long long)Cy, (long long)stride);
    if (L < 1 || L > dfk::kWienerMaxUnknowns || Cx * L > dfk::kWienerMaxUnknowns)
        return fail(DFK_ERR_ARG, "bad filter length: L=%lld, Cx L=%lld (at most %d)", (long long)L, (long long)(Cx * L),
                    dfk::kWienerMaxUnknowns);
    if (lead < 0 || lead > L - 1) return fail(DFK_ERR_ARG, "lead %lld outside 0..%lld", (long long)lead, (long long)(L - 1));
    if (!(ridge >= 0.0) || !std::isfinite(ridge)) return fail(DFK_ERR_ARG, "ridge must be finite and >= 0");
    const long long nu = Cx * L, M = N - L + 1, n0 = L - 1 - lead;
    if (M < nu)
        return fail(DFK_ERR_ARG, "N=%lld gives %lld rows for %lld unknowns (need N >= Cx L + L - 1)", (long long)N, M, nu);
    if (res_dev && (Cy > 1 && ld_res < M))
        return fail(DFK_ERR_ARG, "ld_res=%lld below the %lld residual samples", (long long)ld_res, M);
    const long long ns = Cx + Cy;
    // lag sums: column tiles, chunk length T sized so that the staging fits 48 KB, slices for about 2048 CTAs
    dfk::LagParams P;
    P.S.x = x_dev;
    P.S.y = y_dev;
    P.S.ldx = ldx;
    P.S.ldy = ldy;
    P.S.stride = stride;
    P.S.cx = Cx;
    P.S.cy = Cy;
    P.S.N = N;
    P.L = L;
    P.k0 = lead;
    P.ncx = Cx * (2 * L - 1);
    P.ncols = P.ncx + Cy * L;
    P.col_tiles = (P.ncols + dfk::kLagCols - 1) / dfk::kLagCols;
    const long long row_tiles = (Cx + dfk::kLagRows - 1) / dfk::kLagRows, tiles = row_tiles * P.col_tiles;
    long long nser = 1;
    for (long long ct = 0; ct < P.col_tiles; ++ct) {
        const long long c0 = ct * dfk::kLagCols, c1 = std::min(c0 + dfk::kLagCols, P.ncols) - 1;
        nser = std::max(nser, dfk::lag_col_series(c1, Cx, P.ncx, L) - dfk::lag_col_series(c0, Cx, P.ncx, L) + 1);
    }
    constexpr long long kStage = 6144;
    long long T = (kStage - dfk::kLagCols + nser) / (dfk::kLagRows + nser);
    T = std::max(4ll, std::min(512ll, T & ~3ll));
    P.T = static_cast<int>(T);
    P.q_begin = L - 1;
    P.q_end = N - L + 1;
    const long long Q = P.q_end - P.q_begin;
    long long nslices = std::max(1ll, std::min((2048 + tiles - 1) / tiles, (Q + T - 1) / T));
    P.slice = (((Q + nslices - 1) / nslices + T - 1) / T) * T;
    nslices = (Q + P.slice - 1) / P.slice;
    P.part_stride = tiles * dfk::kLagTileEntries;
    const size_t lag_smem =
        sizeof(double) * static_cast<size_t>(std::max(dfk::kLagRows * T + nser * (T - 1) + dfk::kLagCols,
                                                      static_cast<long long>(4 * dfk::kLagTileEntries)));
    const long long apply_tiles = (M + dfk::kApplyTile - 1) / dfk::kApplyTile;
    if (tiles > 0x7fffffffll || nslices > 65535 || apply_tiles > 0x7fffffffll)
        return fail(DFK_ERR_ARG, "Wiener problem too large for one launch");
    const bool apply = res_dev || var_res_host;
    // post[0]: means [ns], var_y [Cy], var_res [Cy], diag0 [nu], the factored diagonal tile of the current Cholesky
    // step [64][64], tile sums of e^2 [Cy][apply_tiles], flag
    // post[1]: lag-sum slice partials; post[2]: G [nu][nu], then p / h [Cy][nu]
    DevBuf& small_dev = ctx->post[0];
    DevBuf& part_dev = ctx->post[1];
    DevBuf& mat_dev = ctx->post[2];
    const size_t small_doubles =
        static_cast<size_t>(ns + 2 * Cy + nu + dfk::kCholBlock * dfk::kCholBlock + Cy * apply_tiles + 1);
    int rc = ensure(ctx, small_dev, sizeof(double) * small_doubles);
    if (!rc) rc = ensure(ctx, part_dev, sizeof(double) * static_cast<size_t>(nslices) * static_cast<size_t>(P.part_stride));
    if (!rc) rc = ensure(ctx, mat_dev, sizeof(double) * static_cast<size_t>(nu) * static_cast<size_t>(nu + Cy));
    if (rc) return rc;
    double* mean_dev = static_cast<double*>(small_dev.ptr);
    double* var_y_dev = mean_dev + ns;
    double* var_res_dev = var_y_dev + Cy;
    double* diag0_dev = var_res_dev + Cy;
    double* lkk_dev = diag0_dev + nu;
    double* vpart_dev = lkk_dev + dfk::kCholBlock * dfk::kCholBlock;
    int* flag_dev = reinterpret_cast<int*>(vpart_dev + Cy * apply_tiles);
    double* G_dev = static_cast<double*>(mat_dev.ptr);
    double* rhs_dev = G_dev + nu * nu;
    P.S.mean = mean_dev;
    P.part = static_cast<double*>(part_dev.ptr);
    cudaStream_t st = ctx->stream();
    long long launches = 0;

    dfk::wiener_means_kernel<<<static_cast<unsigned>(ns), dfk::kWMeanThreads, 0, st>>>(P.S, n0, M, mean_dev, var_y_dev);
    DFK_CUDA(cudaGetLastError());
    DFK_CUDA(cudaFuncSetAttribute(dfk::wiener_lag_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  static_cast<int>(lag_smem)));
    dfk::wiener_lag_kernel<<<dim3(static_cast<unsigned>(tiles), static_cast<unsigned>(nslices)), dfk::kLagThreads,
                             lag_smem, st>>>(P);
    DFK_CUDA(cudaGetLastError());
    dfk::AssembleParams A;
    A.P = P;
    A.nslices = nslices;
    A.nu = nu;
    A.G = G_dev;
    A.rhs = rhs_dev;
    const long long assemble_threads = nu * (nu + Cy);
    dfk::wiener_assemble_kernel<<<static_cast<unsigned>((assemble_threads + dfk::kAssembleThreads - 1) /
                                                        dfk::kAssembleThreads),
                                  dfk::kAssembleThreads, 0, st>>>(A);
    DFK_CUDA(cudaGetLastError());
    dfk::wiener_load_kernel<<<1, dfk::kWMeanThreads, 0, st>>>(G_dev, nu, ridge, diag0_dev, flag_dev);
    DFK_CUDA(cudaGetLastError());
    launches += 4;
    DFK_CUDA(cudaFuncSetAttribute(dfk::chol_panel_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  dfk::kCholPanelSmem));
    for (long long k0 = 0; k0 < nu; k0 += dfk::kCholBlock) {
        const long long below = nu - std::min(nu, k0 + dfk::kCholBlock);
        const long long bt = (below + dfk::kCholBlock - 1) / dfk::kCholBlock;
        dfk::chol_panel_kernel<<<static_cast<unsigned>(1 + bt), dfk::kCholThreads, dfk::kCholPanelSmem, st>>>(
            G_dev, nu, k0, diag0_dev, flag_dev, lkk_dev);
        DFK_CUDA(cudaGetLastError());
        ++launches;
        if (bt == 0) break;
        const unsigned update_tiles = static_cast<unsigned>(bt * (bt + 1) / 2);
        dfk::chol_update_kernel<<<update_tiles, dfk::kCholThreads, 0, st>>>(G_dev, nu, k0, lkk_dev);
        DFK_CUDA(cudaGetLastError());
        ++launches;
    }
    dfk::wiener_solve_kernel<<<static_cast<unsigned>(Cy), dfk::kSolveThreads, 0, st>>>(G_dev, nu, rhs_dev, flag_dev);
    DFK_CUDA(cudaGetLastError());
    ++launches;
    if (apply) {
        dfk::ApplyParams Y;
        Y.S = P.S;
        Y.L = L;
        Y.nu = nu;
        Y.n0 = n0;
        Y.M = M;
        const long long span = dfk::kApplyTile + L - 1;
        Y.chunk = static_cast<int>(std::max(1ll, std::min(static_cast<long long>(Cx), dfk::kApplyStageDoubles / span)));
        Y.h = rhs_dev;
        Y.flag = flag_dev;
        Y.res = res_dev;
        Y.ld_res = ld_res;
        Y.vpart = var_res_host ? vpart_dev : nullptr;
        Y.tiles = apply_tiles;
        const size_t apply_smem = sizeof(double) * static_cast<size_t>(dfk::kApplyTargets * nu + Y.chunk * span);
        DFK_CUDA(cudaFuncSetAttribute(dfk::wiener_apply_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      static_cast<int>(apply_smem)));
        const dim3 grid(static_cast<unsigned>(apply_tiles),
                        static_cast<unsigned>((Cy + dfk::kApplyTargets - 1) / dfk::kApplyTargets));
        dfk::wiener_apply_kernel<<<grid, dfk::kApplyThreads, apply_smem, st>>>(Y);
        DFK_CUDA(cudaGetLastError());
        ++launches;
        if (var_res_host) {
            dfk::wiener_var_kernel<<<static_cast<unsigned>((Cy + 127) / 128), 128, 0, st>>>(vpart_dev, apply_tiles, Cy,
                                                                                           M, var_res_dev);
            DFK_CUDA(cudaGetLastError());
            ++launches;
        }
    }
    ctx->launches += launches;
    if (h_host) DFK_CUDA(cudaMemcpyAsync(h_host, rhs_dev, sizeof(double) * Cy * nu, cudaMemcpyDeviceToHost, st));
    if (var_y_host) DFK_CUDA(cudaMemcpyAsync(var_y_host, var_y_dev, sizeof(double) * Cy, cudaMemcpyDeviceToHost, st));
    if (var_res_host)
        DFK_CUDA(cudaMemcpyAsync(var_res_host, var_res_dev, sizeof(double) * Cy, cudaMemcpyDeviceToHost, st));
    int32_t flag = 0;
    DFK_CUDA(cudaMemcpyAsync(&flag, flag_dev, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    DFK_CUDA(cudaStreamSynchronize(st));
    if (singular_out) *singular_out = flag;
    return DFK_OK;
}

int dfk_stability_dev(dfk_ctx* ctx, const double* v_dev, int64_t N, int64_t stride, int64_t C, int64_t ld_c, double fs,
                      int32_t data_type, int32_t kinds, const int64_t* m_host, int32_t n_m, double* dev_host,
                      int64_t* n_host) {
    DFK_ENTER(ctx);
    if (!v_dev || !m_host || !dev_host || !n_host) return fail(DFK_ERR_ARG, "null pointer");
    if (C < 1 || stride < 1) return fail(DFK_ERR_ARG, "bad geometry: C=%lld stride=%lld", (long long)C, (long long)stride);
    if (!(fs > 0.0) || !std::isfinite(fs)) return fail(DFK_ERR_ARG, "fs must be positive and finite");
    if (data_type != DFK_STAB_PHASE && data_type != DFK_STAB_FREQ)
        return fail(DFK_ERR_ARG, "unknown data_type %d (0 phase, 1 freq)", data_type);
    if (kinds == 0 || (kinds & ~DFK_STAB_ALL)) return fail(DFK_ERR_ARG, "kinds 0x%x: a non-empty subset of 0xf", kinds);
    const bool freq = data_type == DFK_STAB_FREQ;
    if (N < 1 || N > (int64_t(1) << 40)) return fail(DFK_ERR_ARG, "bad length N=%lld", (long long)N);
    const long long Nx = freq ? N + 1 : N;
    if (Nx < 3) return fail(DFK_ERR_ARG, "%lld phase points: at least 3 are needed", Nx);
    if (n_m < 1) return fail(DFK_ERR_ARG, "no averaging factors");
    for (int32_t t = 0; t < n_m; ++t)
        if (m_host[t] < 1) return fail(DFK_ERR_ARG, "averaging factor m[%d] = %lld below 1", t, (long long)m_host[t]);
    const bool want_a = kinds & DFK_STAB_OADEV, want_m = kinds & (DFK_STAB_MDEV | DFK_STAB_TDEV),
               want_h = kinds & DFK_STAB_OHDEV;

    // the slice table: every m gets ceil(n / 4096) slices of its largest requested term count n (none when m is
    // outside every requested kind's range); an m above Nx is clamped there, where every count is already <= 0
    std::vector<dfk::StabSlice> slices;
    std::vector<dfk::StabTau> taus(n_m);
    const int slot_bits[4] = {DFK_STAB_OADEV, DFK_STAB_MDEV, DFK_STAB_TDEV, DFK_STAB_OHDEV};
    for (int32_t t = 0; t < n_m; ++t) {
        const long long m = std::min<long long>(m_host[t], Nx);
        const long long na = dfk::stab_n_oadev(Nx, m), nm = dfk::stab_n_mdev(Nx, m), nh = dfk::stab_n_ohdev(Nx, m);
        long long nmax = 0;
        if (want_a) nmax = std::max(nmax, na);
        if (want_m) nmax = std::max(nmax, nm);
        if (want_h) nmax = std::max(nmax, nh);
        const long long ns = (nmax + dfk::kStabSlice - 1) / dfk::kStabSlice;
        taus[t] = {m, static_cast<long long>(slices.size()), ns};
        for (long long s = 0; s < ns; ++s) slices.push_back({m, s * dfk::kStabSlice});
        if (slices.size() > (size_t(1) << 31)) return fail(DFK_ERR_ARG, "stability problem too large for one launch");
        const long long n_slot[4] = {na, nm, nm, nh};
        for (int k = 0; k < 4; ++k)
            if (kinds & slot_bits[k]) n_host[k * n_m + t] = std::max(0ll, n_slot[k]);
    }
    const long long nslices = static_cast<long long>(slices.size());
    const long long ld = Nx + 1;
    const long long in_len = freq ? N : Nx;  // samples the X pass reads
    const long long tiles_x = (in_len + dfk::kStabTile - 1) / dfk::kStabTile;
    const long long tiles_s = (Nx + dfk::kStabTile - 1) / dfk::kStabTile;
    if (nslices * C > 0x7fffffffll || tiles_s * C > 0x7fffffffll)
        return fail(DFK_ERR_ARG, "stability problem too large for one launch");

    // post[0]: X [C][Nx + 1] double-double; post[1]: S, the same, when mdev or tdev is requested; post[2]: tile sums
    // [C][tiles], slices, taus, partials [C][nslices][3], outputs [4][C][n_m], flags [C]
    const auto align = [](size_t b) { return (b + 255) & ~static_cast<size_t>(255); };
    const size_t rows_b = static_cast<size_t>(C) * static_cast<size_t>(ld) * sizeof(double2);
    const size_t tsum_b = align(sizeof(double2) * static_cast<size_t>(C) * static_cast<size_t>(std::max(tiles_x, tiles_s)));
    const size_t slice_b = align(sizeof(dfk::StabSlice) * std::max<size_t>(1, slices.size()));
    const size_t tau_b = align(sizeof(dfk::StabTau) * static_cast<size_t>(n_m));
    const size_t part_b = align(sizeof(double) * dfk::kStabSums * static_cast<size_t>(std::max(1ll, nslices * C)));
    const size_t out_b = align(sizeof(double) * 4 * static_cast<size_t>(C) * static_cast<size_t>(n_m));
    const size_t small_b = tsum_b + slice_b + tau_b + part_b + out_b + sizeof(int) * static_cast<size_t>(C);
    DevBuf& x_buf = ctx->post[0];
    DevBuf& s_buf = ctx->post[1];
    DevBuf& small_buf = ctx->post[2];
    {
        const size_t want = rows_b * (want_m ? 2 : 1) + small_b;
        const size_t held = x_buf.bytes + (want_m ? s_buf.bytes : 0) + small_buf.bytes;
        size_t free_b = 0, total_b = 0;
        DFK_CUDA(cudaMemGetInfo(&free_b, &total_b));
        if (want > free_b + held)
            return fail(DFK_ERR_NOMEM, "stability scratch of %zu bytes (running sums of %lld x %lld points in "
                        "double-double) does not fit the device's %zu free bytes", want, (long long)C, ld, free_b + held);
    }
    int rc = ensure(ctx, x_buf, rows_b);
    if (!rc && want_m) rc = ensure(ctx, s_buf, rows_b);
    if (!rc) rc = ensure(ctx, small_buf, small_b);
    if (rc) return rc;
    char* small = static_cast<char*>(small_buf.ptr);
    double2* tsum_dev = reinterpret_cast<double2*>(small);
    auto* slice_dev = reinterpret_cast<dfk::StabSlice*>(small + tsum_b);
    auto* tau_dev = reinterpret_cast<dfk::StabTau*>(small + tsum_b + slice_b);
    double* part_dev = reinterpret_cast<double*>(small + tsum_b + slice_b + tau_b);
    double* out_dev = reinterpret_cast<double*>(small + tsum_b + slice_b + tau_b + part_b);
    int* bad_dev = reinterpret_cast<int*>(small + tsum_b + slice_b + tau_b + part_b + out_b);
    double2* X = static_cast<double2*>(x_buf.ptr);
    double2* S = want_m ? static_cast<double2*>(s_buf.ptr) : nullptr;
    cudaStream_t st = ctx->stream();
    if (nslices)
        DFK_CUDA(cudaMemcpyAsync(slice_dev, slices.data(), sizeof(dfk::StabSlice) * nslices, cudaMemcpyHostToDevice, st));
    DFK_CUDA(cudaMemcpyAsync(tau_dev, taus.data(), sizeof(dfk::StabTau) * n_m, cudaMemcpyHostToDevice, st));
    DFK_CUDA(cudaMemsetAsync(bad_dev, 0, sizeof(int) * C, st));
    long long launches = 0;

    // running sums as exclusive scans: out[0] = 0, out[k] = sum_{i<k} in_i (tile sums, carries, write)
    auto scan = [&](dfk::StabScanParams P, bool dd) -> int {
        const unsigned grid = static_cast<unsigned>(P.ntiles * C);
        if (dd)
            dfk::stab_scan_kernel<true, false><<<grid, dfk::kStabScanThreads, 0, st>>>(P);
        else
            dfk::stab_scan_kernel<false, false><<<grid, dfk::kStabScanThreads, 0, st>>>(P);
        DFK_CUDA(cudaGetLastError());
        dfk::stab_carry_kernel<<<static_cast<unsigned>((C + 3) / 4), 128, 0, st>>>(P.tsum, P.ntiles, C);
        DFK_CUDA(cudaGetLastError());
        if (dd)
            dfk::stab_scan_kernel<true, true><<<grid, dfk::kStabScanThreads, 0, st>>>(P);
        else
            dfk::stab_scan_kernel<false, true><<<grid, dfk::kStabScanThreads, 0, st>>>(P);
        DFK_CUDA(cudaGetLastError());
        launches += 3;
        return DFK_OK;
    };
    dfk::StabScanParams P;
    P.v = v_dev;
    P.X = nullptr;
    P.ld_c = ld_c;
    P.stride = stride;
    P.L = in_len;
    P.ntiles = tiles_x;
    P.tsum = tsum_dev;
    P.out = X;
    P.ld_out = ld;
    P.bad = bad_dev;
    if (freq) {
        rc = scan(P, false);
        if (rc) return rc;
    } else {
        dfk::stab_load_kernel<<<static_cast<unsigned>(tiles_x * C), dfk::kStabScanThreads, 0, st>>>(P);
        DFK_CUDA(cudaGetLastError());
        ++launches;
    }
    if (want_m) {
        dfk::StabScanParams Q = P;
        Q.v = nullptr;
        Q.X = X;
        Q.ld_c = ld;
        Q.stride = 1;
        Q.L = Nx;
        Q.ntiles = tiles_s;
        Q.out = S;
        rc = scan(Q, true);
        if (rc) return rc;
    }
    dfk::StabTermsParams T;
    T.X = X;
    T.S = S;
    T.ld = ld;
    T.Nx = Nx;
    T.slices = slice_dev;
    T.nslices = nslices;
    T.want_a = want_a;
    T.want_m = want_m;
    T.want_h = want_h;
    T.part = part_dev;
    dfk::stab_terms_kernel<<<static_cast<unsigned>(std::max(1ll, nslices * C)), dfk::kStabTermThreads, 0, st>>>(T);
    DFK_CUDA(cudaGetLastError());
    const long long nout = C * n_m;
    dfk::stab_finish_kernel<<<static_cast<unsigned>((nout + dfk::kStabFinishThreads - 1) / dfk::kStabFinishThreads),
                              dfk::kStabFinishThreads, 0, st>>>(tau_dev, n_m, C, part_dev, nslices, bad_dev, Nx, fs,
                                                                freq ? 1.0 : fs, out_dev);
    DFK_CUDA(cudaGetLastError());
    launches += 2;
    ctx->launches += launches;
    for (int k = 0; k < 4; ++k)
        if (kinds & slot_bits[k])
            DFK_CUDA(cudaMemcpyAsync(dev_host + k * nout, out_dev + k * nout, sizeof(double) * nout,
                                     cudaMemcpyDeviceToHost, st));
    DFK_CUDA(cudaStreamSynchronize(st));
    return DFK_OK;
}

int dfk_downsample_dev(dfk_ctx* ctx, const double* x_dev, int64_t n, int64_t R, double* out_dev) {
    DFK_ENTER(ctx);
    if (R <= 0 || n < 0) return fail(DFK_ERR_ARG, "bad geometry: n=%lld R=%lld", (long long)n, (long long)R);
    const int64_t nblk = n / R;  // the tail that does not fill a block is dropped (dsp.py:43)
    if (nblk == 0) return DFK_OK;
    if (!x_dev || !out_dev) return fail(DFK_ERR_ARG, "null pointer");
    const int64_t per_cta = R >= dfk::kDsCtaMin ? 1 : dfk::kDsThreads / 32;
    const int64_t want = (nblk + per_cta - 1) / per_cta;
    const int grid = static_cast<int>(std::min<int64_t>(want, static_cast<int64_t>(ctx->sm_count) * 8));
    dfk::downsample_kernel<<<grid, dfk::kDsThreads, 0, ctx->stream()>>>(x_dev, nblk, R, out_dev);
    ctx->launches++;
    DFK_CUDA(cudaGetLastError());
    return DFK_OK;
}

int dfk_downsample_host(dfk_ctx* ctx, const double* x_host, int64_t n, int64_t R, double* out_host) {
    DFK_ENTER(ctx);
    if (R <= 0 || n < 0) return fail(DFK_ERR_ARG, "bad geometry: n=%lld R=%lld", (long long)n, (long long)R);
    const int64_t nblk = n / R;
    if (nblk == 0) return DFK_OK;
    if (!x_host || !out_host) return fail(DFK_ERR_ARG, "null pointer");
    HostCallGuard hg(ctx);
    // slabs of whole blocks, double-buffered: the copy of slab i+1 overlaps the reduction of slab i
    const size_t slab_bytes = ctx->host_slab_bytes ? ctx->host_slab_bytes : (static_cast<size_t>(128) << 20);
    int64_t per_slab = std::max<int64_t>(1, static_cast<int64_t>(slab_bytes / (sizeof(double) * R)));
    per_slab = std::min(per_slab, nblk);
    int rc = ensure(ctx, ctx->rows, sizeof(double) * nblk);
    for (int i = 0; i < 2 && !rc; ++i) rc = ensure(ctx, ctx->slab[i], sizeof(double) * per_slab * R);
    if (rc) return rc;
    const bool pageable = is_pageable(x_host);
    cudaStream_t st = ctx->stream();
    double* out_dev = static_cast<double*>(ctx->rows.ptr);
    int64_t done = 0;
    for (int i = 0; done < nblk; ++i, done += per_slab) {
        const int s = i & 1;
        const int64_t nb = std::min(per_slab, nblk - done);
        if (i >= 2) DFK_CUDA(cudaStreamWaitEvent(ctx->copy_stream, ctx->consumed[s], 0));
        rc = copy_slab_to_device(ctx, ctx->slab[s].ptr, x_host + done * R, sizeof(double) * nb * R, pageable);
        if (rc) return rc;
        DFK_CUDA(cudaEventRecord(ctx->copied[s], ctx->copy_stream));
        DFK_CUDA(cudaStreamWaitEvent(st, ctx->copied[s], 0));
        rc = dfk_downsample_dev(ctx, static_cast<const double*>(ctx->slab[s].ptr), nb * R, R, out_dev + done);
        if (rc) return rc;
        DFK_CUDA(cudaEventRecord(ctx->consumed[s], st));
    }
    DFK_CUDA(cudaMemcpyAsync(out_host, out_dev, sizeof(double) * nblk, cudaMemcpyDeviceToHost, st));
    DFK_CUDA(cudaStreamSynchronize(st));
    DFK_CUDA(cudaStreamSynchronize(ctx->copy_stream));
    hg.done();
    return DFK_OK;
}

}  // extern "C"
