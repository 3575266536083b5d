// Post-fit entries of the C ABI (include/dfk_b200.h, "post-fit step"): block means and log-frequency spectra.
#include "dfk_host.h"

#include <cmath>
#include <vector>

#include "dfk_spectra.cuh"

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
