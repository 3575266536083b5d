#!/usr/bin/env python
"""Per-config device timings of the three kernels (development tool; bench.py is the contract benchmark).

    python benchmarks/run_configs.py [cfg1 cfg2 cfg3 cfg4 cfg5 ...] [--reps 5]

Geometries follow BASELINE.json's configs; records that do not fit one GPU are cut to a resident wave
(stated in the output).  Everything is generated on the device; times are CUDA events on the launching
stream, best-of-reps after one warm-up.  One JSON line per config.  (The CPU baseline beside each config is
`python bench.py --impl reference --workload cfgN`: only bench.py's CPU leg may run the oracle.)
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from deepfmkit_b200 import _lib  # noqa: E402
from deepfmkit_b200 import fit as tun  # noqa: E402

PEAK = 6550.7
try:
    PEAK = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
except Exception:
    pass


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    best = 1e30
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        best = min(best, a.elapsed_time(b))
    return best


def nls_case(ctx, name, f_samp, n, ndata, channels, seconds, reps, m=6.0, init_m=None, seeded=True, note=""):
    f_mod = 1000.0
    R = int(f_samp / f_mod * n)
    T = int(seconds * f_samp) // R * R
    bpc = T // R
    nbuf = channels * bpc
    w0 = 2.0 * np.pi * f_mod / f_samp
    x = torch.empty(channels * T, dtype=torch.float64, device="cuda")
    if np.ndim(m) == 0:
        ctx.synth_snr_dev(x.data_ptr(), T, channels, f_samp, f_mod, float(m), dphi=2 * np.pi / max(channels, 1), seed=1)
    else:  # blocks of channels with their own m (cfg 5)
        per = channels // len(m)
        for i, mi in enumerate(m):
            ctx.synth_snr_dev(x.data_ptr() + i * per * T * 8, T, per, f_samp, f_mod, float(mi), seed=1 + i * per)
    qi = torch.empty((nbuf, 2 * ndata), dtype=torch.float64, device="cuda")
    dc = torch.empty(nbuf, dtype=torch.float64, device="cuda")
    rows = torch.empty((nbuf, 8), dtype=torch.float64, device="cuda")
    opts = tun.current_lm_opts()
    init_dev = None
    if init_m is not None:
        g = np.zeros((channels, 4))
        g[:, 0], g[:, 1] = 1.6, init_m
        init_dev = torch.from_numpy(g).cuda()
    t_demod = timed(lambda: ctx.demod(x.data_ptr(), nbuf, R, ndata, w0, qi.data_ptr(), dc.data_ptr()), reps)
    ctx.lm_counters(reset=True)

    def whole():
        ctx.nls_fit_batch_dev(x.data_ptr(), channels, bpc, T, R, ndata, w0, [1.6, 6.0, 0.0, 0.0],
                              init_dev.data_ptr() if init_dev is not None else None, 4 if init_dev is not None else 0,
                              seeded, opts, rows.data_ptr())
    t_all = timed(whole, reps)
    cnt = ctx.lm_counters(reset=True)
    ctx.profile_enable(True)
    ctx.profile_read(reset=True)
    whole()
    prof = ctx.profile_read(reset=True)
    ctx.profile_enable(False)
    r = rows.cpu().numpy()
    alg = (8 * R + 8 * (2 * ndata + 1)) * nbuf
    fits = nbuf * (reps + 1)
    out = {"config": name, "note": note, "f_samp": f_samp, "R": R, "ndata": ndata, "channels": channels, "buffers": nbuf,
           "bytes": nbuf * R * 8, "demod_ms": t_demod, "demod_GBps": alg / t_demod / 1e6, "demod_frac_of_hbm_peak": alg / t_demod / 1e6 / PEAK,
           "nls_ms": t_all, "lm_ms": t_all - t_demod, "buffers_per_s": nbuf / t_all * 1e3, "samples_per_s": nbuf * R / t_all * 1e3,
           "lm_fits_per_s": nbuf / max(t_all - t_demod, 1e-9) * 1e3,
           "fitok_counts": {str(int(k)): int(v) for k, v in zip(*np.unique(r[:, 6], return_counts=True))},
           "prof": {k: round(v, 4) for k, v in prof.items()}, "m_mean": float(r[:, 1].mean()), "per_fit": {k: v / fits for k, v in cnt.items()}}
    print(json.dumps(out), flush=True)
    del x, qi, dc, rows


def ekf_case(ctx, name, channels, seconds, reps, time_major, note="", start_s=0.0):
    f_samp, f_mod, n = 200e3, 1000.0, 20
    R = int(f_samp / f_mod * n)
    T = int(seconds * f_samp)
    k0 = int(start_s * f_samp) // R * R
    x = torch.empty(channels * T, dtype=torch.float64, device="cuda")
    ctx.synth_snr_slab_dev(x.data_ptr(), T, channels, T, k0, f_samp, f_mod, 6.0, dphi=2 * np.pi / channels, seed=3)
    z = x.view(channels, T)
    ld_t, ld_c = 1, T
    if time_major:
        z = z.t().contiguous()
        ld_t, ld_c = channels, 1
    rows = torch.empty((channels, T // R, 8), dtype=torch.float64, device="cuda")
    opts = _lib.default_ekf_opts()
    state = torch.zeros((channels, 32), dtype=torch.float64, device="cuda")
    if k0 > 0:  # a slab late in the record: start from a converged-looking state
        state[:, 0], state[:, 1], state[:, 4], state[:, 30] = 1.0, 6.0, 1.15, 1e-4
        state[:, 2] = torch.arange(channels, device="cuda") * (2 * np.pi / channels)
        for idx in (0, 5, 9, 12, 14):  # diagonal of the packed upper triangle
            state[:, 5 + idx] = 1e-6
    keep = state.clone()

    def run():
        state.copy_(keep)
        ctx.ekf_stream_dev(z.data_ptr(), T, channels, ld_t, ld_c, R, f_samp, f_mod, opts, k0, state.data_ptr(), rows.data_ptr())
    t = timed(run, reps)
    r = rows.cpu().numpy()
    out = {"config": name, "note": note, "start_s": start_s, "channels": channels, "samples_per_channel": T, "layout": "time-major" if time_major else "channel-major",
           "ekf_ms": t, "samples_per_s": channels * T / t * 1e3, "steps_per_s_per_channel": T / t * 1e3,
           "read_GBps": channels * T * 8 / t / 1e6, "m_last_mean": float(r[:, -1, 1].mean()), "m_last_std": float(r[:, -1, 1].std())}
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("configs", nargs="*", default=["cfg1", "cfg2", "cfg3", "cfg4", "cfg5"])
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    ctx = _lib.Context(0)
    ctx.use_torch_stream()
    for c in args.configs:
        if c == "cfg1":
            nls_case(ctx, "cfg1", 200e3, 20, 10, 1, 10.0, args.reps, note="README quickstart: 500 buffers")
        elif c == "cfg2":
            nls_case(ctx, "cfg2", 1e6, 20, 10, 1, 3600.0, args.reps, note="full size, 28.8 GB")
        elif c == "cfg3":
            nls_case(ctx, "cfg3", 200e3, 20, 10, 256, 100.0, args.reps,
                     note="resident wave: 256 channels x 100 s (41 GB) of the 1000 s config")
        elif c == "cfg5":
            ms = list(range(2, 21))
            per = 1_000_000
            init_m = np.repeat(np.array(ms, dtype=float), per)
            nls_case(ctx, "cfg5", 200e3, 1, 15, len(ms) * per, 1e-3, args.reps, m=ms, init_m=init_m, seeded=False,
                     note="full size: 1e6 realisations x 19 m values, one period each, init_m = m_true")
        elif c == "cfg5small":
            ms = list(range(2, 21))
            per = 50_000
            init_m = np.repeat(np.array(ms, dtype=float), per)
            nls_case(ctx, "cfg5small", 200e3, 1, 15, len(ms) * per, 1e-3, args.reps, m=ms, init_m=init_m, seeded=False,
                     note="5e4 realisations x 19 m values")
        elif c == "cfg4":
            ekf_case(ctx, "cfg4", 4096, 1.0, max(1, args.reps // 2), False, note="4096 channels x 1 s of the 100 s config")
            ekf_case(ctx, "cfg4", 4096, 1.0, max(1, args.reps // 2), True, note="4096 channels x 1 s of the 100 s config")
        elif c == "cfg4late":
            ekf_case(ctx, "cfg4late", 4096, 0.25, 1, False, note="slab starting at t = 90 s", start_s=90.0)
            ekf_case(ctx, "cfg4late", 4096, 0.25, 1, False, note="slab starting at t = 0 s", start_s=0.0)
        elif c == "cfg4cpw":  # channels per warp: does a one-warp block get a scheduler of its own?
            for cpw in (4, 8, 16, 32):
                _lib.load_library().dfk_dev_set(b"DFK_EKF_CPW", cpw)
                ekf_case(ctx, f"cfg4 cpw={cpw}", 4096, 0.25, 2, False)
            _lib.load_library().dfk_dev_clear()
        elif c == "cfg4small":
            ekf_case(ctx, "cfg4small", 4096, 0.1, 1, False)
            ekf_case(ctx, "cfg4small", 4096, 0.1, 1, True)
    ctx.close()


if __name__ == "__main__":
    main()
