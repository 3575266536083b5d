#!/usr/bin/env python
"""Cost of the per-buffer parameter covariance (development tool).

  1. cfg 2, one resident device-generated record (180 000 buffers, 28.8 GB): dfk_nls_fit_dev against
     dfk_nls_fit_cov_dev, alternated in one process, CUDA events around each call.
  2. lm_cov_kernel alone (dfk_lm_cov) on the harmonic vectors and rows of the same record, with the bytes it must move,
     nfit * (16 N + 128): the harmonic vector, the result row and the covariance row.
  3. cfg 5 at full size (m = 2..20 x 1e6 trials, 1.9e7 fits): dfk_nls_sweep_dev against dfk_nls_sweep_cov_dev.

One JSON line per measurement, with the card's name and power limit, to stdout and to --out
(default profiles/r03_cov_cost.jsonl).
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from deepfmkit_b200 import _lib  # noqa: E402


def card():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in q.split(",")]
    except Exception as e:  # the numbers are still recorded; the line says what is missing
        info["power_limit"] = f"unavailable ({type(e).__name__})"
    return info


def timed(fn, stream):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    fn()
    e1.record(stream)
    e1.synchronize()
    return e0.elapsed_time(e1)


def summary(ms):
    ms = np.asarray(ms)
    return {"median_ms": float(np.median(ms)), "min_ms": float(ms.min()), "max_ms": float(ms.max()),
            "p10_ms": float(np.percentile(ms, 10)), "p90_ms": float(np.percentile(ms, 90)), "reps": len(ms)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--sweep-trials", type=float, default=1e6)
    ap.add_argument("--sweep-reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_cov_cost.jsonl"))
    args = ap.parse_args()
    info = card()
    lines = []

    def emit(d):
        d = {**d, **info}
        print(json.dumps(d), flush=True)
        lines.append(d)

    ctx = _lib.Context(0, own_stream=True)
    stream = torch.cuda.Stream()
    ctx.use_torch_stream(stream)
    with torch.cuda.stream(stream):
        # ---- cfg 2 -------------------------------------------------------------------------------------------
        f_samp, f_mod, n, N = 1e6, 1000.0, 20, 10
        R = int(f_samp / f_mod * n)
        nbuf = int(3600 * f_samp) // R
        w0 = 2 * np.pi * f_mod / f_samp
        sched = max(1, os.cpu_count() or 1)
        init = [1.6, 6.0, 0.0, 0.0]
        x = torch.empty(nbuf * R, dtype=torch.float64, device="cuda")
        rows = torch.empty((nbuf, 8), dtype=torch.float64, device="cuda")
        rows_c = torch.empty_like(rows)
        cov = torch.empty_like(rows)
        ctx.synth_snr_dev(x.data_ptr(), nbuf * R, 1, f_samp, f_mod, 6.0, snr_db=40.0, seed=1000)

        def plain():
            ctx.nls_fit_dev(x.data_ptr(), nbuf, R, N, w0, init, sched, None, rows.data_ptr())

        def with_cov():
            ctx.nls_fit_dev(x.data_ptr(), nbuf, R, N, w0, init, sched, None, rows_c.data_ptr(), cov_ptr=cov.data_ptr())

        for _ in range(3):
            plain()
            with_cov()
        t_plain, t_cov = [], []
        for _ in range(args.reps):
            t_plain.append(timed(plain, stream))
            t_cov.append(timed(with_cov, stream))
        same = bool(torch.equal(rows, rows_c))
        a, b = summary(t_plain), summary(t_cov)
        emit({"what": "cfg2_readout", "buffers": nbuf, "plain": a, "cov": b, "rows_identical": same,
              "overhead_median_pct": 100.0 * (b["median_ms"] / a["median_ms"] - 1.0)})

        # ---- the kernel alone on the same record -------------------------------------------------------------
        qi = torch.empty((nbuf, 2 * N), dtype=torch.float64, device="cuda")
        dc = torch.empty(nbuf, dtype=torch.float64, device="cuda")
        ctx.demod(x.data_ptr(), nbuf, R, N, w0, qi.data_ptr(), dc.data_ptr())
        cov2 = torch.empty_like(cov)
        del x
        torch.cuda.empty_cache()

        def kernel():
            ctx.lm_cov(qi.data_ptr(), nbuf, N, rows_c.data_ptr(), cov2.data_ptr())

        for _ in range(3):
            kernel()
        t_k = [timed(kernel, stream) for _ in range(args.reps)]
        k = summary(t_k)
        nbytes = nbuf * (16 * N + 128)
        emit({"what": "lm_cov_kernel_cfg2", "fits": nbuf, "N": N, "kernel": k, "bytes": nbytes,
              "gb_per_s_median": nbytes / (k["median_ms"] * 1e-3) / 1e9,
              "cov_equals_record_entry": bool(torch.equal(cov, cov2)),
              "note": "qi, rows and cov (33 MB) fit in L2: after the first pass the kernel reads them from there"})
        del qi, dc, rows, rows_c, cov, cov2
        torch.cuda.empty_cache()

        # ---- cfg 5 at full size --------------------------------------------------------------------------------
        ms = np.arange(2.0, 21.0)
        nt = int(args.sweep_trials)
        Rs, Ns = 200, 15
        srows = torch.empty((len(ms), nt, 8), dtype=torch.float64, device="cuda")
        srows_c = torch.empty_like(srows)
        scov = torch.empty_like(srows)

        def sweep():
            ctx.nls_sweep_dev(ms, nt, 0, nt, Rs, Ns, 200e3, 1000.0, srows.data_ptr(), snr_db=40.0, seed=0)

        def sweep_cov():
            ctx.nls_sweep_dev(ms, nt, 0, nt, Rs, Ns, 200e3, 1000.0, srows_c.data_ptr(), snr_db=40.0, seed=0,
                              cov_ptr=scov.data_ptr())

        sweep()
        sweep_cov()
        s_plain, s_cov = [], []
        for _ in range(args.sweep_reps):
            s_plain.append(timed(sweep, stream))
            s_cov.append(timed(sweep_cov, stream))
        a, b = summary(s_plain), summary(s_cov)
        emit({"what": "cfg5_sweep", "fits": len(ms) * nt, "plain": a, "cov": b, "rows_identical": bool(torch.equal(srows, srows_c)),
              "overhead_median_pct": 100.0 * (b["median_ms"] / a["median_ms"] - 1.0),
              "cov_bytes": len(ms) * nt * (16 * Ns + 128)})
    ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for d in lines:
            f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
