#!/usr/bin/env python
"""Timings of the cfg-5 pipeline pieces (development tool): generator shapes, single-period demod, the cold LM kernel."""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from deepfmkit_b200 import _lib  # noqa: E402


def timed(fn, reps=5):
    fn(); torch.cuda.synchronize()
    best = 1e30
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); b.synchronize()
        best = min(best, a.elapsed_time(b))
    return best


def main():
    ctx = _lib.Context(0)
    ctx.use_torch_stream()
    what = sys.argv[1:] or ["synth", "lm"]
    if "synth" in what:
        x = torch.empty(1_600_000_000, dtype=torch.float64, device="cuda")
        for T, C in ((1_600_000_000, 1), (200, 400_000), (200, 4_000_000), (2000, 400_000), (20000, 40_000), (200_000, 4000),
                     (200, 8_000_000)):
            t = timed(lambda: ctx.synth_snr_dev(x.data_ptr(), T, C, 200e3 if T < 1e9 else 1e6, 1000.0, 6.0, seed=1), 3)
            print(json.dumps({"what": f"synth T={T} C={C}", "ms": t, "GBps": T * C * 8 / t / 1e6}), flush=True)
        del x
    if "lm" in what:
        ms = list(range(2, 21)); per = 400_000; C = per * len(ms); R = 200; nd = 15
        x = torch.empty(C * R, dtype=torch.float64, device="cuda")
        for i, m in enumerate(ms):
            ctx.synth_snr_dev(x.data_ptr() + i * per * R * 8, R, per, 200e3, 1000.0, float(m), seed=1000 * i)
        w0 = 2 * np.pi * 1000 / 200e3
        qi = torch.empty((C, 2 * nd), dtype=torch.float64, device="cuda"); dc = torch.empty(C, dtype=torch.float64, device="cuda")
        t = timed(lambda: ctx.demod(x.data_ptr(), C, R, nd, w0, qi.data_ptr(), dc.data_ptr()))
        alg = (8 * R + 8 * (2 * nd + 1)) * C
        print(json.dumps({"what": "demod_period", "ms": t, "GBps": alg / t / 1e6, "buffers": C}), flush=True)
        g = np.zeros((C, 4)); g[:, 0] = 1.6; g[:, 1] = np.repeat(np.array(ms, dtype=float), per)
        guess = torch.from_numpy(g).cuda()
        rows = torch.zeros((C, 8), dtype=torch.float64, device="cuda")
        opts = _lib.default_lm_opts()
        t = timed(lambda: ctx.lm_fit(qi.data_ptr(), C, nd, guess.data_ptr(), 4, dc.data_ptr(), opts, rows.data_ptr()))
        print(json.dumps({"what": "lm_flat", "ms": t, "Mfits_per_s": C / t / 1e3}), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
