#!/usr/bin/env python
"""Cost of the EKF fixed-interval smoother, ``dfk_ekf_smooth_dev``, against the filter, ``dfk_ekf_dev`` (development
tool).

Shapes ('snr'-mode records generated on the device, channel-major, default options, R = 4000):

  - 4096 channels x 2 s at 200 kHz (3.3e9 samples, 13 GB resident);
  - 8 channels x 20 s;
  - 1 channel x 20 s.

At each shape the filter and the smoother at checkpoint intervals B in {64, 256, 1024, 4096} and the library's
default (block = 0) are timed with CUDA events around each call (statistics, forward and backward launches included),
after a warm-up call of every arm, the arms alternated over the repetitions.  Reported per arm: median / min / max ms,
samples per second, the smoother / filter ratio of medians and the scratch bytes C (ceil(T / B) + B) 20 x 8.  The
smoothed rows of every B are checked to be bit-identical.

One JSON line per measurement, with the card's name and power limit read in the same run, to stdout and to --out
(default profiles/r03_ekf_smooth_cost.jsonl).
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

F_SAMP, F_MOD, R = 200e3, 1000.0, 4000
SHAPES = {"4096x2s": (4096, 400_000), "8x20s": (8, 4_000_000), "1x20s": (1, 4_000_000)}
BLOCKS = (64, 256, 1024, 4096, 0)


def card():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in q.split(",")]
    except Exception as e:  # the numbers are still recorded; the line says what is missing
        info["power_limit"] = f"unavailable ({type(e).__name__})"
    return info


def scratch_bytes(C, T, B):
    t_round = -(-T // 32) * 32
    B = min(B or 256, t_round)  # kSmoothBlockDefault
    return C * (-(-T // B) + B) * 20 * 8


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--shapes", default=",".join(SHAPES))
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_ekf_smooth_cost.jsonl"))
    args = ap.parse_args()
    info = card()
    ctx = _lib.get_context(0)
    lines = []

    def emit(d):
        d.update(info)
        lines.append(d)
        print(json.dumps(d), flush=True)

    for name in args.shapes.split(","):
        C, T = SHAPES[name]
        z = torch.empty((C, T), dtype=torch.float64, device="cuda")
        ctx.synth_snr_dev(z.data_ptr(), T, C, F_SAMP, F_MOD, 6.0, dphi=0.37, snr_db=40.0, seed=7)
        nbuf = T // R
        rows = {B: torch.empty((C, nbuf, 8), dtype=torch.float64, device="cuda") for B in BLOCKS}
        var = torch.empty((C, nbuf, 5), dtype=torch.float64, device="cuda")
        frows = torch.empty((C, nbuf, 8), dtype=torch.float64, device="cuda")
        arms = {"filter": lambda: ctx.ekf_dev(z.data_ptr(), T, C, 1, T, R, F_SAMP, F_MOD, None, frows.data_ptr())}
        for B in BLOCKS:
            arms[f"smooth_B{B}"] = (lambda B=B: ctx.ekf_smooth_dev(z.data_ptr(), T, C, 1, T, R, F_SAMP, F_MOD, None, 0,
                                                                   None, B, rows[B].data_ptr(), var.data_ptr()))
        ctx.use_torch_stream()
        times = {k: [] for k in arms}
        for fn in arms.values():
            fn()
        torch.cuda.synchronize()
        for _ in range(args.reps):
            for k, fn in arms.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn()
                e1.record()
                e1.synchronize()
                times[k].append(e0.elapsed_time(e1))
        ctx.use_default_stream()
        same = all(torch.equal(rows[B], rows[BLOCKS[0]]) for B in BLOCKS)
        f_med = float(np.median(times["filter"]))
        for k, ms in times.items():
            ms = np.asarray(ms)
            med = float(np.median(ms))
            d = {"shape": name, "channels": C, "samples": T, "arm": k, "median_ms": med, "min_ms": float(ms.min()),
                 "max_ms": float(ms.max()), "reps": len(ms), "samples_per_s": C * T / (med / 1e3)}
            if k != "filter":
                B = int(k.split("B")[1])
                d.update(block=B, ratio_to_filter=med / f_med, scratch_bytes=scratch_bytes(C, T, B),
                         rows_bit_identical_over_B=same)
            emit(d)
        del z, rows, var, frows
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("".join(json.dumps(d) + "\n" for d in lines))


if __name__ == "__main__":
    main()
