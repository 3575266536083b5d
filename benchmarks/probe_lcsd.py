#!/usr/bin/env python
"""Cost of the log-frequency cross-spectral estimate (development tool).

At N = 180 000 points (the cfg-2 phase series at 50 Hz) and at N = 1.8e6, on seeded random-walk series resident on the
device:

  1. call time, alternated repetitions after a warm-up of every arm: ``lpsd`` on 1 and 2 series, ``lcsd`` on 1 x 1,
     1 x 8 and 8 x 8 pairs (CUDA events around each public call, which includes the plan, the copies back and, for
     ``lcsd``, the host-side coherence and transfer function);
  2. kernel time per call from one ``torch.profiler`` pass per arm, after the timed ones: the per-segment stage
     (``lpsd_segment_kernel`` / ``lcsd_segment_kernel``) and the finish (``lpsd_finish_kernel`` /
     ``lcsd_finish_kernel``).

One JSON line per measurement, with the card's name and power limit, to stdout and to --out
(default profiles/r03_lcsd_cost.jsonl).
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
from deepfmkit_b200 import lcsd, lpsd  # noqa: E402

FS = 50.0


def card():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in q.split(",")]
    except Exception as e:  # the numbers are still recorded; the line says what is missing
        info["power_limit"] = f"unavailable ({type(e).__name__})"
    return info


def summary(ms):
    ms = np.asarray(ms)
    return {"median_ms": float(np.median(ms)), "min_ms": float(ms.min()), "max_ms": float(ms.max()),
            "p10_ms": float(np.percentile(ms, 10)), "p90_ms": float(np.percentile(ms, 90)), "reps": len(ms)}


def arms(x, y):
    return {"lpsd_1": lambda: lpsd(x[:1], FS, return_type="dict"),
            "lpsd_2": lambda: lpsd(x[:2], FS, return_type="dict"),
            "lcsd_1x1": lambda: lcsd(x[:1], y[:1], FS),
            "lcsd_1x8": lambda: lcsd(x[:1], y, FS),
            "lcsd_8x8": lambda: lcsd(x, y, FS)}


def timed(fn):
    s = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(s)
    fn()
    e1.record(s)
    e1.synchronize()
    return e0.elapsed_time(e1)


def kernel_ms(fn):
    """Device time per kernel name of one call."""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.events():
        if ev.device_type == DeviceType.CUDA and ("lpsd_" in ev.name or "lcsd_" in ev.name):
            key = ev.name.split("(")[0].split("::")[-1]
            out[key] = out.get(key, 0.0) + ev.time_range.elapsed_us() / 1e3
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10, help="alternated repetitions at N = 180 000")
    ap.add_argument("--reps-long", type=int, default=5, help="alternated repetitions at N = 1.8e6")
    ap.add_argument("--sizes", default="180000,1800000")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_lcsd_cost.jsonl"))
    args = ap.parse_args()
    info = card()
    lines = []

    def emit(d):
        d = {**d, **info}
        print(json.dumps(d), flush=True)
        lines.append(d)

    for n in (int(s) for s in args.sizes.split(",")):
        rng = np.random.RandomState(n % 9973)
        x = torch.from_numpy(np.cumsum(rng.randn(8, n), axis=1) * 1e-3).cuda()
        y = torch.from_numpy(0.5 * x.cpu().numpy() + np.cumsum(rng.randn(8, n), axis=1) * 1e-3).cuda()
        fns = arms(x, y)
        nf = len(fns["lcsd_1x1"]()["f"])
        for fn in fns.values():  # warm-up: every shape the timed loop uses
            fn()
        torch.cuda.synchronize()
        ms = {k: [] for k in fns}
        for _ in range(args.reps if n < 1_000_000 else args.reps_long):
            for k, fn in fns.items():
                ms[k].append(timed(fn))
        for k, fn in fns.items():
            emit({"points": n, "fs": FS, "frequencies": nf, "arm": k, **summary(ms[k]), "kernels_ms": kernel_ms(fn)})
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("".join(json.dumps(d) + "\n" for d in lines))


if __name__ == "__main__":
    main()
