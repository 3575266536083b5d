#!/usr/bin/env python
"""Cost of the time-domain stability estimates, ``stability`` (development tool).

Shapes (seeded 'freq' series resident on the device, fs = 50 Hz, all four kinds):

  - 1 x 1.8e5 at octave tau (the phi column of a cfg-2 fit), 1 x 1.8e6 and 256 x 1.8e5 at octave tau;
  - 1 x 1.8e6 at 100 tau per decade.

At each shape:

  1. call time, alternated repetitions after a warm-up of every arm (CUDA events around each public call, which
     includes the copies back and the final synchronise);
  2. kernel time per call from one ``torch.profiler`` pass, after the timed ones;
  3. the terms kernel's traffic in units of whole passes over the double-double running sums: one pass reads x and S
     once, 2 C (Nx + 1) 16 bytes; the kernel's time over (number of tau x one pass at the HBM data-sheet rate);
  4. the host route a user has without this function, numpy fp64 cumsum over the mean-removed series (as allantools
     computes it), timed with a host clock (1 repetition where it takes seconds), and the largest relative difference
     between the two.

One JSON line per measurement, with the card's name and power limit read in the same run, to stdout and to --out
(default profiles/r03_stability_cost.jsonl).
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from deepfmkit_b200 import stability  # noqa: E402

FS = 50.0
KINDS = ("oadev", "mdev", "tdev", "ohdev")
# name: (C, N, taus per decade or None for octave, host repetitions)
SHAPES = {"1x1.8e5_octave": (1, 180_000, None, 3), "1x1.8e6_octave": (1, 1_800_000, None, 1),
          "256x1.8e5_octave": (256, 180_000, None, 1), "1x1.8e6_100perdecade": (1, 1_800_000, 100, 1)}
HBM_BYTES_PER_S = 7.7e12  # NVIDIA's HGX B200 data sheet, one GPU


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
            "reps": len(ms)}


def series(c, n, seed):
    """White noise plus a random walk plus a linear drift: every kind sees a different noise type dominate."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    y = torch.randn(c, n, generator=g, device="cuda", dtype=torch.float64)
    y += 1e-2 * torch.cumsum(torch.randn(c, n, generator=g, device="cuda", dtype=torch.float64), 1)
    y += 1e-6 * torch.arange(n, device="cuda", dtype=torch.float64)
    return y.contiguous()


def host_route(y, ms):
    """[4, C, n_m] from fp64 phase = cumsum of the mean-removed series / fs, mdev by allantools' running form."""
    C = y.shape[0]
    out = np.full((4, C, len(ms)), np.nan)
    for c in range(C):
        x = np.concatenate([[0.0], np.cumsum(y[c] - y[c].mean())]) / FS
        Nx = x.size
        for t, m in enumerate(int(m) for m in ms):
            tau = m / FS
            na, nh = Nx - 2 * m, Nx - 3 * m
            if na > 0:
                d = x[2 * m:2 * m + na] - 2 * x[m:m + na] + x[:na]
                out[0, c, t] = np.sqrt(np.sum(d * d) / (2 * tau * tau * na))
            if nh >= 0:
                v = np.sum(x[2 * m:3 * m] - 2 * x[m:2 * m] + x[:m])
                va = v + np.cumsum(x[3 * m:3 * m + nh] - 3 * x[2 * m:2 * m + nh] + 3 * x[m:m + nh] - x[:nh])
                out[1, c, t] = np.sqrt((v * v + np.sum(va * va)) / (2.0 * m * m * tau * tau * (nh + 1)))
                out[2, c, t] = tau * out[1, c, t] / np.sqrt(3)
            if nh > 0:
                d = x[3 * m:3 * m + nh] - 3 * x[2 * m:2 * m + nh] + 3 * x[m:m + nh] - x[:nh]
                out[3, c, t] = np.sqrt(np.sum(d * d) / (6 * tau * tau * nh))
    return out


def timed(fn):
    s = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(s)
    fn()
    e1.record(s)
    e1.synchronize()
    return e0.elapsed_time(e1)


def kernel_ms(fn, calls=1):
    """Device time per kernel name, per call, over `calls` calls."""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.events():
        if ev.device_type == DeviceType.CUDA and "stab_" in ev.name:
            key = ev.name.split("(")[0].split("::")[-1]
            out[key] = out.get(key, 0.0) + ev.time_range.elapsed_us() / 1e3 / calls
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default=",".join(SHAPES), help=f"any of {sorted(SHAPES)}")
    ap.add_argument("--reps", type=int, default=10, help="repetitions of the device arm")
    ap.add_argument("--profile-calls", type=int, default=3, help="profiled calls for the kernel times")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_stability_cost.jsonl"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("probe_stability needs a CUDA device")
    info = card()
    lines = []

    def emit(d):
        d = {**d, **info}
        print(json.dumps(d), flush=True)
        lines.append(d)

    for name in args.shapes.split(","):
        C, n, per_decade, host_reps = SHAPES[name]
        y = series(C, n, seed=C * 7 + n % 1000)
        Nx = n + 1
        taus = "octave" if per_decade is None else \
            np.logspace(0, np.log10(Nx / 2), int(per_decade * np.log10(Nx / 2)) + 1) / FS
        dev_fn = lambda: stability(y, FS, KINDS, taus, "freq")  # noqa: E731
        got = dev_fn()
        torch.cuda.synchronize()
        yh = y.cpu().numpy()
        t0 = time.perf_counter()
        host = host_route(yh, got["m"])
        host_ms = [1e3 * (time.perf_counter() - t0)]
        for _ in range(host_reps - 1):
            t0 = time.perf_counter()
            host_route(yh, got["m"])
            host_ms.append(1e3 * (time.perf_counter() - t0))
        ms = [timed(dev_fn) for _ in range(args.reps)]
        dev = np.stack([got[k] for k in KINDS])
        rel = np.abs(host / dev - 1)
        kern = kernel_ms(dev_fn, args.profile_calls)
        one_pass = 2.0 * C * (Nx + 1) * 16
        terms = kern.get("stab_terms_kernel", float("nan"))
        base = {"shape": name, "C": C, "N": n, "n_tau": int(got["m"].size), "m_max": int(got["m"].max())}
        emit({**base, "arm": "stability", **summary(ms), "kernels_ms": kern, "bytes_per_pass": one_pass,
              "terms_passes_at_datasheet_hbm": terms * 1e-3 * HBM_BYTES_PER_S / one_pass / got["m"].size})
        emit({**base, "arm": "host_numpy_cumsum", **summary(host_ms),
              "max_rel_diff_from_device": {k: float(np.nanmax(rel[i])) for i, k in enumerate(KINDS)}})
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("".join(json.dumps(d) + "\n" for d in lines))


if __name__ == "__main__":
    main()
