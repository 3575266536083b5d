#!/usr/bin/env python
"""Cost of the time-domain witness subtraction, ``wiener_subtract`` (development tool).

Shapes (seeded series resident on the device; Cx witnesses, Cy targets, L taps, N points):

  - Cx = 1, L = 1, N = 1.8e5: the smallest problem, all overhead;
  - Cx = 8, L = 128 (1024 unknowns, the cap) at N = 1.8e5 (the cfg-2 fit-series length) and N = 1.8e6;
  - Cx = 64, L = 16 (1024 unknowns), N = 1.8e5;
  - Cx = 8, L = 32, Cy = 256, N = 5e4: many targets sharing one factorisation;
  - Cx = 8, L = 16, N = 1.8e5, also through the host route a user has without this function: the explicit lagged
    design matrix (184 MB here) and a numpy solve of its normal equations.

At each shape:

  1. call time, alternated repetitions after a warm-up of every arm (CUDA events around each public call, which
     includes the copies back and the final synchronise);
  2. kernel time per call from one ``torch.profiler`` pass, after the timed ones;
  3. the lag-sum kernel's fp64 rate from the algorithmic count 2 (Cx (Cx + 1) / 2 (2L - 1) + Cx Cy L) N flops (the
     witness lag sums halved by symmetry, then the target lag sums) over its profiled time;
  4. for the host route, the largest differences from it in h (over max |h|) and in the residual (over rms y~).

One JSON line per measurement, with the card's name and power limit read in the same run, to stdout and to --out
(default profiles/r03_wiener_cost.jsonl).
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
from deepfmkit_b200 import wiener_subtract  # noqa: E402

# name: (Cx, Cy, L, N, with the host route)
SHAPES = {"1x1_L1": (1, 1, 1, 180_000, False), "8x1_L128": (8, 1, 128, 180_000, False),
          "8x1_L128_1.8e6": (8, 1, 128, 1_800_000, False), "64x1_L16": (64, 1, 16, 180_000, False),
          "8x256_L32": (8, 256, 32, 50_000, False), "8x1_L16": (8, 1, 16, 180_000, True)}


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


def series(cx, cy, n, seed):
    """Witnesses: white noise plus a slow random walk; targets: a random 3-tap mix of the witnesses plus noise."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(cx, n, generator=g, device="cuda", dtype=torch.float64)
    x += 1e-3 * torch.cumsum(torch.randn(cx, n, generator=g, device="cuda", dtype=torch.float64), 1)
    y = 0.1 * torch.randn(cy, n, generator=g, device="cuda", dtype=torch.float64)
    mix = torch.randn(cy, cx, 3, generator=g, device="cuda", dtype=torch.float64) / cx ** 0.5
    for k in range(3):
        y[:, k:] += mix[:, :, k] @ x[:, :n - k]
    return x.contiguous(), y.contiguous()


def host_route(x, y, L):
    """The route without wiener_subtract: the explicit lagged design matrix on the host and its normal equations."""
    xs, ys = x.cpu().numpy(), y.cpu().numpy()
    cx, n = xs.shape
    k0 = (L - 1) // 2
    n0, M = L - 1 - k0, n - L + 1
    xt = xs - xs.mean(axis=1, keepdims=True)
    yt = (ys - ys.mean(axis=1, keepdims=True))[:, n0:n0 + M].T
    phi = np.empty((M, cx * L))
    for a in range(cx):
        for k in range(L):
            phi[:, a * L + k] = xt[a, n0 + k0 - k:n0 + k0 - k + M]
    h = np.linalg.solve(phi.T @ phi, phi.T @ yt)
    return {"h": h.T.reshape(len(ys), cx, L), "residual": (yt - phi @ h).T}


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
        if ev.device_type == DeviceType.CUDA and ("wiener_" in ev.name or "chol_" in ev.name):
            key = ev.name.split("(")[0].split("::")[-1]
            out[key] = out.get(key, 0.0) + ev.time_range.elapsed_us() / 1e3 / calls
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default=",".join(SHAPES), help=f"any of {sorted(SHAPES)}")
    ap.add_argument("--reps", type=int, default=5, help="alternated repetitions per arm")
    ap.add_argument("--profile-calls", type=int, default=3, help="profiled calls for the kernel times")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_wiener_cost.jsonl"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("probe_wiener needs a CUDA device")
    info = card()
    lines = []

    def emit(d):
        d = {**d, **info}
        print(json.dumps(d), flush=True)
        lines.append(d)

    for name in args.shapes.split(","):
        cx, cy, L, n, with_host = SHAPES[name]
        x, y = series(cx, cy, n, seed=cx * 1000 + cy + L)
        fns = {"wiener_subtract": lambda: wiener_subtract(x, y, L)}
        if with_host:
            fns["host_numpy"] = lambda: host_route(x, y, L)
        res = {k: fn() for k, fn in fns.items()}  # warm-up of every arm, and their results
        torch.cuda.synchronize()
        got = res["wiener_subtract"]
        ms = {k: [] for k in fns}
        for _ in range(args.reps):
            for k, fn in fns.items():
                ms[k].append(timed(fn))
        flops = 2.0 * (cx * (cx + 1) / 2 * (2 * L - 1) + cx * cy * L) * n
        base = {"shape": name, "Cx": cx, "Cy": cy, "taps": L, "points": n, "unknowns": cx * L,
                "explained_median": float(np.median(got["explained"])), "singular": got["singular"]}
        for k in fns:
            d = {**base, "arm": k, **summary(ms[k])}
            if k == "wiener_subtract":
                kern = kernel_ms(fns[k], args.profile_calls)
                lag = kern.get("wiener_lag_kernel", float("nan"))
                d.update({"kernels_ms": kern, "lag_flops": flops, "lag_ms": lag,
                          "lag_fp64_tflops": flops / (lag * 1e-3) / 1e12})
            else:
                ref = res[k]
                rms = float(np.sqrt(np.min(got["var_y"])))
                d["agreement"] = {
                    "max_dh_over_max_h": float(np.max(np.abs(got["h"] - ref["h"])) / np.max(np.abs(ref["h"]))),
                    "max_dres_over_rms_y": float(np.max(np.abs(got["residual"].cpu().numpy() - ref["residual"])) / rms)}
            emit(d)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("".join(json.dumps(d) + "\n" for d in lines))


if __name__ == "__main__":
    main()
