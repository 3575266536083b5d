#!/usr/bin/env python
"""Cost of the conditioned spectra on the LPSD plan, ``lcsd_conditioned`` (development tool).

Shapes (seeded series resident on the device, fs = 50 Hz):

  - Cx = 8 witnesses, Cy = 256 targets at N = 50 000 points (one cfg-3 record of 1000 s at the 50 Hz fit rate);
  - Cx = 64 witnesses, Cy = 1 target at N = 1.8e6 points, and at N = 50 000.

The pairwise route runs at the two 50 000-point shapes only.  Its ``lcsd`` finish sums every term of a frequency row
one after another in one CTA; at 64 witnesses and 1.8e6 points the row of K = 1.1e5 segments alone streams ~14 GB
through one SM, minutes per call.

At each shape:

  1. call time, alternated repetitions after a warm-up of both arms (CUDA events around each public call, which
     includes the plan and the copies back): ``lcsd_conditioned``, and the pairwise route a user has without it --
     ``lcsd(x, x)`` + ``lcsd(x, y)`` + a batched ``numpy.linalg.solve`` per frequency on the host;
  2. kernel time per call from one ``torch.profiler`` pass per arm, after the timed ones (``lcsd_segment_kernel``,
     ``lcsd_gram_kernel``, ``lcsd_cond_kernel``, ``lcsd_finish_kernel``);
  3. the Gram kernel's fp64 rate from the algorithmic count sum_j 8 K_j (Cx (Cx + 1) / 2 + Cx Cy + Cy) flops (a
     complex multiply-add is 8 flops) over its profiled time;
  4. the largest difference between the two routes' H and Sres (scaled as the tests scale them), so that the times
     compared are of the same result.

One JSON line per measurement, with the card's name and power limit read in the same run, to stdout and to --out
(default profiles/r03_lcsd_cond_cost.jsonl).
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
from deepfmkit_b200 import lcsd, lcsd_conditioned  # noqa: E402

FS = 50.0
SHAPES = {"8x256": (8, 256, 50_000, True), "64x1": (64, 1, 1_800_000, False), "64x1_50k": (64, 1, 50_000, True)}


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
    """Witnesses: independent random walks plus white noise; targets: a random mix of the witnesses plus noise."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = 1e-3 * torch.cumsum(torch.randn(cx, n, generator=g, device="cuda", dtype=torch.float64), 1)
    x += 1e-3 * torch.randn(cx, n, generator=g, device="cuda", dtype=torch.float64)
    mix = torch.randn(cy, cx, generator=g, device="cuda", dtype=torch.float64) / cx ** 0.5
    y = mix @ x + 1e-3 * torch.randn(cy, n, generator=g, device="cuda", dtype=torch.float64)
    return x.contiguous(), y.contiguous()


def pairwise(x, y):
    """The route without lcsd_conditioned: the witness matrix and the cross terms from two lcsd calls, then a batched
    solve per frequency on the host (rows with fewer segments than witnesses left NaN)."""
    cx = x.shape[0]
    xx, xy = lcsd(x, x, FS), lcsd(x, y, FS)
    S = np.moveaxis(xx["Sxy"], -1, 0)  # [nf, Cx, Cx]
    B = np.moveaxis(xy["Sxy"], -1, 0)  # [nf, Cx, Cy]
    ok = xx["navs"] >= cx
    H = np.full(B.shape, np.nan + 1j * np.nan)
    H[ok] = np.linalg.solve(S[ok], B[ok])
    sres = xy["Syy"] - np.sum(np.conj(B) * H, axis=1).real.T
    return {"H": np.moveaxis(H, 0, -1), "Sres": sres, "Syy": xy["Syy"], "Sxx": xy["Sxx"], "navs": xy["navs"]}


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
        if ev.device_type == DeviceType.CUDA and "lcsd_" in ev.name:
            key = ev.name.split("(")[0].split("::")[-1]
            out[key] = out.get(key, 0.0) + ev.time_range.elapsed_us() / 1e3 / calls
    return out


def compare(got, ref):
    """Largest differences between the two routes' H (scaled by sqrt(Syy / Sxx_aa)) and Sres (over Syy)."""
    hs = np.sqrt(got["Syy"][None, :, :] / np.real(np.einsum("aaj->aj", got["Sxx"]))[:, None, :])
    okh = ~np.isnan(ref["H"]) & ~np.isnan(got["H"])
    oks = ~np.isnan(ref["Sres"]) & ~np.isnan(got["Sres"])
    return {"max_dH_scaled": float(np.max((np.abs(got["H"] - ref["H"]) / hs)[okh], initial=0.0)),
            "max_dSres_over_Syy": float(np.max((np.abs(got["Sres"] - ref["Sres"]) / got["Syy"])[oks], initial=0.0)),
            "nan_rows_equal": bool(np.array_equal(np.isnan(got["Sres"]), np.isnan(ref["Sres"])))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default=",".join(SHAPES), help=f"any of {sorted(SHAPES)}")
    ap.add_argument("--reps", type=int, default=5, help="alternated repetitions per arm")
    ap.add_argument("--gram-calls", type=int, default=5, help="profiled calls for the Gram kernel's time")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_lcsd_cond_cost.jsonl"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("probe_lcsd_cond needs a CUDA device")
    info = card()
    lines = []

    def emit(d):
        d = {**d, **info}
        print(json.dumps(d), flush=True)
        lines.append(d)

    for name in args.shapes.split(","):
        cx, cy, n, with_pairwise = SHAPES[name]
        x, y = series(cx, cy, n, seed=cx * 1000 + cy)
        fns = {"lcsd_conditioned": lambda: lcsd_conditioned(x, y, FS)}
        if with_pairwise:
            fns["pairwise"] = lambda: pairwise(x, y)
        res = {k: fn() for k, fn in fns.items()}  # warm-up of every arm, and their results
        torch.cuda.synchronize()
        got = res["lcsd_conditioned"]
        navs = got["navs"]
        agree = compare(got, res["pairwise"]) if with_pairwise else None
        ms = {k: [] for k in fns}
        for _ in range(args.reps):
            for k, fn in fns.items():
                ms[k].append(timed(fn))
        flops = float(np.sum(8.0 * navs * (cx * (cx + 1) / 2 + cx * cy + cy)))
        base = {"shape": name, "Cx": cx, "Cy": cy, "points": n, "fs": FS, "frequencies": len(got["f"]),
                "segments": int(navs.sum())}
        for k, fn in fns.items():
            kern = kernel_ms(fn, args.gram_calls if k == "lcsd_conditioned" else 1)
            d = {**base, "arm": k, **summary(ms[k]), "kernels_ms": kern}
            if k == "lcsd_conditioned":
                gram = kern.get("lcsd_gram_kernel", float("nan"))
                d.update({"gram_flops": flops, "gram_ms": gram, "gram_fp64_tflops": flops / (gram * 1e-3) / 1e12,
                          "agreement_with_pairwise": agree})
            emit(d)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("".join(json.dumps(d) + "\n" for d in lines))


if __name__ == "__main__":
    main()
