#!/usr/bin/env python
"""Monte-Carlo driver at BASELINE config-5 size (development tool): nls_sweep over m = 2..20, generation included."""
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from deepfmkit_b200 import _lib, nls_sweep  # noqa: E402


def main():
    n_trials = int(float(sys.argv[1])) if len(sys.argv) > 1 else 1_000_000
    ms = list(range(2, 21))
    ctx = _lib.get_context(0)
    lib = _lib.load_library()
    if len(sys.argv) > 2:
        lib.dfk_dev_set(b"DFK_NO_SWEEP_FUSE", int(sys.argv[2]))
    for rep in range(3):
        ctx.profile_enable(True)
        ctx.profile_read(reset=True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = nls_sweep(ms, n_trials, snr_db=40.0, ndata=15, seed=rep, max_resident_bytes=16 << 30)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        prof = ctx.profile_read(reset=True)
        print(json.dumps({"what": "nls_sweep", "n_trials": n_trials, "fits": n_trials * len(ms), "wall_ms": dt * 1e3,
                          "fits_per_s": n_trials * len(ms) / dt, "gen_demod_ms": prof["demod_ms"], "lm_ms": prof["lm_ms"],
                          "fitok0": float(out["fitok"][:, 0].min()), "std_over_crlb": float((out["m_std"] / out["crlb_sigma_m"]).mean())}),
              flush=True)


if __name__ == "__main__":
    main()
