#!/usr/bin/env python
"""Ring depth of the single-period lock-in kernel (development tool)."""
import json, os, sys
import numpy as np
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from deepfmkit_b200 import _lib  # noqa: E402

def main():
    ctx = _lib.Context(0); ctx.use_torch_stream(); lib = _lib.load_library()
    C, R, N = 7_600_000, 200, 15
    x = torch.empty(C * R, dtype=torch.float64, device="cuda")
    ctx.synth_snr_dev(x.data_ptr(), R, C, 200e3, 1000.0, 6.0, seed=5)
    qi = torch.empty((C, 2 * N), dtype=torch.float64, device="cuda"); dc = torch.empty(C, dtype=torch.float64, device="cuda")
    ref = None
    for nst in (12, 8, 6, 5):
        lib.dfk_dev_clear(); lib.dfk_dev_set(b"DFK_PERIOD_NSTAGES", nst)
        best = 1e30
        for _ in range(4):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); ctx.demod(x.data_ptr(), C, R, N, 2 * np.pi / 200, qi.data_ptr(), dc.data_ptr()); b.record(); b.synchronize()
            best = min(best, a.elapsed_time(b))
        same = True if ref is None else bool(torch.equal(qi, ref))
        ref = qi.clone() if ref is None else ref
        print(json.dumps({"nstages_max": nst, "ms": best, "GBps": C * (R * 8 + 8 * (2 * N + 1)) / best / 1e6, "same": same}), flush=True)
    lib.dfk_dev_clear()

if __name__ == "__main__":
    main()
