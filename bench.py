#!/usr/bin/env python
"""Benchmark of the DFMI readout hot path (BASELINE.json: NLS fit buffers/s; demod HBM GB/s vs peak).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--no-configs] [--dump-outputs DIR]

Headline workload (config.workload): BASELINE config 2, "long single channel" -- f_mod = 1 kHz, f_samp = 1 MHz,
3600 s of synthetic 'snr'-mode DFMI (m = 6, 40 dB), n = 20 periods per buffer (R = 20000 samples), N = 10
harmonics: 180 000 buffers = 3.6e9 samples = 28.8 GB of fp64 per GPU.  A step is one whole NLS readout of the
record (demodulate + fit every buffer).  With N > 1 GPUs (torchrun, one process per GPU) every rank holds its own
3600 s record (weak scaling): the path has no exchange step, so ranks share nothing but the barrier around the timed
region.

value         buffers/s over all ranks, record resident in HBM (28.8 GB >> 126 MB L2: no flush needed)
e2e           the same through the drop-in fitter call, StandardNLSFitter.fit(raw) on a pandas frame in ordinary
              (pageable) host memory: staged H2D slabs -> kernels -> D2H rows -> result frame, all timed, max over
              ranks; e2e.pinned_c_abi is the C-ABI call on a pinned record beside it
roofline      the demodulation kernel: algorithmic bytes (8 R + 8 (2N+1) per buffer) / its CUDA-event time
cpu_baseline  the reference itself (baseline/_ref) -- else the oracle port -- on the host cores, bounded sample
configs       (N = 1) the other four BASELINE configs measured in the same process under the same clock sampling:
              cfg 1, cfg 3 (one resident wave), cfg 4 (the whole 100 s, streamed slab by slab), cfg 5
strong        (N > 1) ONE cfg-2 record, and one cfg-3 wave, split over the N GPUs: wall time incl. seed broadcast
              and row gather

--dump-outputs DIR writes what the last timed step computed, rank 0's result columns (amp, m, phi, psi, dc, ssq,
fitok: 180 000 float64 each, 10 MB in all) as DIR/<column>.npy.  The record is generated from a fixed seed, so two
builds run with the same arguments can be compared output for output (on hosts with the same core count: the
warm-start schedule, SCHED, follows it).
"""
import argparse
import json
import os
import sys
import threading
import time

os.environ.setdefault("TQDM_DISABLE", "1")  # the reference wraps its pool in tqdm

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

F_SAMP, F_MOD, N_CYCLES, NDATA = 1e6, 1000.0, 20, 10
SECONDS = 3600.0
M_TRUE, SNR_DB = 6.0, 40.0
R = int(F_SAMP / F_MOD * N_CYCLES)
NBUF = int(SECONDS * F_SAMP) // R
INIT = [1.6, 6.0, 0.0, 0.0]
# warm-start schedule of the timed readouts: the drop-in default, StandardNLSFitter.fit(parallel=True, n_cores=None)
# = the reference's pool schedule with one chunk per host core (fitters.py:397-417)
SCHED = max(1, os.cpu_count() or 1)
METRIC, UNIT = "nls_fit_buffers_per_sec", "buffers/s"
WORKLOAD = ("cfg2 long single channel: f_mod=1kHz f_samp=1MHz 3600s synthetic DFMI (m=6, SNR 40dB), "
            "n=20 (R=20000), ndata=10, NLS fit per buffer")


def config_dict(n_gpus):
    return {"workload": WORKLOAD, "buffers_per_gpu": NBUF, "samples_per_gpu": NBUF * R, "R": R, "ndata": NDATA,
            "record_bytes_per_gpu": NBUF * R * 8, "schedule": f"buffer 0 cold, the rest in {SCHED} warm-start chunks (the "
            "drop-in default: parallel=True, n_cores=os.cpu_count())", "sharding": f"{n_gpus} contiguous time slabs, one per GPU, no collective",
            "l2": "inputs (28.8 GB per GPU) exceed the 126 MB L2; no flush between steps"}


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic_per_launch():
    """dram bytes per demod launch from the committed ncu capture of this command, if there is one."""
    path = os.path.join(ROOT, "profiles", "demod_traffic.json")
    try:
        with open(path) as f:
            return json.load(f).get("dram_bytes_per_launch")
    except Exception:
        return None


def lm_flops_per_fit(counters, fits, ndata):
    """Algorithmic flops per fit from the work the kernels counted (SURVEY 8d's per-call costs, N harmonics):
    model+Jacobian F_c = 3M + 90N + 2S, residual F_s = 3M + 12N + 2S with the Miller steps M counted on device,
    S = 60 flop per sincos, F_m = 100 per damped solve."""
    per = {k: v / max(fits, 1) for k, v in counters.items()}
    return (per["n_state"] * (90 * ndata + 120) + per["n_ssq"] * (12 * ndata + 120) + per["n_solve"] * 100 +
            3 * per["n_bessel_steps"]), per


def lm_roofline(counters, fits, nbuf, lm_ms, peak_tflops, ndata=NDATA):
    flop_per_fit, _ = lm_flops_per_fit(counters, fits, ndata)
    achieved = flop_per_fit * nbuf / (lm_ms * 1e-3) / 1e12
    return {"bound": "fp64", "achieved": achieved, "peak": peak_tflops, "unit": "TFLOP/s",
            "frac": achieved / peak_tflops if peak_tflops else None, "flop_per_fit": flop_per_fit,
            "peak_source": "dfk_probe_fp64: DFMA chains measured on this GPU in this run",
            "note": "algorithmic flops of the reference's formulation; the kernel's block-diagonal normal equations "
                    "execute about half of the model+Jacobian figure"}


# ---- clocks sampled during the timed regions ------------------------------------------------------------
class ClockSampler:
    """Samples SM clock and throttle reasons while inside a `with` block; blocks accumulate."""
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x10: "sync_boost"}

    def __init__(self, device):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            uuid = str(torch.cuda.get_device_properties(device).uuid)
            try:
                self.h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(device)
            self.nv = pynvml
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                get = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                    nv.nvmlDeviceGetCurrentClocksThrottleReasons
                mask = get(self.h)
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.01)

    def __enter__(self):
        if self.nv is not None:
            self._stop.clear()
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._thread is not None:
            self._thread.join()
            self._thread = None

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ---- CPU arm: the reference itself when baseline/_ref holds it, else the oracle port --------------------
def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


class CpuArm:
    """The reference's own CPU implementation of the path (fitters.py) from baseline/_ref when it is importable
    (kind "reference"), else the oracle's restatement of it (kind "port").  Inputs come from the oracle's 'snr'
    generator, which is pinned bit-exactly to the reference's (tests/test_oracle_golden.py)."""

    def __init__(self):
        from oracle import dfmi_oracle as orc
        self.orc = orc
        self.kind, self.why = "port", None
        try:
            sys.path.insert(0, os.path.join(ROOT, "baseline"))
            import install_ref
            self.core, self.rfit, self.rfitters = install_ref.import_reference()
            import logging
            logging.getLogger().setLevel(logging.ERROR)
            self.kind = "reference"
        except Exception as e:  # no baseline/_ref on this box: time the port
            self.why = f"{type(e).__name__}: {e}"[:160]

    def _raw(self, x, f_samp, f_mod):
        import pandas as pd
        raw = self.core.DeepRawObject(data=pd.DataFrame(x, columns=["ch0"]))
        raw.f_samp, raw.f_mod, raw.label = f_samp, f_mod, "bench"
        return raw

    def nls_pool(self, x, f_samp, f_mod, n, ndata, cores):
        """Seconds for StandardNLSFitter.fit(parallel=True, n_cores=cores) on record x (pool start-up included)."""
        if self.kind == "reference":
            raw = self._raw(x, f_samp, f_mod)
            fitter = self.rfitters.StandardNLSFitter({"n": n, "ndata": ndata})
            t0 = time.perf_counter()
            df = fitter.fit(raw, parallel=True, n_cores=cores)
            dt = time.perf_counter() - t0
            assert len(df) == len(x) // int(f_samp / f_mod * n)
            return dt
        t0 = time.perf_counter()
        rows = self.orc.nls_fit_pool(x, f_samp, f_mod, n, ndata, n_procs=cores)
        dt = time.perf_counter() - t0
        assert rows.shape[0] == len(x) // int(f_samp / f_mod * n)
        return dt

    def ekf(self, x, f_samp, f_mod, n):
        if self.kind == "reference":
            raw = self._raw(x, f_samp, f_mod)
            fitter = self.rfitters.EKFFitter({"n": n})
            t0 = time.perf_counter()
            fitter.fit(raw, verbose=False)
            return time.perf_counter() - t0
        t0 = time.perf_counter()
        self.orc.ekf_track(x, f_samp, f_mod, n)
        return time.perf_counter() - t0


_ARM = None


def cpu_arm():
    global _ARM
    if _ARM is None:
        _ARM = CpuArm()
    return _ARM


def _cfg5_job(job):
    """One realisation of the CRLB sweep as workers.py:132-189 runs it: synthesise one period, fit it cold at m_true."""
    m, seed = job
    arm = cpu_arm()
    x = arm.orc.snr_signal(float(m), 200e3, 1000.0, 1e-3, 40.0, seed=seed)
    if arm.kind == "reference":
        raw = arm._raw(x, 200e3, 1000.0)
        return float(arm.rfitters.StandardNLSFitter({"n": 1, "ndata": 15}).fit(raw, parallel=False, init_m=float(m))["m"][0])
    return float(arm.orc.nls_fit(x, 200e3, 1000.0, 1, 15, init_m=float(m))[0, 1])


def cpu_baseline_for(cfg, cores):
    """Bounded CPU sample of one BASELINE config -> a cpu_baseline object."""
    from multiprocessing import Pool
    arm = cpu_arm()
    orc = arm.orc
    if cfg == "cfg2":
        n_buf = max(200, min(2000, 25 * cores))
        x = orc.snr_signal(M_TRUE, F_SAMP, F_MOD, n_buf * R / F_SAMP, SNR_DB, seed=1)
        dt = arm.nls_pool(x, F_SAMP, F_MOD, N_CYCLES, NDATA, cores)
        return {"value": n_buf / dt, "unit": UNIT, "cores": cores, "kind": arm.kind,
                "sample": f"{n_buf} buffers ({n_buf * R / F_SAMP:.0f} s of the cfg2 record), "
                          "StandardNLSFitter.fit(parallel=True, n_cores=cores), pool start-up included"}
    if cfg in ("cfg1", "cfg3"):
        secs = 10.0 if cfg == "cfg1" else 20.0
        x = orc.snr_signal(6.0, 200e3, 1000.0, secs, 40.0, seed=0)
        dt = arm.nls_pool(x, 200e3, 1000.0, 20, 10, cores)
        nb = int(secs * 200e3) // 4000
        return {"value": nb / dt, "unit": UNIT, "cores": cores, "kind": arm.kind,
                "sample": f"1 channel x {secs:.0f} s ({nb} buffers of 4000 samples), pool schedule, start-up included"}
    if cfg == "cfg5":
        jobs = [(m, s) for m in range(2, 21) for s in range(100)]
        t0 = time.perf_counter()
        with Pool(cores) as pool:
            out = pool.map(_cfg5_job, jobs, chunksize=25)
        dt = time.perf_counter() - t0
        assert len(out) == len(jobs)
        return {"value": len(jobs) / dt, "unit": "fits/s", "cores": cores, "kind": arm.kind,
                "sample": f"{len(jobs)} realisations (100 per m in 2..20), Pool over realisations, signal synthesis "
                          "included as in workers.py:132-189"}
    if cfg == "cfg4":
        x = orc.snr_signal(6.0, 200e3, 1000.0, 0.25, 40.0, seed=0)
        dt = arm.ekf(x, 200e3, 1000.0, 20)
        return {"value": len(x) / dt, "unit": "samples/s", "cores": 1, "kind": arm.kind,
                "sample": "1 channel x 0.25 s (50000 steps) on one core; channels are independent, so a box scales this "
                          f"by its core count ({cores} here)"}
    raise SystemExit(f"unknown workload {cfg}")


def run_reference(args):
    """--impl reference: the reference's CPU path (fitters.py:395-428: buffer 0, then a process pool over chunks of
    the rest) on all host cores, each step a bounded sample of cfg 2.  Rank 0 alone works."""
    if int(os.environ.get("RANK", "0")) != 0:
        return 0
    cores = host_cores()
    arm = cpu_arm()
    if args.workload != "cfg2":
        out = cpu_baseline_for(args.workload, cores)
        out.update({"impl": "reference", "workload": args.workload, "metric": METRIC if out["unit"] == UNIT else
                    ("single_buffer_fits_per_sec" if out["unit"] == "fits/s" else "ekf_samples_per_sec")})
        emit(out)
        return 0
    # size the per-step sample so that the whole K + W run stays within ~2 minutes
    cal = arm.orc.snr_signal(M_TRUE, F_SAMP, F_MOD, 200 * R / F_SAMP, SNR_DB, seed=1)
    rate = 200 / arm.nls_pool(cal, F_SAMP, F_MOD, N_CYCLES, NDATA, cores)
    budget_s = min(10.0, 100.0 / (args.steps + args.warmup))
    n_buffers = int(max(200, min(4000, rate * budget_s)))
    x = arm.orc.snr_signal(M_TRUE, F_SAMP, F_MOD, n_buffers * R / F_SAMP, SNR_DB, seed=1)
    for _ in range(args.warmup):
        arm.nls_pool(x, F_SAMP, F_MOD, N_CYCLES, NDATA, cores)
    times = [arm.nls_pool(x, F_SAMP, F_MOD, N_CYCLES, NDATA, cores) for _ in range(args.steps)]
    dt = sum(times) / len(times)
    value = n_buffers / dt
    sample = (f"{n_buffers} buffers ({n_buffers * R / F_SAMP:.0f} s of the cfg2 record) per step, "
              "StandardNLSFitter.fit(parallel=True, n_cores=cores), pool start-up included")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "samples_per_sec": value * R, "config": config_dict(args.gpus),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": arm.kind, "sample": sample,
                             "port_because": arm.why},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)
    return 0


def bind_to_gpu_numa_node(device):
    """Pin this rank to the CPUs of its GPU's NUMA node before it allocates host memory, so that the e2e leg's
    host record is first-touched on the socket the GPU hangs off (matters once several ranks stream at once)."""
    try:
        import torch
        prop = torch.cuda.get_device_properties(device)
        bus, dom, dev = prop.pci_bus_id, getattr(prop, "pci_domain_id", 0), getattr(prop, "pci_device_id", 0)
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev:02x}.0/numa_node"
        node = int(open(path).read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = cpus & set(os.sched_getaffinity(0))
        if allowed:
            os.sched_setaffinity(0, allowed)
            return node
    except Exception:
        pass
    return None


# ---- GPU arm: the other BASELINE configs (N = 1) -----------------------------------------------------------
def event_timed(torch, stream, fn, reps, warm=1):
    """Mean milliseconds of fn over reps launches (CUDA events on the launching stream, after warm-up)."""
    for _ in range(warm):
        fn()
    stream.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(reps):
        fn()
    e1.record(stream)
    stream.synchronize()
    return e0.elapsed_time(e1) / reps


def nls_config(torch, ctx, stream, clocks, name, f_samp, n, ndata, channels, seconds, reps, peak, fp64_peak, m_list=None,
               note="", waves=1):
    """One NLS config, device-generated and resident: whole readout, demod and LM times, both rooflines."""
    import numpy as np
    from deepfmkit_b200 import _lib
    from deepfmkit_b200 import fit as tunables
    Rc = int(f_samp / F_MOD * n)
    T = int(round(seconds * f_samp)) // Rc * Rc
    bpc = T // Rc
    nbuf = channels * bpc
    w0 = 2.0 * np.pi * F_MOD / f_samp
    opts = tunables.current_lm_opts()
    x = torch.empty(channels * T, dtype=torch.float64, device="cuda")
    rows = torch.empty((nbuf, _lib.ROW_STRIDE), dtype=torch.float64, device="cuda")
    init_dev = None
    if m_list is None:
        ctx.synth_snr_dev(x.data_ptr(), T, channels, f_samp, F_MOD, 6.0, dphi=2 * np.pi / channels, seed=5)
        sched, truth_m = SCHED, 6.0
    else:  # cfg 5: `channels` single-buffer realisations per m, each started cold at its true m (workers.py:167-173)
        per = channels // len(m_list)
        g = np.zeros((channels, 4))
        g[:, 0] = 1.6
        for i, m in enumerate(m_list):
            ctx.synth_snr_dev(x.data_ptr() + i * per * T * 8, T, per, f_samp, F_MOD, float(m), seed=1000 * i)
            g[i * per:(i + 1) * per, 1] = m
        init_dev = torch.from_numpy(g).cuda()
        sched, truth_m = _lib.SCHED_INDEPENDENT, float(np.mean(m_list))
    stream.synchronize()

    def whole():
        ctx.nls_fit_batch_dev(x.data_ptr(), channels, bpc, T, Rc, ndata, w0, INIT, init_dev.data_ptr() if init_dev is not None
                              else None, 4 if init_dev is not None else 0, sched, opts, rows.data_ptr())

    whole()
    stream.synchronize()
    ctx.lm_counters(reset=True)
    ctx.profile_enable(True)
    ctx.profile_read(reset=True)
    with clocks:
        ms = event_timed(torch, stream, whole, reps, warm=3)
    prof = ctx.profile_read(reset=True)
    ctx.profile_enable(False)
    cnt = ctx.lm_counters(reset=True)
    r = rows[:: max(1, nbuf // 4096)].cpu().numpy()
    assert abs(float(np.mean(r[:, 1])) - truth_m) < 0.05 and np.mean(r[:, 6] == 0) > 0.9, f"{name}: fits are wrong"
    demod_ms = prof["demod_ms"] / max(prof["demod_regions"], 1)
    lm_ms = prof["lm_ms"] / max(prof["lm_regions"], 1)
    alg = (8 * Rc + 8 * (2 * ndata + 1)) * nbuf
    fits = nbuf * (reps + 3)
    flop_per_fit, per_fit = lm_flops_per_fit(cnt, fits, ndata)
    lm_tf = flop_per_fit * nbuf / (lm_ms * 1e-3) / 1e12
    out = {"workload": note, "value": nbuf / (ms * 1e-3), "unit": UNIT if m_list is None else "fits/s",
           "ms_per_step": ms, "buffers": nbuf, "samples": nbuf * Rc, "R": Rc, "ndata": ndata, "channels": channels,
           "record_bytes": nbuf * Rc * 8, "samples_per_sec": nbuf * Rc / (ms * 1e-3), "kernel_ms": demod_ms,
           "roofline": {"bound": "hbm", "kernel": "demod", "achieved": alg / (demod_ms * 1e-3) / 1e9, "peak": peak,
                        "unit": "GB/s", "frac": alg / (demod_ms * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_launch": alg,
                        "kernel_ms": demod_ms, "share_of_step": demod_ms / ms},
           "lm": {"kernel_ms": lm_ms, "share_of_step": lm_ms / ms, "fits_per_sec": nbuf / (lm_ms * 1e-3), "per_fit": per_fit,
                  "roofline": {"bound": "fp64", "achieved": lm_tf, "peak": fp64_peak, "unit": "TFLOP/s",
                               "frac": lm_tf / fp64_peak if fp64_peak else None, "flop_per_fit": flop_per_fit}}}
    if waves > 1:
        # the whole config: `waves` consecutive waves of every channel, each generated on the device where the previous
        # one lay (t0 advances, so the record is the continuous one) and fitted -- generation inside the timed region
        def all_waves():
            for w in range(waves):
                ctx.synth_snr_slab_dev(x.data_ptr(), T, channels, T, w * T, f_samp, F_MOD, 6.0, dphi=2 * np.pi / channels, seed=5)
                whole()

        with clocks:
            ms_all = event_timed(torch, stream, all_waves, 2, warm=1)
        r = rows[:: max(1, nbuf // 4096)].cpu().numpy()
        assert abs(float(np.mean(r[:, 1])) - truth_m) < 0.05 and np.mean(r[:, 6] == 0) > 0.9, f"{name}: last wave is wrong"
        out["whole_config"] = {"waves": waves, "buffers": nbuf * waves, "samples": nbuf * Rc * waves,
                               "record_bytes": nbuf * Rc * 8 * waves, "ms_incl_generator": ms_all,
                               "buffers_per_sec": nbuf * waves / (ms_all * 1e-3),
                               "note": "each wave device-generated in place of the previous one, then fitted; every "
                                       "wave fits its own buffer 0 cold"}
    del x, rows, init_dev
    torch.cuda.empty_cache()
    return out


def ekf_config(torch, ctx, stream, clocks, channels, seconds, slab_seconds, peak, fp64_peak):
    """cfg 4 whole: every channel for `seconds`, generated slab by slab on the device (the 655 GB record never
    exists) and filtered by dfk_ekf_stream_dev with the state carried from slab to slab; the generator runs on a
    second buffer so that it is not inside the EKF kernel's own timing (both are inside the wall time)."""
    import numpy as np
    from deepfmkit_b200 import _lib
    f_samp, n = 200e3, 20
    Rc = int(f_samp / F_MOD * n)
    Ts = int(slab_seconds * f_samp) // Rc * Rc
    nslab = int(round(seconds / slab_seconds))
    slabs = [torch.empty(channels * Ts, dtype=torch.float64, device="cuda") for _ in range(2)]
    rows = torch.empty((channels, Ts // Rc, _lib.ROW_STRIDE), dtype=torch.float64, device="cuda")
    state = torch.zeros((channels, 32), dtype=torch.float64, device="cuda")
    opts = _lib.default_ekf_opts()
    # whole-record moments of the clean signal + noise are known in closed form for the synthetic record; the
    # filter takes them as the caller-supplied init_dc / R_val, as dfk_ekf_host's first pass would provide them
    opts.init_dc = 1.0
    opts.r_val = 0.5

    def gen(i):
        ctx.synth_snr_slab_dev(slabs[i & 1].data_ptr(), Ts, channels, Ts, i * Ts, f_samp, F_MOD, 6.0,
                               dphi=2 * np.pi / channels, seed=3)

    def run(nsl):
        for i in range(nsl):
            gen(i)
            ctx.ekf_stream_dev(slabs[i & 1].data_ptr(), Ts, channels, 1, Ts, Rc, f_samp, F_MOD, opts, i * Ts,
                               state.data_ptr(), rows.data_ptr())

    run(2)  # warm-up
    stream.synchronize()
    ctx.profile_enable(True)
    ctx.profile_read(reset=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with clocks:
        e0.record(stream)
        run(nslab)
        e1.record(stream)
        stream.synchronize()
    wall_ms = e0.elapsed_time(e1)
    prof = ctx.profile_read(reset=True)
    ctx.profile_enable(False)
    last = rows[:, -1, :].cpu().numpy()
    assert abs(float(np.mean(last[:, 1])) - 6.0) < 0.01 and np.all(last[:, 6] == 1), "cfg4: the filter lost the signal"
    samples = channels * Ts * nslab
    ekf_ms = prof["ekf_ms"]
    flops = 330.0 * samples  # SURVEY 8d: ~330 flop per sample as the reference writes the update (2 sincos = 120 of them)
    tf = flops / (ekf_ms * 1e-3) / 1e12
    out = {"workload": f"cfg4: EKF over {channels} channels x {seconds:.0f} s at 200 kHz ({samples:.3g} samples, "
                       f"{samples * 8 / 1e9:.0f} GB streamed from the device generator in {slab_seconds:g} s slabs)",
           "value": samples / (ekf_ms * 1e-3), "unit": "samples/s", "kernel_ms": ekf_ms, "wall_ms_incl_generator": wall_ms,
           "samples": samples, "channels": channels, "seconds_per_channel": seconds,
           "steps_per_sec_per_channel": Ts * nslab / (ekf_ms * 1e-3), "m_last_mean": float(np.mean(last[:, 1])),
           "roofline": {"bound": "fp64-latency", "achieved": tf, "peak": fp64_peak, "unit": "TFLOP/s",
                        "frac": tf / fp64_peak if fp64_peak else None, "flop_per_sample": 330.0,
                        "hbm_GBps": samples * 8 / (ekf_ms * 1e-3) / 1e9, "hbm_frac": samples * 8 / (ekf_ms * 1e-3) / 1e9 / peak,
                        "note": "one thread per channel, sequential in time: bounded by the latency of the ~33-operation "
                                "dependent chain per sample, not by either roofline (DESIGN.md 4-K3)"}}
    del slabs, rows, state
    torch.cuda.empty_cache()
    return out


def other_configs(torch, ctx, stream, clocks, peak, fp64_peak, with_cpu):
    out = {}
    out["cfg1"] = nls_config(torch, ctx, stream, clocks, "cfg1", 200e3, 20, 10, 1, 10.0, 200, peak, fp64_peak,
                             note="cfg1 README quickstart: 1 channel x 10 s at 200 kHz = 500 buffers of 4000 (launch bound)")
    out["cfg3"] = nls_config(torch, ctx, stream, clocks, "cfg3", 200e3, 20, 10, 256, 100.0, 20, peak, fp64_peak,
                             note="cfg3 resident wave: 256 channels x 100 s of the 1000 s config = 1.28e6 buffers, 41 GB "
                                  "(the full config is ten such waves per GPU, or 1.25 per GPU on 8: whole_config)", waves=10)
    out["cfg4"] = ekf_config(torch, ctx, stream, clocks, 4096, 100.0, 1.0, peak, fp64_peak)
    ms = list(range(2, 21))
    out["cfg5"] = nls_config(torch, ctx, stream, clocks, "cfg5", 200e3, 1, 15, 1_000_000 * len(ms), 1e-3, 10, peak,
                             fp64_peak, m_list=ms,
                             note="cfg5 CRLB Monte Carlo: 1e6 realisations x 19 m in 2..20, one period (200 samples) each, "
                                  "ndata = 15, cold start at m_true = 1.9e7 single-buffer fits, 30.4 GB")
    out["cfg5"]["monte_carlo_driver"] = sweep_config(torch, ctx, ms, 1_000_000)
    if with_cpu:
        cores = host_cores()
        for name in out:
            out[name]["cpu_baseline"] = cpu_baseline_for(name, cores)
    return out


def sweep_config(torch, ctx, ms, n_trials):
    """The same study through the Monte-Carlo driver (deepfmkit_b200.nls_sweep): realisations generated inside the
    demodulation kernel, one cold fit launch, per-m statistics on the device -- generation INCLUDED, nothing resident
    but harmonic vectors and rows."""
    from deepfmkit_b200 import _lib, nls_sweep
    hctx = _lib.get_context(torch.cuda.current_device())
    nls_sweep(ms, n_trials // 10, seed=1)  # warm-up
    best, prof = 1e30, None
    for rep in range(3):
        hctx.profile_enable(True)
        hctx.profile_read(reset=True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = nls_sweep(ms, n_trials, snr_db=40.0, ndata=15, seed=rep, max_resident_bytes=16 << 30)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        p_ = hctx.profile_read(reset=True)
        hctx.profile_enable(False)
        if dt < best:
            best, prof = dt, p_
    fits = n_trials * len(ms)
    return {"value": fits / best, "unit": "fits/s", "wall_ms": best * 1e3, "fits": fits,
            "generate_and_demodulate_ms": prof["demod_ms"], "lm_ms": prof["lm_ms"],
            "fitok0_min": float(out["fitok"][:, 0].min()),
            "std_over_crlb_mean": float((out["m_std"] / out["crlb_sigma_m"]).mean()),
            "api": "deepfmkit_b200.nls_sweep(range(2, 21), 1e6, ndata=15): host wall clock incl. generation, fits, statistics"}


# ---- GPU arm: ingest and post-fit steps around the readout (SURVEY 8f-2, 8f-4) ---------------------------------
def ingest_and_post(torch, ctx, stream, x, rows, nbuf, w0, opts, local):
    """(a) the record as 16-bit ADC counts in host memory -> widened on the device -> fitted where it lies;
    (b) a DFMSWPM text file parsed on the device; (c) block means of the resident record and the LPSD of the fitted
    phase.  Host wall clock, rank 0, one GPU."""
    import numpy as np
    import tempfile
    from deepfmkit_b200 import StandardNLSFitter, _lib, load_binary, load_raw_device, lpsd, vectorized_downsample
    out = {}
    hctx = _lib.get_context(local)
    n = nbuf * R
    # (c) post-fit: boxcar of the raw-rate record to the fit rate, LPSD of phi (180 000 points, the reference's defaults)
    y = vectorized_downsample(x, R)  # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    y = vectorized_downsample(x, R)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    out["downsample"] = {"GBps": n * 8 / dt / 1e9, "ms": dt * 1e3, "samples": n, "R": R,
                         "api": "vectorized_downsample(record, R) on the resident record (dsp.py:3-56)"}
    del y
    phi = rows[:, 2].contiguous()
    lpsd(phi, F_MOD / N_CYCLES)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = lpsd(phi, F_MOD / N_CYCLES, return_type="dict")
    dt = time.perf_counter() - t0
    out["lpsd"] = {"ms": dt * 1e3, "points": int(phi.shape[0]), "frequencies": int(len(res["f"])),
                   "api": "lpsd(fit.phi, fs) with DeepFitObject's defaults: Kaiser 200 dB, Jdes 500, Kdes 100 (core.py:590-609)"}
    # (a) 16-bit acquisition format: a quarter of the fp64 bytes cross PCIe
    scale = 2.5 / 32768.0
    host = np.empty(n, dtype=np.int16)
    chunk = 1 << 27
    for off in range(0, n, chunk):  # quantise chunk by chunk: no record-sized temporaries
        host[off:off + chunk] = torch.clamp(torch.round(x[off:off + chunk] / scale), -32768, 32767).to(torch.int16).cpu().numpy()
    fitter = StandardNLSFitter({"n": N_CYCLES, "ndata": NDATA})

    def go():
        raw = load_binary(host, F_SAMP, F_MOD, time_major=True, scale=scale, device=local)[0]
        return fitter.fit(raw)
    df = go()
    t0 = time.perf_counter()
    df = go()
    dt = time.perf_counter() - t0
    got = df.to_numpy(dtype=float)
    assert got.shape[0] == nbuf and np.all(got[:, 6] == 0) and abs(got[:, 1].mean() - M_TRUE) < 1e-2
    out["int16_record"] = {"value": nbuf / dt, "unit": UNIT, "ms": dt * 1e3, "h2d_bytes": n * 2, "h2d_GBps": n * 2 / dt / 1e9,
                           "api": "load_binary(int16 counts in pageable host memory) -> StandardNLSFitter.fit on the "
                                  "device-resident record -> result frame"}
    del host
    # (b) text: 1e6 rows x 2 channels of repr() floats written 12 times over (~470 MB) to a temporary file
    block_rows, reps = 1_000_000, 12
    vals = x[:block_rows * 2].cpu().numpy().reshape(block_rows, 2)
    block = "".join(f"{a!r} {b!r} \n" for a, b in vals.tolist())
    with tempfile.NamedTemporaryFile("w", suffix=".txt", delete=False) as f:
        path = f.name
        f.write("% raw_data\n% bench\n% Number of channels: 2\n% Start time: 0\n% Sampling frequency: 1000000.0\n"
                "% Modulation frequency: 1000.0\n%\n%\n%\n%\n%\n%\nch0 ch1 \n")
        for _ in range(reps):
            f.write(block)
    del block
    nbytes = os.path.getsize(path)
    rows_txt = block_rows * reps
    load_raw_device(path, device=local)  # warm-up: staging buffers, page cache
    t0 = time.perf_counter()
    data, hdr = load_raw_device(path, device=local)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    # the two device phases on their own: upload + row index, then the parse
    off = hdr["data_offset"]
    t1 = time.perf_counter()
    _, nr = hctx.text_load_file(path, off)
    t2 = time.perf_counter()
    hctx.text_parse_dev(2, data.data_ptr(), nr)
    torch.cuda.synchronize()
    t3 = time.perf_counter()
    hctx.text_release()
    got = data[:, :1000].cpu().numpy()
    ok = bool(nr == rows_txt and hdr["nbad"] == 0 and np.allclose(got, vals[:1000].T, rtol=1e-11, atol=0)
              and np.array_equal(got, data[:, block_rows:block_rows + 1000].cpu().numpy()))
    os.unlink(path)
    out["text_file"] = {"GBps_text": nbytes / dt / 1e9, "samples_per_sec": rows_txt * 2 / dt, "ms": dt * 1e3, "bytes": nbytes,
                        "rows": rows_txt, "channels": 2, "matches_input": ok,
                        "file_to_hbm_and_row_index_ms": (t2 - t1) * 1e3, "parse_kernels_ms": (t3 - t2) * 1e3,
                        "parse_kernels_GBps_text": nbytes / (t3 - t2) / 1e9,
                        "api": "load_raw_device(DFMSWPM raw_data text file): file -> pinned stagers -> HBM -> device parser "
                               "(bit-identical to the reference's pandas.read_csv); page cache warm"}
    return out


# ---- GPU arm: strong scaling of one record over the ranks (N > 1) --------------------------------------------
def strong_scaling(torch, dist, ctx, local, rank, world, w0, opts, single_gpu_ms):
    """ONE cfg-2 record split over the ranks as contiguous time slabs (sharding.nls_fit_sharded: rank 0 fits buffer
    0, 32-byte broadcast, all slabs concurrently, rows gathered on rank 0) and one cfg-3 wave split by channel."""
    import numpy as np
    from deepfmkit_b200 import _lib
    from deepfmkit_b200.fitters import nls_fit_batch
    from deepfmkit_b200.sharding import gather_rows, nls_fit_sharded, slab_bounds
    lo, hi = slab_bounds(NBUF, world, rank)
    xs = torch.empty((hi - lo) * R, dtype=torch.float64, device="cuda")
    ctx.use_torch_stream()
    ctx.synth_snr_slab_dev(xs.data_ptr(), (hi - lo) * R, 1, (hi - lo) * R, lo * R, F_SAMP, F_MOD, M_TRUE, snr_db=SNR_DB, seed=1000)
    torch.cuda.synchronize()
    ctx.use_default_stream()
    first = torch.empty(R, dtype=torch.float64, device="cuda")  # buffer 0 of the record, on every rank (160 kB)
    ctx.use_torch_stream()
    ctx.synth_snr_slab_dev(first.data_ptr(), R, 1, R, 0, F_SAMP, F_MOD, M_TRUE, snr_db=SNR_DB, seed=1000)
    torch.cuda.synchronize()
    ctx.use_default_stream()
    times = []
    table = None
    for it in range(5):  # the first two passes warm allocations (device scratch, the two page-locked return buffers)
        dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        table = nls_fit_sharded(xs, NBUF, R, NDATA, w0, INIT, device=local, first_buffer=first)
        dt = time.perf_counter() - t0
        t = torch.tensor([dt], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        if it >= 2:
            times.append(float(t.item()))
    rec_s = sum(times) / len(times)
    if rank == 0:
        assert table.shape == (NBUF, 8) and np.all(table[:, 6] == 0) and abs(table[:, 1].mean() - M_TRUE) < 1e-3
    del xs
    # cfg 3 wave by channel: 256 channels x 100 s, 256 / world channels per rank, rows gathered on rank 0
    C, Rc = 256, 4000
    T = int(100.0 * 200e3)
    clo, chi = slab_bounds(C, world, rank)
    xc = torch.empty((chi - clo, T), dtype=torch.float64, device="cuda")
    ctx.use_torch_stream()
    ctx.synth_snr_dev(xc.data_ptr(), T, chi - clo, 200e3, F_MOD, 6.0, phi0=2 * np.pi * clo / C, dphi=2 * np.pi / C, seed=5 + clo)
    torch.cuda.synchronize()
    ctx.use_default_stream()
    ctimes = []
    for it in range(5):
        dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        rows = nls_fit_batch(xc, 200e3, F_MOD, 20, ndata=10, seeded=True, device=local, return_tensor=True)
        flat = rows.reshape(chi - clo, -1)
        tab = gather_rows(flat, C, dst=0)  # GPU to GPU over NVLink, then one D2H of the 82 MB table on rank 0
        dt = time.perf_counter() - t0
        t = torch.tensor([dt], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        if it >= 2:
            ctimes.append(float(t.item()))
    wave_s = sum(ctimes) / len(ctimes)
    if rank == 0:
        assert tab.shape == (C, (T // Rc) * 8)
    del xc
    torch.cuda.empty_cache()
    nb3 = C * (T // Rc)
    return {"scaling": "strong", "n_gpus": world,
            "cfg2_one_record": {"buffers": NBUF, "wall_ms": rec_s * 1e3, "buffers_per_sec": NBUF / rec_s,
                                "single_gpu_kernel_ms": single_gpu_ms,
                                "includes": "buffer 0 fitted on every rank (no exchange before the kernels), slab kernels on every rank, "
                                            "NCCL gather of the rows to rank 0 (GPU to GPU), one D2H of the 11.5 MB table (host "
                                            "wall clock, max over ranks)"},
            "cfg3_wave_by_channel": {"buffers": nb3, "wall_ms": wave_s * 1e3, "buffers_per_sec": nb3 / wave_s,
                                     "includes": "per-rank batched readout of its channels, NCCL gather to rank 0, one D2H of the 82 MB table"}}


# ---- GPU arm --------------------------------------------------------------------------------------------
def dump_outputs(out_dir, rows):
    """The frame's columns of the row table (what StandardNLSFitter.fit returns for the record) as <column>.npy."""
    import numpy as np
    from deepfmkit_b200.fitters import RESULT_COLUMNS
    os.makedirs(out_dir, exist_ok=True)
    table = rows.cpu().numpy()
    for i, name in enumerate(RESULT_COLUMNS):
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(table[:, i], dtype=np.float64))


def run_gpu(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from deepfmkit_b200 import DeepRawObject, StandardNLSFitter, _lib
    from deepfmkit_b200 import fit as tunables

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun --nproc-per-node {args.gpus}")
    torch.cuda.set_device(local)
    numa_node = bind_to_gpu_numa_node(local) if world > 1 else None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    ctx = _lib.Context(local, own_stream=True)
    stream = torch.cuda.Stream(device=local)
    w0 = 2.0 * np.pi * F_MOD / F_SAMP
    opts = tunables.current_lm_opts()
    clocks = ClockSampler(local)

    with torch.cuda.stream(stream):
        x = torch.empty(NBUF * R, dtype=torch.float64, device="cuda")
        rows = torch.empty((NBUF, _lib.ROW_STRIDE), dtype=torch.float64, device="cuda")
        ctx.use_torch_stream(stream)
        ctx.synth_snr_dev(x.data_ptr(), NBUF * R, 1, F_SAMP, F_MOD, M_TRUE, snr_db=SNR_DB, seed=1000 + rank)

        def step():
            ctx.nls_fit_dev(x.data_ptr(), NBUF, R, NDATA, w0, INIT, SCHED, opts, rows.data_ptr())

        for _ in range(args.warmup):
            step()
        stream.synchronize()
        ctx.lm_counters(reset=True)
        ctx.profile_enable(True)
        ctx.profile_read(reset=True)
        launches0 = ctx.launch_count()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        with clocks:
            ev0.record(stream)
            for _ in range(args.steps):
                step()
            ev1.record(stream)
            stream.synchronize()
        barrier()
        elapsed_ms = ev0.elapsed_time(ev1)
        launches = ctx.launch_count() - launches0
        prof = ctx.profile_read(reset=True)
        ctx.profile_enable(False)
        counters = ctx.lm_counters(reset=True)
        head = rows[:4096].cpu().numpy()
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, rows)
        fp64_peak = ctx.probe_fp64_tflops() if rank == 0 else None

    # sanity: the timed work produced real fits
    assert np.all(head[:, 6] == 0) and abs(head[:, 1].mean() - M_TRUE) < 1e-3, "bench fits are wrong"
    ms_per_step = max_over_ranks(elapsed_ms) / args.steps
    value = world * NBUF / (ms_per_step * 1e-3)

    # ---- end to end through the drop-in fitter call ---------------------------------------------------------
    import pandas as pd
    import psutil
    # every rank holds its own host copy; keep the sum under 40% of the box's RAM (same answer on every rank)
    host_total = psutil.virtual_memory().total
    e2e_nbuf = NBUF
    while e2e_nbuf * R * 8 * world > 0.40 * host_total and e2e_nbuf > 1000:
        e2e_nbuf //= 2
    x_pg = np.empty(e2e_nbuf * R, dtype=np.float64)  # ordinary pageable memory: what a pandas frame holds
    chunk = 1 << 26
    for off in range(0, e2e_nbuf * R, chunk):
        x_pg[off:off + chunk] = x[off:min(off + chunk, e2e_nbuf * R)].cpu().numpy()
    raw = DeepRawObject(data=pd.DataFrame(x_pg.reshape(-1, 1), columns=["ch0"], copy=False), f_samp=F_SAMP, f_mod=F_MOD,
                        label="bench")
    fitter = StandardNLSFitter({"n": N_CYCLES, "ndata": NDATA})
    e2e_steps = max(1, min(args.steps, 3))
    df = fitter.fit(raw, device=local)  # warm-up (allocations, stagers)
    barrier()
    with clocks:
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            df = fitter.fit(raw, device=local)
        e2e_local = (time.perf_counter() - t0) / e2e_steps
    barrier()
    e2e_s = max_over_ranks(e2e_local)
    e2e_value = world * e2e_nbuf / e2e_s
    got = df.to_numpy(dtype=float)
    assert got.shape == (e2e_nbuf, 7) and np.array_equal(got[:1024, 6], head[:1024, 6])
    assert np.max(np.abs(got[:1024, :4] - head[:1024, :4])) < 1e-9
    h2d_rank = e2e_nbuf * R * 8 / e2e_local / 1e9
    per_rank = [None] * world
    if world > 1:
        dist.all_gather_object(per_rank, {"rank": rank, "h2d_GBps": h2d_rank, "numa_node": numa_node})
    else:
        per_rank = [{"rank": 0, "h2d_GBps": h2d_rank, "numa_node": numa_node}]
    del raw, df
    # the C-ABI host entry on a pinned record (DMA straight from the caller's memory), for comparison
    xh = torch.empty(e2e_nbuf * R, dtype=torch.float64, pin_memory=True)
    xh.numpy()[:] = x_pg
    del x_pg
    rows_h = torch.empty((e2e_nbuf, _lib.ROW_STRIDE), dtype=torch.float64, pin_memory=True).numpy()
    hctx = _lib.get_context(local)
    hctx.nls_fit_host(xh.numpy(), R, NDATA, w0, INIT, seeded=SCHED, opts=opts, rows_out=rows_h)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        hctx.nls_fit_host(xh.numpy(), R, NDATA, w0, INIT, seeded=SCHED, opts=opts, rows_out=rows_h)
    pinned_local = (time.perf_counter() - t0) / e2e_steps
    barrier()
    pinned_s = max_over_ranks(pinned_local)
    del xh

    configs = strong = around = None
    if world == 1 and not args.no_configs:
        around = ingest_and_post(torch, ctx, stream, x, rows, NBUF, w0, opts, local)
    if world == 1 and not args.no_configs:
        peak, _ = measured_peak()
        del x, rows
        torch.cuda.empty_cache()
        with torch.cuda.stream(stream):
            ctx.use_torch_stream(stream)
            configs = other_configs(torch, ctx, stream, clocks, peak, fp64_peak, with_cpu=True)
    elif world > 1 and not args.no_strong:
        del x, rows
        torch.cuda.empty_cache()
        strong = strong_scaling(torch, dist, _lib.get_context(local), local, rank, world, w0, opts, None)

    if rank == 0:
        peak, peak_src = measured_peak()
        demod_ms = prof["demod_ms"] / max(prof["demod_regions"], 1)
        lm_ms = prof["lm_ms"] / max(prof["lm_regions"], 1)
        alg_bytes = (8 * R + 8 * (2 * NDATA + 1)) * NBUF
        achieved = alg_bytes / (demod_ms * 1e-3) / 1e9
        fits = max(args.steps * NBUF, 1)
        cores = host_cores()
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "samples_per_sec": value * R, "config": config_dict(world),
            "roofline": {"bound": "hbm", "kernel": "demod_fold_kernel", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "traffic": ncu_traffic_per_launch(),
                         "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes,
                         "kernel_ms": demod_ms, "share_of_step": demod_ms / ms_per_step},
            "lm": {"kernel_ms_per_step": lm_ms, "share_of_step": lm_ms / ms_per_step,
                   "fits_per_sec": NBUF / (lm_ms * 1e-3),
                   "per_fit": {k: v / fits for k, v in counters.items()},
                   "roofline": lm_roofline(counters, fits, NBUF, lm_ms, fp64_peak)},
            "cpu_baseline": cpu_baseline_for("cfg2", cores),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": e2e_nbuf * R * 8,
                    "d2h_bytes_per_step": e2e_nbuf * _lib.ROW_STRIDE * 8, "ms_per_step": e2e_s * 1e3,
                    "buffers_per_gpu": e2e_nbuf,
                    "api": "StandardNLSFitter({'n': 20, 'ndata': 10}).fit(raw) on a pandas frame in pageable host memory "
                           "(staged by the library through pinned buffers); includes building the result frame; max over ranks",
                    "per_rank": per_rank,
                    "pinned_c_abi": {"value": world * e2e_nbuf / pinned_s, "unit": UNIT, "ms_per_step": pinned_s * 1e3,
                                     "api": "dfk_nls_fit_host on a pinned host record, rows into pinned memory"}},
            "gpu_launches": launches,
        }
        if around is not None:
            line["ingest_and_post"] = around
        if configs is not None:
            line["configs"] = configs
        if strong is not None:
            strong["cfg2_one_record"]["single_gpu_kernel_ms"] = ms_per_step
            line["strong"] = strong
        line["clocks"] = clocks.summary()
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    ctx.close()
    return 0


_JSON_FD = None


def emit(line):
    """The one JSON line goes to the real stdout; everything else any library prints was sent to stderr."""
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main():
    global _JSON_FD
    # NCCL and friends print banners on fd 1; keep stdout clean for the JSON line
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=["cfg1", "cfg2", "cfg3", "cfg4", "cfg5"],
                    help="reference arm only: which BASELINE config's bounded CPU sample to time (default: the contract's cfg2)")
    ap.add_argument("--no-configs", action="store_true", help="skip the cfg 1/3/4/5 block of the N = 1 line")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling block of the N > 1 line")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's result columns (rank 0) to DIR/<column>.npy, float64")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        raise SystemExit("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl == "reference":
        raise SystemExit("--dump-outputs applies to the GPU arm, not --impl reference")
    if args.impl == "reference":
        return run_reference(args)
    return run_gpu(args)


if __name__ == "__main__":
    sys.exit(main())
