"""Batched Monte-Carlo sweep of single-buffer NLS fits (SURVEY 8f-3; BASELINE config 5).

The reference runs this study one trial per process: ``run_efficiency_trial`` (workers.py:132-189) simulates
one buffer in 'snr' mode with ``trial_num`` as the noise seed and fits it with ``init_m = m_true`` and
``parallel=False``; ``Experiment.run`` (experiments.py:288-458) maps that over a grid x trials with a
``multiprocessing.Pool`` and reduces each grid point to mean / std / min / max / worst-case.  Notebook
``1.1_CRLB-test`` (cells 3-6) compares Var(m_hat) with ``calculate_crlb_for_m`` (helpers.py:16-45).

Here the whole grid is one pass (``dfk_nls_sweep_dev``): every realisation is drawn by the counter-based 'snr' generator
(statistically, not bitwise, the reference's MT19937 noise) inside the demodulation kernel's shared memory -- no record
ever touches HBM; the samples are bit for bit those ``dfk_synth_snr_slab_dev`` writes for the same seed -- fitted cold
in one launch, and reduced on the device.  Waves bound the resident harmonic vectors and rows (default 8 GB).
"""
from __future__ import annotations

import math

import numpy as np

from . import _lib
from . import fit as fit_tunables


def bessel_j(nmax: int, x: float) -> np.ndarray:
    """J_0..J_nmax(x) by Miller's backward recurrence (host copy of csrc/dfk_bessel.cuh, |x| <= 200)."""
    ax = abs(float(x))
    out = np.zeros(nmax + 1)
    if ax == 0.0:
        out[0] = 1.0
        return out
    mstart = max(int(ax + 12.0 * (0.5 * ax) ** (1.0 / 3.0) + 5.0), nmax + 2)
    mstart += mstart & 1
    tox = 2.0 / ax
    bp, b, total = 0.0, 1.0e-200, 0.0
    for k in range(mstart, 0, -1):
        if k <= nmax:
            out[k] = b
        if k % 2 == 0:
            total += 2.0 * b
        bp, b = b, k * tox * b - bp
        if abs(b) > 1e200:
            b *= 1e-200
            bp *= 1e-200
            total *= 1e-200
            out *= 1e-200
    out[0] = b
    out /= total + b
    if x < 0:
        out[1::2] *= -1.0
    return out


def crlb_sigma_m(m_true: float, ndata: int, snr_db: float, buffer_size: int) -> float:
    """Cramer-Rao bound on sigma(m) as the reference defines it (helpers.py:16-45): Fisher matrix = J^T J of the
    harmonic model at [a, m, phi, psi] = [1, m_true, 0, 0], I/Q noise variance 0.5 / SNR / (2 R)."""
    sigma_iq_sq = 0.5 / 10 ** (snr_db / 10.0) / (2 * buffer_size)
    j = np.arange(1, ndata + 1)
    bes = bessel_j(ndata + 1, m_true)
    B, dB = bes[1:ndata + 1], 0.5 * (bes[0:ndata] - bes[2:ndata + 2])
    q, dq = np.cos(j * np.pi / 2.0), np.cos(j * np.pi / 2.0 + np.pi / 2.0)
    # at psi = 0 the sine half of the model vanishes except in the psi column
    jac = np.zeros((2 * ndata, 4))
    jac[:ndata, 0] = q * B
    jac[:ndata, 1] = q * dB
    jac[:ndata, 2] = dq * B
    jac[ndata:, 3] = -(q * B) * j
    try:
        cov = np.linalg.inv(jac.T @ jac)
    except np.linalg.LinAlgError:
        return float("nan")
    return float(math.sqrt(cov[1, 1] * sigma_iq_sq))


def nls_sweep(m_values, n_trials, snr_db=40.0, f_samp=200e3, f_mod=1000.0, n=1, ndata=15, init_a=1.6, init_m=None,
              amp=1.0, visibility=1.0, phi0=0.0, psi0=0.0, seed=0, device=0, max_resident_bytes=8 << 30,
              tunables_from=None, return_rows=False, uncertainties=False, _seed_stride=None, _raw_stats=False):
    """Fit ``n_trials`` independent single-buffer realisations at every m in ``m_values``.

    init_m: None -> each realisation starts from its true m (workers.py:167-173); a float -> the same cold start
    everywhere (the grid fallback then does the work, as in the reference).
    Returns a dict of per-m arrays: ``m_mean, m_std, m_min, m_max, m_worst`` (largest |m_hat - m|), the same for
    ``amp, phi, psi``, ``ssq_mean``, ``fitok`` fractions ``[len(m), 3]``, ``crlb_sigma_m``, and with return_rows the
    raw ``[len(m), n_trials, 8]`` table.
    uncertainties: also fit every realisation's parameter covariance (``dfk_nls_sweep_cov_dev``) and report per m
    ``amp_err_rms, m_err_rms, phi_err_rms, psi_err_rms``, the square root of the mean predicted variance over all trials
    -- to set beside ``*_std`` and ``crlb_sigma_m``; with return_rows also the ``[len(m), n_trials, 8]`` table ``cov``.
    """
    import torch
    ms = np.atleast_1d(np.asarray(m_values, dtype=np.float64))
    ctx = _lib.get_context(device)
    dev = torch.device("cuda", device)
    R = int(f_samp / f_mod * n)
    w0 = 2.0 * np.pi * f_mod / f_samp
    opts = fit_tunables.current_lm_opts(tunables_from)
    # no record is ever resident: a wave holds harmonic vectors, means and result rows only
    per_fit = 8 * (2 * int(ndata) + 1) + 8 * _lib.ROW_STRIDE + 16
    per_wave = max(1, min(int(n_trials), int(max_resident_bytes // (len(ms) * per_fit))))
    seed_stride = int(n_trials) if _seed_stride is None else int(_seed_stride)
    # (uncertainties add 64 bytes of covariance per fit on top; the waves, and so the rows, stay those without them)
    waves = []
    all_rows = [] if return_rows else None
    all_cov = [] if return_rows and uncertainties else None
    with torch.cuda.device(dev):
        rows = torch.empty((len(ms), per_wave, _lib.ROW_STRIDE), dtype=torch.float64, device=dev)
        cov = torch.empty((len(ms), per_wave, _lib.COV_STRIDE), dtype=torch.float64, device=dev) if uncertainties else None
        truth = torch.from_numpy(np.stack([np.full_like(ms, amp), ms, np.full_like(ms, phi0), np.full_like(ms, psi0)], 1)).to(dev)
        center = torch.zeros((len(ms), 7), dtype=torch.float64, device=dev)
        center[:, :4] = truth
        ctx.use_torch_stream()
        try:
            done = 0
            while done < n_trials:
                nw = min(per_wave, n_trials - done)
                rv = rows[:, :nw] if nw == per_wave else torch.empty((len(ms), nw, _lib.ROW_STRIDE), dtype=torch.float64,
                                                                      device=dev)
                cv = None
                if uncertainties:
                    cv = cov[:, :nw] if nw == per_wave else torch.empty((len(ms), nw, _lib.COV_STRIDE), dtype=torch.float64,
                                                                         device=dev)
                # realisation t of grid point i is noise stream seed + i * seed_stride + t, whatever the wave it falls
                # in: generated inside the demodulation kernel (dfk_nls_sweep_dev), fitted cold in one launch
                ctx.nls_sweep_dev(ms, nw, done, seed_stride, R, int(ndata), f_samp, f_mod, rv.data_ptr(), amp=amp,
                                  visibility=visibility, phi0=phi0, psi0=psi0, snr_db=snr_db, seed=seed, init_a=init_a,
                                  init_m=init_m, opts=opts, cov_ptr=cv.data_ptr() if uncertainties else None)
                # per-m statistics of the wave in one pass of the reduction kernel: columns amp, m, phi, psi, (dc,) ssq,
                # fitok; "worst" measured from the true parameters
                st = torch.empty((len(ms), 7, _lib.TRIAL_STATS_DOUBLES), dtype=torch.float64, device=dev)
                ctx.trial_stats_dev(rv.data_ptr(), len(ms), nw, 7, _lib.ROW_STRIDE, st.data_ptr(), center_ptr=center.data_ptr())
                cst = None
                if uncertainties:  # mean predicted variance per m: covariance columns 0, 3, 5, 6 of the same reduction
                    cst = torch.empty((len(ms), 7, _lib.TRIAL_STATS_DOUBLES), dtype=torch.float64, device=dev)
                    ctx.trial_stats_dev(cv.data_ptr(), len(ms), nw, 7, _lib.COV_STRIDE, cst.data_ptr())
                waves.append((nw, st, cst))
                if return_rows:
                    all_rows.append(rv.cpu().numpy().copy())
                    if uncertainties:
                        all_cov.append(cv.cpu().numpy().copy())
                done += nw
            torch.cuda.current_stream(dev).synchronize()
        finally:
            ctx.use_default_stream()
    tr = truth.cpu().numpy()
    part = {"n": int(n_trials), "truth": tr, "sum": 0.0, "sumsq": 0.0, "ok": 0.0, "ssq": 0.0,
            "min": np.full((len(ms), 4), np.inf), "max": np.full((len(ms), 4), -np.inf), "worst": np.zeros((len(ms), 4))}
    if uncertainties:
        part["var_sum"], part["var_n"] = 0.0, 0.0
    for nw, st, cst in waves:
        if cst is not None:  # nan-aware: weight each wave's mean by its number of finite trials
            c_ = cst.cpu().numpy()[:, [0, 3, 5, 6]]
            part["var_sum"] = part["var_sum"] + np.nan_to_num(c_[:, :, 0]) * c_[:, :, 5]
            part["var_n"] = part["var_n"] + c_[:, :, 5]
        s_ = st.cpu().numpy()
        mean, std = s_[:, :4, 0], s_[:, :4, 1]
        part["sum"] = part["sum"] + mean * nw
        part["sumsq"] = part["sumsq"] + nw * (std ** 2 + (mean - tr) ** 2)  # about the truth
        part["min"] = np.minimum(part["min"], s_[:, :4, 2])
        part["max"] = np.maximum(part["max"], s_[:, :4, 3])
        part["worst"] = np.maximum(part["worst"], np.abs(s_[:, :4, 4] - tr))
        part["ssq"] = part["ssq"] + s_[:, 5, 0] * nw
        # fitok takes the values 0, 1, 2: its first two moments give the three counts
        f1 = s_[:, 6, 0] * nw
        f2 = (s_[:, 6, 1] ** 2 + s_[:, 6, 0] ** 2) * nw
        n2 = np.rint((f2 - f1) / 2.0)
        n1 = np.rint(f1 - 2.0 * n2)
        part["ok"] = part["ok"] + np.stack([nw - n1 - n2, n1, n2], 1)
    if _raw_stats:
        return part
    out = _combine_partials(ms, [part], ndata, snr_db, R)
    if uncertainties:
        with np.errstate(invalid="ignore", divide="ignore"):
            rms = np.sqrt(part["var_sum"] / part["var_n"])
        for c, name in enumerate(("amp", "m", "phi", "psi")):
            out[f"{name}_err_rms"] = rms[:, c]
    if return_rows:
        out["rows"] = np.concatenate(all_rows, axis=1)
        if uncertainties:
            out["cov"] = np.concatenate(all_cov, axis=1)
    return out


def nls_sweep_sharded(m_values, n_trials, group=None, device=None, seed=0, **kwargs):
    """``nls_sweep`` with the realisations split over the ranks of a ``torch.distributed`` group (one process per GPU).

    Realisations are independent, so the split is by realisation index: rank r draws trials
    ``slab_bounds(n_trials, world, r)`` with its own disjoint seed range and nothing crosses the GPUs but the per-m
    sufficient statistics at the end (a few hundred bytes, gathered as Python objects).  Every rank returns the
    combined result; ``return_rows`` is not supported here.
    """
    import torch
    import torch.distributed as dist
    from .sharding import slab_bounds

    if kwargs.pop("return_rows", False):
        raise ValueError("return_rows is a single-GPU option")
    if kwargs.pop("uncertainties", False):
        raise ValueError("uncertainties is a single-GPU option")
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    lo, hi = slab_bounds(int(n_trials), world, rank)
    if device is None:
        device = torch.cuda.current_device()
    ms = np.atleast_1d(np.asarray(m_values, dtype=np.float64))
    part = None
    if hi > lo:
        # the seed of realisation t of grid point i must not depend on the split: nls_sweep uses
        # seed + done + i * n_trials with `done` counting from 0, so shift by lo and keep the per-m stride global
        part = _sweep_partial(ms, hi - lo, seed + lo, int(n_trials), device, **kwargs)
    parts = [None] * world
    dist.all_gather_object(parts, part, group=group)
    return _combine_partials(ms, [p for p in parts if p is not None], kwargs.get("ndata", 15), kwargs.get("snr_db", 40.0),
                             int(kwargs.get("f_samp", 200e3) / kwargs.get("f_mod", 1000.0) * kwargs.get("n", 1)))


def _sweep_partial(ms, n_local, seed0, seed_stride, device, **kwargs):
    """Sufficient statistics of n_local realisations per m (numpy, host)."""
    out = nls_sweep(ms, n_local, seed=seed0, device=device, _seed_stride=seed_stride, _raw_stats=True, **kwargs)
    return out


def _combine_partials(ms, parts, ndata, snr_db, R):
    nt = float(sum(p["n"] for p in parts))
    total = sum(p["sum"] for p in parts)
    sq = sum(p["sumsq"] for p in parts)
    mean = total / nt
    tr = parts[0]["truth"]
    var = np.maximum(sq / nt - (mean - tr) ** 2, 0.0)
    out = {"m_values": ms, "n_trials": int(nt), "fitok": sum(p["ok"] for p in parts) / nt,
           "ssq_mean": sum(p["ssq"] for p in parts) / nt,
           "crlb_sigma_m": np.array([crlb_sigma_m(m, ndata, snr_db, R) for m in ms])}
    mn = np.min([p["min"] for p in parts], axis=0)
    mx = np.max([p["max"] for p in parts], axis=0)
    worst = np.max([p["worst"] for p in parts], axis=0)
    for c, name in enumerate(("amp", "m", "phi", "psi")):
        out[f"{name}_mean"], out[f"{name}_std"] = mean[:, c], np.sqrt(var[:, c])
        out[f"{name}_min"], out[f"{name}_max"], out[f"{name}_worst"] = mn[:, c], mx[:, c], worst[:, c]
    return out
