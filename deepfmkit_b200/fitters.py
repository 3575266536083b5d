"""Fitter strategy API of the reference (fitters.py:164-479), backed by the sm_100a library.

``BaseFitter(fit_config).fit(main_raw, **kwargs) -> pandas.DataFrame`` with columns
``amp, m, phi, psi, dc, ssq, fitok`` is unchanged, so these classes drop into the reference's
``fitter_map`` (core.py:452-459).  What changes is what runs underneath: instead of a
``multiprocessing.Pool`` of per-chunk Python loops (fitters.py:395-428), the record goes to the GPU
once and three kernels demodulate and fit every buffer.  There is no CPU path here.

Schedule.  The reference's parallel mode fits buffer 0 from the user's initial guess and seeds every
chunk of the remaining buffers with that result (fitters.py:404-417); within a chunk the warm start
chains from buffer to buffer, and ``parallel=False`` is one chain over the whole record
(fitters.py:370-393).  ``parallel`` and ``n_cores`` keep that meaning here: they select the chunking
(``n_cores`` defaults to ``os.cpu_count()`` as in the reference).  On the GPU every buffer is first
fitted from its chunk's seed in one launch; on a stationary record that is the whole job (the schedules
agree to <= 1e-10 there).  Buffers whose first descent fails -- a record whose phase walks away from
buffer 0 -- are then walked in record order from their predecessor's result, as the chain does
(``lm_chain_kernel``), so flags and parameters follow the reference's schedule on drifting records too.

Additive API for what the reference can only do in a Python loop: :func:`nls_fit_batch` (many channels
/ Monte-Carlo realisations in one launch) and :func:`ekf_fit_batch`.
"""
from __future__ import annotations

import logging
import os
from abc import ABC, abstractmethod

import numpy as np
import pandas as pd

from . import _lib
from . import fit as fit_tunables

RESULT_COLUMNS = ["amp", "m", "phi", "psi", "dc", "ssq", "fitok"]
# uncertainties=True: one-sigma errors from the covariance row (_lib.COV_STRIDE): column -> its variance's index
ERROR_COLUMNS = {"amp_err": 0, "m_err": 3, "phi_err": 5, "psi_err": 6}


def _calculate_fit_params(main_raw, n):
    """(R, fs, nbuf) as fitters.py:62-86: R = int(f_samp / f_mod * n), nbuf = int(len / R)."""
    R = int(main_raw.f_samp / main_raw.f_mod * n)
    fs = main_raw.f_samp / R
    nbuf = int(_record_length(main_raw) / R)
    if nbuf == 0:
        logging.error("Check buffer size !! Calculated nbuf is zero.")
    return R, fs, nbuf


def _device_record(main_raw):
    """The channel's samples as a 1-D float64 CUDA tensor when the record already lives on a GPU, else None."""
    t = getattr(main_raw, "device_data", None)
    if t is None:
        return None
    import torch
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float64):
        return None
    return t.contiguous().view(-1)


def _record_length(main_raw):
    t = _device_record(main_raw)
    if t is not None:
        return int(t.shape[0])
    data = main_raw.data
    return int(data.shape[0])


def _record_values(main_raw, column=None) -> np.ndarray:
    """The channel's samples as one contiguous float64 vector (the caller's object is never modified)."""
    data = main_raw.data
    if column is not None and hasattr(data, "columns"):
        vals = data[column].to_numpy()
    elif hasattr(data, "values"):
        vals = data.values
    else:
        vals = np.asarray(data)
    return np.ascontiguousarray(vals, dtype=np.float64).reshape(-1)


def rows_to_frame(rows: np.ndarray, cov: np.ndarray | None = None) -> pd.DataFrame:
    """[nbuf, >=7] row table -> the reference's result frame (fitok int64, the rest float64).  With the covariance
    rows [nbuf, COV_STRIDE] the frame gains the float64 columns amp_err, m_err, phi_err, psi_err after fitok."""
    df = pd.DataFrame({c: np.asarray(rows[:, i], dtype=np.float64) for i, c in enumerate(RESULT_COLUMNS[:6])})
    df["fitok"] = np.asarray(rows[:, 6]).astype(np.int64)
    if cov is not None:
        for c, i in ERROR_COLUMNS.items():
            df[c] = np.sqrt(np.asarray(cov[:, i], dtype=np.float64))
    return df


class BaseFitter(ABC):
    """Common interface of all fitters (fitters.py:164-208)."""

    def __init__(self, fit_config: dict):
        self.config = fit_config
        if "n" not in self.config:
            raise ValueError("Fit configuration must include 'n'.")

    @abstractmethod
    def fit(self, main_raw, **kwargs) -> pd.DataFrame:
        ...


class StandardNLSFitter(BaseFitter):
    """Frequency-domain NLS readout: lock-in demodulation + 4-parameter LM fit per buffer (fitters.py:322-447).

    ``uncertainties=True`` adds the one-sigma errors ``amp_err, m_err, phi_err, psi_err`` of every buffer: square roots
    of the diagonal of s^2 (J^T J)^-1 at the fitted parameters, s^2 = ssq / (2 ndata - 4) (``dfk_lm_cov``).  They are
    reported whatever the buffer's ``fitok``; filter on it as for the parameters."""

    def fit(self, main_raw, **kwargs) -> pd.DataFrame:
        n = self.config["n"]
        uncertainties = bool(kwargs.get("uncertainties", False))
        ndata = self.config.get("ndata", 10)
        if "ndata" in kwargs:
            ndata = kwargs.pop("ndata")
        init_a = kwargs.get("init_a", 1.6)
        init_m = kwargs.get("init_m", 6.0)
        init_psi = kwargs.get("init_psi", 0.0)
        device = kwargs.get("device", 0)
        # fitters.py:356-368: parallel=True -> n_cores chunks (default: every core), parallel=False -> one chain
        parallel = kwargs.get("parallel", True)
        n_cores = kwargs.get("n_cores", None)
        chunks = max(1, int(n_cores if n_cores is not None else (os.cpu_count() or 1))) if parallel else 1

        R, _, nbuf = _calculate_fit_params(main_raw, n)
        if nbuf == 0:
            return pd.DataFrame()
        w0 = 2.0 * np.pi * main_raw.f_mod / main_raw.f_samp  # fitters.py:39
        opts = fit_tunables.current_lm_opts(kwargs.get("tunables_from"))
        xd = _device_record(main_raw)
        if xd is not None:  # record already on a GPU (io.load_raw / load_binary): fitted where it lies
            import torch
            ctx = _lib.get_context(xd.device.index)
            rows_d = torch.empty((nbuf, _lib.ROW_STRIDE), dtype=torch.float64, device=xd.device)
            cov_d = torch.empty((nbuf, _lib.COV_STRIDE), dtype=torch.float64, device=xd.device) if uncertainties else None
            with torch.cuda.device(xd.device):
                ctx.use_torch_stream()
                try:
                    ctx.nls_fit_dev(xd.data_ptr(), nbuf, R, int(ndata), w0, [init_a, init_m, 0.0, init_psi], chunks, opts,
                                    rows_d.data_ptr(), cov_ptr=cov_d.data_ptr() if uncertainties else None)
                finally:
                    ctx.use_default_stream()
            return rows_to_frame(rows_d.cpu().numpy(), cov_d.cpu().numpy() if uncertainties else None)
        x = _record_values(main_raw)[: nbuf * R]  # the reference's reshape(-1, R) raises on a ragged tail (Q7)
        ctx = _lib.get_context(device)
        cov = np.empty((nbuf, _lib.COV_STRIDE), dtype=np.float64) if uncertainties else None
        rows = ctx.nls_fit_host(x, R, int(ndata), w0, [init_a, init_m, 0.0, init_psi], seeded=chunks, opts=opts, cov_out=cov)
        return rows_to_frame(rows, cov)


class EKFFitter(BaseFitter):
    """Time-domain 5-state EKF (fitters.py:210-320): one thread per channel, sequential in time."""

    def fit(self, main_raw, **kwargs) -> pd.DataFrame:
        if kwargs.get("uncertainties", False):
            # the filter's covariance P is not a per-buffer parameter covariance (its update is deferred inside the
            # hot loop); only the NLS readout reports uncertainties
            raise ValueError("uncertainties=True is supported by the NLS fitter only, not by the EKF")
        n = self.config["n"]
        opts = _lib.default_ekf_opts()
        opts.init[0] = kwargs.get("init_a", 1.6)
        opts.init[1] = kwargs.get("init_m", 6.0)
        opts.init[2] = kwargs.get("init_phi", 0.0)
        opts.init[3] = kwargs.get("init_psi", 0.0)
        p0 = kwargs.get("P0_diag", [1.0] * 5)
        q = kwargs.get("Q_diag", [1e-8, 1e-8, 1e-6, 1e-6, 1e-8])
        if len(p0) != 5 or len(q) != 5:
            raise ValueError("P0_diag and Q_diag must have 5 entries")
        for i in range(5):
            opts.p0_diag[i] = float(p0[i])
            opts.q_diag[i] = float(q[i])
        r_val = kwargs.get("R_val", None)
        opts.r_val = float("nan") if r_val is None else float(r_val)  # NaN -> var(record), fitters.py:256
        device = kwargs.get("device", 0)

        R, _, nbuf = _calculate_fit_params(main_raw, n)
        zd = _device_record(main_raw)
        if zd is not None:
            import torch
            ctx = _lib.get_context(zd.device.index)
            rows_d = torch.empty((nbuf, _lib.ROW_STRIDE), dtype=torch.float64, device=zd.device)
            with torch.cuda.device(zd.device):
                ctx.use_torch_stream()
                try:
                    T = int(zd.shape[0])
                    ctx.ekf_dev(zd.data_ptr(), T, 1, 1, T, R, float(main_raw.f_samp), float(main_raw.f_mod), opts,
                                rows_d.data_ptr())
                finally:
                    ctx.use_default_stream()
            return rows_to_frame(rows_d.cpu().numpy())
        z = _record_values(main_raw, column="ch0")  # the reference reads column "ch0" by name (fitters.py:238)
        ctx = _lib.get_context(device)
        rows = ctx.ekf_host(z[None, :], R, main_raw.f_samp, main_raw.f_mod, opts)[0]
        return rows_to_frame(rows)


# ------------------------------------------------------------------------------------------------------
# additive batch API
# ------------------------------------------------------------------------------------------------------
def nls_fit_batch(x, f_samp, f_mod, n, ndata=10, init_a=1.6, init_m=6.0, init_psi=0.0, seeded=True, device=0,
                  tunables_from=None, return_tensor=False, time_major=False, return_cov=False):
    """NLS readout of C channel records in one pass.

    x: ``[C, T]`` float64 -- a numpy array (copied to the GPU) or a CUDA torch tensor (used in place).
    time_major: x is ``[T, C]`` (interleaved channels, what acquisition hardware and the DFMSWPM text format produce);
    it is brought to channel-major on the device by the ingest transpose (one extra read + write pass) first.
    init_m (and init_a, init_psi) may be scalars or length-C arrays (per-channel cold starts, the CRLB
    sweep recipe of workers.py:167-173 with ``seeded=False`` and one buffer per realisation).
    seeded: False -> independent cold starts; True -> every buffer from its channel's buffer 0; an int k ->
    the reference's k-chunk chain schedule per channel (1 = ``parallel=False``).
    Returns rows ``[C, nbuf, 8]`` = amp, m, phi, psi, dc, ssq, fitok, accepted LM steps.
    return_cov: return ``(rows, cov)`` with the covariance rows ``[C, nbuf, 8]`` = C_aa, C_am, C_aphi, C_mm, C_mphi,
    C_phiphi, C_psipsi, s^2 of every buffer (``dfk_lm_cov``), of the same kind as rows.
    """
    import torch
    ctx = _lib.get_context(device)
    dev = torch.device("cuda", device)
    xt = x if isinstance(x, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(x, dtype=np.float64))
    if xt.dim() == 1:
        xt = xt[None, :]
    if xt.dtype != torch.float64:
        raise TypeError("records must be float64")
    xt = xt.to(dev, non_blocking=False).contiguous()
    native_tm = False
    if time_major:
        T_, C_ = xt.shape
        R_ = int(f_samp / f_mod * n)
        # the interleaved record folds in place when its geometry allows (whole even period x channels, whole periods
        # per buffer); otherwise it is transposed once on the device and takes the channel-major path
        native_tm = C_ > 0 and T_ >= R_ > 0 and _lib.demod_path(R_, 2.0 * np.pi * f_mod / f_samp) == 1 and \
            R_ * C_ < 2 ** 31 and not (xt.data_ptr() & 15)
        if not native_tm:
            xc = torch.empty((C_, T_), dtype=torch.float64, device=dev)
            with torch.cuda.device(dev):
                ctx.use_torch_stream()
                try:
                    ctx.widen_dev(xt.data_ptr(), "float64", T_, C_, True, xc.data_ptr(), max(T_, 1))
                finally:
                    ctx.use_default_stream()
            xt = xc
    C, T = (xt.shape[1], xt.shape[0]) if native_tm else xt.shape
    R = int(f_samp / f_mod * n)
    bpc = T // R
    w0 = 2.0 * np.pi * f_mod / f_samp
    rows = torch.empty((C, bpc, _lib.ROW_STRIDE), dtype=torch.float64, device=dev)
    cov = torch.empty((C, bpc, _lib.COV_STRIDE), dtype=torch.float64, device=dev) if return_cov else None
    cov_ptr = cov.data_ptr() if return_cov and C * bpc > 0 else None

    def result():
        out = [t if return_tensor else t.cpu().numpy() for t in ((rows, cov) if return_cov else (rows,))]
        return tuple(out) if return_cov else out[0]

    if C * bpc == 0:
        return result()
    per_channel = any(np.ndim(v) > 0 for v in (init_a, init_m, init_psi))
    init_dev_ptr, init_stride, init = None, 0, [float(np.ravel(init_a)[0]), float(np.ravel(init_m)[0]), 0.0,
                                                  float(np.ravel(init_psi)[0])]
    keep = None
    if per_channel:
        g = np.zeros((C, 4))
        g[:, 0] = init_a
        g[:, 1] = init_m
        g[:, 3] = init_psi
        keep = torch.from_numpy(g).to(dev)
        init_dev_ptr, init_stride = keep.data_ptr(), 4
    with torch.cuda.device(dev):
        ctx.use_torch_stream()
        try:
            if native_tm:
                try:
                    ctx.nls_fit_batch_tm_dev(xt.data_ptr(), C, bpc, R, int(ndata), w0, init, init_dev_ptr, init_stride,
                                             seeded, fit_tunables.current_lm_opts(tunables_from), rows.data_ptr(),
                                             cov_ptr=cov_ptr)
                except RuntimeError:  # a geometry the fold cannot take after all: transpose and go channel-major
                    xc = torch.empty((C, T), dtype=torch.float64, device=dev)
                    ctx.widen_dev(xt.data_ptr(), "float64", T, C, True, xc.data_ptr(), max(T, 1))
                    xt, native_tm = xc, False
            if not native_tm:
                ctx.nls_fit_batch_dev(xt.data_ptr(), C, bpc, T, R, int(ndata), w0, init, init_dev_ptr, init_stride, seeded,
                                      fit_tunables.current_lm_opts(tunables_from), rows.data_ptr(), cov_ptr=cov_ptr)
        finally:
            ctx.use_default_stream()
        torch.cuda.current_stream(dev).synchronize()
    del keep
    return result()


def ekf_fit_batch(z, f_samp, f_mod, n, time_major=False, device=0, return_tensor=False, **kwargs):
    """EKF over C channels at once. z: ``[C, T]`` (or ``[T, C]`` with time_major=True), numpy or CUDA tensor.

    kwargs as EKFFitter.fit (init_a, init_m, init_phi, init_psi, P0_diag, Q_diag, R_val).  Returns rows [C, nbuf, 8].
    """
    import torch
    ctx = _lib.get_context(device)
    dev = torch.device("cuda", device)
    zt = z if isinstance(z, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(z, dtype=np.float64))
    if zt.dim() == 1:
        zt = zt[None, :]
    zt = zt.to(dev).contiguous()
    if time_major:
        T, C = zt.shape
        ld_t, ld_c = C, 1
    else:
        C, T = zt.shape
        ld_t, ld_c = 1, T
    R = int(f_samp / f_mod * n)
    nbuf = T // R
    opts = _lib.default_ekf_opts()
    for i, key in enumerate(("init_a", "init_m", "init_phi", "init_psi")):
        if key in kwargs:
            opts.init[i] = float(kwargs[key])
    for i in range(5):
        if "P0_diag" in kwargs:
            opts.p0_diag[i] = float(kwargs["P0_diag"][i])
        if "Q_diag" in kwargs:
            opts.q_diag[i] = float(kwargs["Q_diag"][i])
    if kwargs.get("R_val") is not None:
        opts.r_val = float(kwargs["R_val"])
    rows = torch.empty((C, nbuf, _lib.ROW_STRIDE), dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        ctx.use_torch_stream()
        try:
            ctx.ekf_dev(zt.data_ptr(), T, C, ld_t, ld_c, R, float(f_samp), float(f_mod), opts, rows.data_ptr())
        finally:
            ctx.use_default_stream()
        torch.cuda.current_stream(dev).synchronize()
    return rows if return_tensor else rows.cpu().numpy()
