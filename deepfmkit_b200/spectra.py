"""Post-fit step of the readout on the GPU (SURVEY 8f-4).

``vectorized_downsample`` keeps the name, arguments and edge behaviour of dsp.py:3-56 (block means; the ragged tail
is dropped; a bad ``R`` or a signal shorter than ``R`` gives an empty array).  ``lpsd`` takes the arguments the
reference passes to ``spectools.lpsd.lpsd`` (core.py:590-609, data.py:239-244) and returns, like its ``'legacy'``
form, a 6-tuple whose first element is the frequency vector and whose third is the one-sided power spectral density
the reference stores as ``Sxx``.  ``lcsd`` is the cross-spectral counterpart on the same frequency plan: the CSD,
coherence and transfer function between fitted channels.  All run on the device only.
"""
from __future__ import annotations

import numpy as np

from . import _lib


def _as_device_vector(signal, device):
    import torch
    if isinstance(signal, torch.Tensor) and signal.is_cuda:
        return signal.to(torch.float64).contiguous().view(-1), True
    return np.ascontiguousarray(np.asarray(signal, dtype=np.float64)).reshape(-1), False


def vectorized_downsample(signal, R, device=0):
    """Block means of ``signal`` over blocks of ``R`` samples (dsp.py:3-56).

    A numpy array (streamed through the library's staged host path) gives a numpy array; a CUDA tensor is used in
    place and gives a CUDA tensor."""
    if not isinstance(R, (int, np.integer)) or isinstance(R, bool) or R <= 0:
        print(f"Downsampling factor R must be a positive integer, but got {R}. Returning empty array.")
        return np.array([])
    R = int(R)
    x, on_device = _as_device_vector(signal, device)
    n = int(x.shape[0])
    if n // R == 0:
        return np.array([])
    ctx = _lib.get_context(x.device.index if on_device else device)
    if not on_device:
        return ctx.downsample_host(x, R)
    import torch
    out = torch.empty(n // R, dtype=torch.float64, device=x.device)
    with torch.cuda.device(x.device):
        ctx.use_torch_stream()
        try:
            ctx.downsample_dev(x.data_ptr(), n, R, out.data_ptr())
        finally:
            ctx.use_default_stream()
    return out


def _window_code(win):
    if win is None or win is np.kaiser:
        return 0
    if win is np.hanning:
        return 1
    name = str(getattr(win, "__name__", win)).lower()
    if name.startswith("kaiser"):
        return 0
    if name in ("hann", "hanning"):
        return 1
    raise ValueError(f"window {win!r} is not available on the device (kaiser, hann)")


def lpsd_opts(olap="default", bmin=1, Lmin=0, Jdes=500, Kdes=100, order=0, win=np.kaiser, psll=200):
    o = _lib.default_lpsd_opts()
    o.olap = -1.0 if (olap is None or isinstance(olap, str)) else float(olap)
    o.bmin = float(bmin)
    o.lmin = int(Lmin)
    o.jdes = int(Jdes)
    o.kdes = int(Kdes)
    o.order = int(order)
    o.window = _window_code(win)
    o.psll = float(psll)
    return o


def _device_rows(a, device):
    """[N] or [C, N] numpy array or CUDA tensor -> (contiguous fp64 CUDA tensor [C, N], whether the input was 1-D)."""
    import torch
    if isinstance(a, torch.Tensor) and a.is_cuda:
        t = a.to(torch.float64).contiguous()
    else:
        h = np.ascontiguousarray(np.asarray(a, dtype=np.float64))
        t = torch.from_numpy(h if h.flags.writeable else h.copy()).to(torch.device("cuda", device))
    if t.dim() not in (1, 2):
        raise ValueError(f"expected a series [N] or a batch of series [C, N], got shape {tuple(t.shape)}")
    return (t[None, :], True) if t.dim() == 1 else (t, False)


def lpsd(x, fs, olap="default", bmin=1, Lmin=0, Jdes=500, Kdes=100, order=0, win=np.kaiser, psll=200,
         return_type="legacy", device=0):
    """Log-frequency spectral estimate of one series (or of every row of a 2-D array / tensor).

    return_type 'legacy': ``(f, ps, psd, enbw, navs, plan)`` -- positions 0 and 2 are what the reference reads;
    'dict': the same by name.  For a 2-D input ``ps`` and ``psd`` are ``[C, nf]``."""
    import torch
    if isinstance(x, torch.Tensor) and x.is_cuda:
        device = x.device.index
    xt, one = _device_rows(x, device)
    C, N = xt.shape
    opts = lpsd_opts(olap, bmin, Lmin, Jdes, Kdes, order, win, psll)
    ctx = _lib.get_context(device)
    with torch.cuda.device(xt.device):
        ctx.use_torch_stream()
        try:
            out = ctx.lpsd_dev(xt.data_ptr(), N, 1, C, N, float(fs), opts)
        finally:
            ctx.use_default_stream()
    if one:
        out["ps"], out["psd"] = out["ps"][0], out["psd"][0]
    if return_type == "dict":
        return out
    plan = _lib.lpsd_plan(N, fs, opts)
    return out["f"], out["ps"], out["psd"], out["enbw"], out["navs"], plan


def lcsd(x, y, fs, olap="default", bmin=1, Lmin=0, Jdes=500, Kdes=100, order=0, win=np.kaiser, psll=200, device=0):
    """Log-frequency cross-spectral estimate of the series ``x`` against the series ``y`` on the plan ``lpsd`` uses
    with the same settings (same frequencies, segments, detrending and window).

    ``x`` is ``[N]`` or ``[Cx, N]``, ``y`` is ``[N]`` or ``[Cy, N]``; numpy arrays or CUDA tensors (a tensor is read in
    place on its device; numpy goes to ``device``).  Returns a dict of host arrays:

    - ``f`` [nf], ``enbw`` [nf], ``navs`` [nf] (segments averaged per frequency, K);
    - ``Sxx`` [Cx, nf], ``Syy`` [Cy, nf]: one-sided PSDs, what ``lpsd`` reports as ``psd``;
    - ``Sxy`` [Cx, Cy, nf] complex: the one-sided CSD, E[conj(X) Y] (the usual argument order of ``csd(x, y)``);
    - ``coh`` [Cx, Cy, nf]: magnitude-squared coherence |Sxy|^2 / (Sxx Syy), NaN where the denominator is 0.  Where
      ``navs`` is 1 it is 1 (to rounding) whatever the data: one segment cannot tell common from independent noise;
    - ``tf`` [Cx, Cy, nf] complex: the H1 transfer function Sxy / Sxx, the response of y to x, NaN where Sxx is 0.
      If y(t) = x(t - tau), arg tf = -2 pi f tau.

    A 1-D ``x`` drops the Cx axis and a 1-D ``y`` the Cy axis."""
    import torch
    nx, ny = (tuple(a.shape) if hasattr(a, "shape") else np.shape(a) for a in (x, y))
    if not nx or not ny or nx[-1] != ny[-1]:
        raise ValueError(f"x and y must be series of the same number of samples, got shapes {nx} and {ny}")
    tensors = [a for a in (x, y) if isinstance(a, torch.Tensor) and a.is_cuda]
    if tensors:
        device = tensors[0].device.index
    xt, x1 = _device_rows(x, device)
    yt, y1 = _device_rows(y, device)
    if xt.device != yt.device:
        raise ValueError(f"x and y are on different devices ({xt.device}, {yt.device})")
    (Cx, N), Cy = xt.shape, yt.shape[0]
    opts = lpsd_opts(olap, bmin, Lmin, Jdes, Kdes, order, win, psll)
    ctx = _lib.get_context(device)
    with torch.cuda.device(xt.device):
        ctx.use_torch_stream()
        try:
            out = ctx.lcsd_dev(xt.data_ptr(), Cx, N, yt.data_ptr(), Cy, N, N, 1, float(fs), opts)
        finally:
            ctx.use_default_stream()
    sxx, syy, sxy = out["Sxx"], out["Syy"], out["Sxy"]
    den = sxx[:, None, :] * syy[None, :, :]
    coh = np.full(sxy.shape, np.nan)
    np.divide(sxy.real ** 2 + sxy.imag ** 2, den, out=coh, where=den != 0)
    tf = np.full(sxy.shape, np.nan + 1j * np.nan)
    np.divide(sxy, np.broadcast_to(sxx[:, None, :], sxy.shape), out=tf, where=sxx[:, None, :] != 0)
    out["coh"], out["tf"] = coh, tf
    if x1:
        out["Sxx"] = sxx[0]
        for k in ("Sxy", "coh", "tf"):
            out[k] = out[k][0]
    if y1:
        out["Syy"] = syy[0]
        for k in ("Sxy", "coh", "tf"):
            out[k] = out[k][..., 0, :]
    return out
