"""Post-fit step of the readout on the GPU (SURVEY 8f-4).

``vectorized_downsample`` keeps the name, arguments and edge behaviour of dsp.py:3-56 (block means; the ragged tail
is dropped; a bad ``R`` or a signal shorter than ``R`` gives an empty array).  ``lpsd`` takes the arguments the
reference passes to ``spectools.lpsd.lpsd`` (core.py:590-609, data.py:239-244) and returns, like its ``'legacy'``
form, a 6-tuple whose first element is the frequency vector and whose third is the one-sided power spectral density
the reference stores as ``Sxx``.  ``lcsd`` is the cross-spectral counterpart on the same frequency plan: the CSD,
coherence and transfer function between fitted channels.  ``lcsd_conditioned`` extends it to several witnesses at
once: the joint transfer functions, the conditioned (residual) PSD and the multiple coherence of each target given all
witnesses.  ``wiener_subtract`` does that subtraction in the time domain: least-squares multi-input FIR filters and
the cleaned target series.  All run on the device only.
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


MAX_WITNESSES = 64  # the witness matrix of one frequency is factored in one CTA's shared memory


def lcsd_conditioned(witnesses, targets, fs, olap="default", bmin=1, Lmin=0, Jdes=500, Kdes=100, order=0,
                     win=np.kaiser, psll=200, device=0):
    """Conditioned spectra of ``targets`` given ``witnesses`` on the plan ``lpsd`` uses with the same settings: the
    multiple-input / single-output analysis (Bendat & Piersol, *Random Data*, ch. 7).  It answers how much of each
    target the witnesses explain together and what is left after the best linear subtraction of all of them, without
    counting noise that several witnesses share more than once (as pairwise coherence does).

    ``witnesses`` is ``[N]`` or ``[Cx, N]`` with 1 <= Cx <= 64, ``targets`` is ``[N]`` or ``[Cy, N]``; numpy arrays or
    CUDA tensors, handled as by ``lcsd``.  With the segment projections A of ``lcsd`` and c_j = 2 / (fs S2_j K_j),
    sums over the K_j segments of frequency row j, the result is a dict of host arrays:

    - ``f``, ``enbw``, ``navs`` [nf]: as ``lcsd``;
    - ``Sxx`` [Cx, Cx, nf] complex: c_j sum A_{x_a} conj(A_{x_b}), the Hermitian witness matrix; its diagonal is
      ``lpsd``'s psd and entry (a, b) is ``lcsd``'s Sxy of witness a against witness b;
    - ``Syy`` [Cy, nf]: ``lpsd``'s psd of each target;
    - ``Sxy`` [Cx, Cy, nf] complex: c_j sum A_{x_a} conj(A_{y_t}), ``lcsd``'s convention E[conj(X) Y];
    - ``H`` [Cx, Cy, nf] complex: Sxx^-1 Sxy[:, t], the joint transfer functions.  If y = sum_a h_a * x_a + n with n
      independent of the witnesses, H[a, t] estimates the response h_a(f).  For one witness it is ``lcsd``'s ``tf``;
    - ``Sres`` [Cy, nf]: Syy - Sxy[:, t]^H Sxx^-1 Sxy[:, t], the conditioned PSD: what remains of the target after the
      best linear subtraction of all witnesses (real, >= 0 up to rounding).  For one witness it is Syy (1 - coh);
    - ``mcoh`` [Cy, nf]: the multiple coherence 1 - Sres / Syy, NaN where Syy is 0.

    ``H``, ``Sres`` and ``mcoh`` are NaN on a row with fewer segments than witnesses (K_j < Cx: the estimated Sxx then
    has rank <= K_j), and on a row where the Cholesky factorisation of Sxx meets a pivot not above 1e-10 times its
    diagonal entry: a duplicated or linearly dependent witness.

    Bias: with no true coherence the expected multiple coherence is about Cx / K (K = ``navs``, fewer effective
    averages where segments overlap), and it is 1 on rows where K = Cx whatever the data.  Read it against that floor,
    as ``lcsd``'s coherence is read against 1 / K.

    The witness axis is always kept; a 1-D ``targets`` drops the Cy axis."""
    import torch
    nx, ny = (tuple(a.shape) if hasattr(a, "shape") else np.shape(a) for a in (witnesses, targets))
    if not nx or not ny or nx[-1] != ny[-1]:
        raise ValueError(f"witnesses and targets must be series of the same number of samples, got shapes {nx} and {ny}")
    Cx, Cy = (1 if len(nx) == 1 else nx[0]), (1 if len(ny) == 1 else ny[0])
    if not 1 <= Cx <= MAX_WITNESSES:
        raise ValueError(f"{Cx} witnesses: between 1 and {MAX_WITNESSES} are supported")
    if Cy < 1 or Cx + Cy > 65535:
        raise ValueError(f"{Cy} targets: at least 1, and at most 65535 series in all")
    tensors = [a for a in (witnesses, targets) if isinstance(a, torch.Tensor) and a.is_cuda]
    if tensors:
        device = tensors[0].device.index
    xt, _ = _device_rows(witnesses, device)
    yt, y1 = _device_rows(targets, device)
    if xt.device != yt.device:
        raise ValueError(f"witnesses and targets are on different devices ({xt.device}, {yt.device})")
    N = xt.shape[1]
    opts = lpsd_opts(olap, bmin, Lmin, Jdes, Kdes, order, win, psll)
    ctx = _lib.get_context(device)
    with torch.cuda.device(xt.device):
        ctx.use_torch_stream()
        try:
            out = ctx.lcsd_cond_dev(xt.data_ptr(), Cx, N, yt.data_ptr(), Cy, N, N, 1, float(fs), opts)
        finally:
            ctx.use_default_stream()
    if y1:
        out["Syy"], out["Sres"], out["mcoh"] = out["Syy"][0], out["Sres"][0], out["mcoh"][0]
        out["Sxy"], out["H"] = out["Sxy"][:, 0], out["H"][:, 0]
    return out


MAX_WIENER_UNKNOWNS = 1024  # Cx * taps: the normal matrix (8 MB) stays resident in L2 for the factorisation


def wiener_subtract(witnesses, targets, taps, lead=None, ridge=0.0, device=0):
    """Time-domain witness subtraction: the least-squares multi-input FIR (Wiener) filters that best predict each
    target from all witnesses, and the targets with that prediction subtracted, on the device.

    ``witnesses`` is ``[N]`` or ``[Cx, N]`` with 1 <= Cx <= 64, ``targets`` is ``[N]`` or ``[Cy, N]``; numpy arrays or
    CUDA tensors, handled as by ``lcsd_conditioned``.  With x~, y~ the series less their means over all N samples,
    L = ``taps``, k0 = ``lead`` (default (L - 1) // 2, a centred two-sided filter; 0 is causal), n0 = L - 1 - k0 and
    M = N - L + 1 (the rows n0 .. n0 + M - 1 on which every tap is inside the record):

    - model: yhat_t[n] = sum_a sum_k h[t, a, k] x~_a[n + k0 - k]; tap k looks ``offsets[k]`` = k0 - k samples away;
    - ``h`` [Cy, Cx, L] solves (G + lambda I) h_t = p_t, the normal equations over the M rows
      (G[(a,k),(b,l)] = sum_n x~_a[n+k0-k] x~_b[n+k0-l], p[(a,k),t] = sum_n x~_a[n+k0-k] y~_t[n]), with the diagonal
      loading lambda = ``ridge`` * trace(G) / (Cx L);
    - ``residual`` [Cy, M]: y~_t[n0 + i] - yhat_t[n0 + i]; a CUDA tensor when an input was one, numpy otherwise;
    - ``var_y``, ``var_res`` [Cy]: mean squares of y~ and of the residual over the same rows; ``explained`` [Cy]:
      1 - var_res / var_y, NaN where var_y is 0;
    - ``offsets`` [L], ``n0``, ``lead``, and ``singular``: True when a Cholesky pivot of G + lambda I is not above
      1e-10 times its diagonal entry (a duplicated or linearly dependent witness with ``ridge`` 0).  ``h``, the
      residual, ``var_res`` and ``explained`` are then NaN; ``var_y`` stays finite.

    Limits: Cx * L <= 1024 and M >= Cx * L (no underdetermined systems); Cx + Cy <= 65535.  Callers detrend beyond the
    mean themselves.  A 1-D ``targets`` drops the Cy axis."""
    import torch
    nx, ny = (tuple(a.shape) if hasattr(a, "shape") else np.shape(a) for a in (witnesses, targets))
    if len(nx) not in (1, 2) or len(ny) not in (1, 2) or nx[-1] != ny[-1]:
        raise ValueError(f"witnesses and targets must be series of the same number of samples, got shapes {nx} and {ny}")
    Cx, Cy, N = (1 if len(nx) == 1 else nx[0]), (1 if len(ny) == 1 else ny[0]), nx[-1]
    if not 1 <= Cx <= MAX_WITNESSES:
        raise ValueError(f"{Cx} witnesses: between 1 and {MAX_WITNESSES} are supported")
    if Cy < 1 or Cx + Cy > 65535:
        raise ValueError(f"{Cy} targets: at least 1, and at most 65535 series in all")
    if not isinstance(taps, (int, np.integer)) or isinstance(taps, bool) or taps < 1:
        raise ValueError(f"taps must be a positive integer, got {taps!r}")
    L = int(taps)
    if Cx * L > MAX_WIENER_UNKNOWNS:
        raise ValueError(f"{Cx} witnesses x {L} taps = {Cx * L} unknowns: at most {MAX_WIENER_UNKNOWNS}")
    if lead is None:
        lead = (L - 1) // 2
    if not isinstance(lead, (int, np.integer)) or isinstance(lead, bool) or not 0 <= lead <= L - 1:
        raise ValueError(f"lead must be an integer in 0..{L - 1}, got {lead!r}")
    lead = int(lead)
    if isinstance(ridge, bool) or not np.isscalar(ridge) or not np.isfinite(ridge) or ridge < 0:
        raise ValueError(f"ridge must be finite and >= 0, got {ridge!r}")
    M = N - L + 1
    if M < Cx * L:
        raise ValueError(f"{N} samples give {M} rows for {Cx * L} unknowns: need N >= Cx L + L - 1")
    tensors = [a for a in (witnesses, targets) if isinstance(a, torch.Tensor) and a.is_cuda]
    if tensors:
        device = tensors[0].device.index
    xt, _ = _device_rows(witnesses, device)
    yt, y1 = _device_rows(targets, device)
    if xt.device != yt.device:
        raise ValueError(f"witnesses and targets are on different devices ({xt.device}, {yt.device})")
    res = torch.empty((Cy, M), dtype=torch.float64, device=xt.device)
    ctx = _lib.get_context(device)
    with torch.cuda.device(xt.device):
        ctx.use_torch_stream()
        try:
            out = ctx.wiener_dev(xt.data_ptr(), Cx, N, yt.data_ptr(), Cy, N, N, 1, L, lead, float(ridge),
                                 res.data_ptr(), M)
        finally:
            ctx.use_default_stream()
    var_y, var_res = out["var_y"], out["var_res"]
    explained = np.full(Cy, np.nan)
    np.divide(var_res, var_y, out=explained, where=var_y != 0)
    explained = np.where(var_y != 0, 1.0 - explained, np.nan)
    result = {"h": out["h"], "offsets": lead - np.arange(L), "n0": L - 1 - lead, "lead": lead,
              "residual": res if tensors else res.cpu().numpy(), "var_y": var_y, "var_res": var_res,
              "explained": explained, "singular": out["singular"]}
    if y1:
        for k in ("h", "residual", "var_y", "var_res", "explained"):
            result[k] = result[k][0]
    return result
