"""Post-fit step of the readout on the GPU (SURVEY 8f-4).

``vectorized_downsample`` keeps the name, arguments and edge behaviour of dsp.py:3-56 (block means; the ragged tail
is dropped; a bad ``R`` or a signal shorter than ``R`` gives an empty array).  ``lpsd`` takes the arguments the
reference passes to ``spectools.lpsd.lpsd`` (core.py:590-609, data.py:239-244) and returns, like its ``'legacy'``
form, a 6-tuple whose first element is the frequency vector and whose third is the one-sided power spectral density
the reference stores as ``Sxx``.  ``lcsd`` is the cross-spectral counterpart on the same frequency plan: the CSD,
coherence and transfer function between fitted channels.  ``lcsd_conditioned`` extends it to several witnesses at
once: the joint transfer functions, the conditioned (residual) PSD and the multiple coherence of each target given all
witnesses.  ``wiener_subtract`` does that subtraction in the time domain: least-squares multi-input FIR filters and
the cleaned target series.  ``stability`` (and its one-kind forms ``oadev``, ``mdev``, ``tdev``, ``ohdev``) gives the
time-domain view: overlapping Allan, modified Allan, time and Hadamard deviations against the averaging time.  All run
on the device only.
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


STABILITY_KINDS = _lib.STAB_KINDS


def _stability_counts(Nx, m):
    """Term counts [4, n_m] of each kind (STABILITY_KINDS order) at averaging factors m on Nx phase points."""
    m = np.asarray(m, dtype=np.int64)
    return np.stack([Nx - 2 * m, Nx - 3 * m + 1, Nx - 3 * m + 1, Nx - 3 * m])


def _stability_m(Nx, fs, taus, kinds):
    """The averaging factors of one call: the tau rule's m values that fall inside the range of at least one
    requested kind (those outside every range are dropped), sorted and distinct."""
    if isinstance(taus, str):
        if taus == "octave":
            m = 2 ** np.arange(int(np.floor(np.log2(Nx))) + 1, dtype=np.int64)
        elif taus == "decade":
            k = np.arange(int(np.floor(np.log10(Nx))) + 1, dtype=np.int64)
            m = (np.array([1, 2, 4], dtype=np.int64)[None, :] * 10 ** k[:, None]).ravel()
        elif taus == "all":
            m = np.arange(1, Nx + 1, dtype=np.int64)
        else:
            raise ValueError(f"taus must be 'octave', 'decade', 'all' or an array of averaging times, got {taus!r}")
    else:
        try:
            t = np.asarray(taus, dtype=np.float64)
        except (TypeError, ValueError):
            raise ValueError(f"taus must be 'octave', 'decade', 'all' or an array of averaging times, got {taus!r}")
        if t.ndim != 1 or t.size == 0 or not np.all(np.isfinite(t)) or np.any(t <= 0):
            raise ValueError("an array of taus must be a non-empty 1-D array of positive, finite averaging times")
        m = np.unique(np.clip(np.rint(t * fs), 1, Nx + 1).astype(np.int64))
    n = _stability_counts(Nx, m)[[STABILITY_KINDS.index(k) for k in kinds]]
    return m[np.max(n, axis=0) >= 1]


def _stability_series(x, device):
    """(fp64 CUDA tensor [C, N] read in place where it already is one, whether the input was 1-D, ld_c, stride)."""
    import torch
    if isinstance(x, torch.Tensor) and x.is_cuda:
        t = x if x.dtype == torch.float64 else x.to(torch.float64)
    else:
        h = np.ascontiguousarray(np.asarray(x, dtype=np.float64))
        t = torch.from_numpy(h if h.flags.writeable else h.copy()).to(torch.device("cuda", device))
    one = t.dim() == 1
    if one:
        t = t[None, :]
    if t.stride(1) < 1:  # an expanded tensor
        t = t.contiguous()
    return t, one, int(t.stride(0)), int(t.stride(1))


def stability(x, fs, kinds=STABILITY_KINDS, taus="octave", data_type="phase", device=0):
    """Time-domain stability of one series or of every row of a 2-D array / tensor on the device: the overlapping
    Allan ("oadev"), modified Allan ("mdev"), time ("tdev") and overlapping Hadamard ("ohdev") deviations against the
    averaging time tau = m / fs (NIST SP 1065; the definitions and tau rules of allantools).

    ``x`` is ``[N]`` or ``[C, N]``, a numpy array or a CUDA tensor (read in place on its device, strides included, so
    a column of a row table needs no copy).  ``data_type`` "phase": x is phase-time, Nx = N points.  "freq": x is
    fractional frequency (or any series whose averages are wanted, such as a fitted phase column), integrated as
    x_0 = 0, x_n = sum_{i<n} y_i / fs, Nx = N + 1; the deviations come out in the series' own units.

    ``taus``: "octave" (m = 1, 2, 4, ...), "decade" (m = 1, 2, 4 x 10^k), "all" (every m: O(N^2) work per series) or
    an array of averaging times in seconds (m = round(tau fs), at least 1, sorted and distinct).  m values outside the
    range of every requested kind are dropped; one inside some kind's range but not another's gives NaN and n = 0 for
    the other.  Term counts n: oadev Nx - 2m, mdev and tdev Nx - 3m + 1, ohdev Nx - 3m.

    Returns a dict of host arrays: ``taus`` and ``m`` [n_m], and per requested kind ``<kind>`` [C, n_m],
    ``<kind>_err`` [C, n_m] (the simple error dev / sqrt(n) of allantools, not an EDF confidence interval) and
    ``<kind>_n`` [n_m].  A 1-D input drops the C axis.  A NaN or infinite sample makes every deviation of its series
    NaN.  The running sums are carried in double-double, so a drifting series keeps the differences that an fp64
    cumulative sum would lose to cancellation; results are bit-identical between runs and for a series alone or in a
    batch."""
    import torch
    if isinstance(kinds, str):
        kinds = (kinds,)
    kinds = tuple(kinds)
    if not kinds or any(k not in STABILITY_KINDS for k in kinds):
        raise ValueError(f"kinds must be a non-empty selection of {STABILITY_KINDS}, got {kinds!r}")
    kinds = tuple(k for k in STABILITY_KINDS if k in kinds)
    codes = {"phase": _lib.STAB_PHASE, "freq": _lib.STAB_FREQ}
    if not isinstance(data_type, str) or data_type not in codes:
        raise ValueError(f"data_type must be 'phase' or 'freq', got {data_type!r}")
    if isinstance(fs, bool) or not np.isscalar(fs) or not np.isfinite(fs) or fs <= 0:
        raise ValueError(f"fs must be positive and finite, got {fs!r}")
    shape = tuple(x.shape) if hasattr(x, "shape") else np.shape(x)
    if len(shape) not in (1, 2) or (len(shape) == 2 and shape[0] < 1):
        raise ValueError(f"expected a series [N] or a batch of series [C, N], got shape {shape}")
    N = shape[-1]
    Nx = N + (data_type == "freq")
    if Nx < 3:
        raise ValueError(f"{N} samples give {Nx} phase points: at least 3 are needed")
    m = _stability_m(Nx, float(fs), taus, kinds)
    if m.size == 0:
        raise ValueError(f"{N} samples are too short for any requested averaging factor of {kinds}")
    if isinstance(x, torch.Tensor) and x.is_cuda:
        device = x.device.index
    t, one, ld_c, stride = _stability_series(x, device)
    mask = sum(_lib.STAB_BITS[k] for k in kinds)
    ctx = _lib.get_context(device)
    with torch.cuda.device(t.device):
        ctx.use_torch_stream()
        try:
            dev, n = ctx.stability_dev(t.data_ptr(), N, stride, t.shape[0], ld_c, float(fs), codes[data_type], mask, m)
        finally:
            ctx.use_default_stream()
    out = {"taus": m / float(fs), "m": m}
    for k in kinds:
        i = STABILITY_KINDS.index(k)
        err = np.full(dev[i].shape, np.nan)
        np.divide(dev[i], np.sqrt(n[i].astype(np.float64)), out=err, where=n[i] > 0)
        out[k], out[k + "_err"] = (dev[i][0], err[0]) if one else (dev[i], err)
        out[k + "_n"] = n[i]
    return out


def _one_kind(kind, data, rate, data_type, taus):
    out = stability(data, rate, kinds=(kind,), taus="octave" if taus is None else taus, data_type=data_type)
    return out["taus"], out[kind], out[kind + "_err"], out[kind + "_n"]


def oadev(data, rate=1.0, data_type="phase", taus=None):
    """Overlapping Allan deviation with allantools' interface: ``(taus, dev, err, n)``; see ``stability``."""
    return _one_kind("oadev", data, rate, data_type, taus)


def mdev(data, rate=1.0, data_type="phase", taus=None):
    """Modified Allan deviation with allantools' interface: ``(taus, dev, err, n)``; see ``stability``."""
    return _one_kind("mdev", data, rate, data_type, taus)


def tdev(data, rate=1.0, data_type="phase", taus=None):
    """Time deviation, tau mdev / sqrt(3), with allantools' interface: ``(taus, dev, err, n)``; see ``stability``."""
    return _one_kind("tdev", data, rate, data_type, taus)


def ohdev(data, rate=1.0, data_type="phase", taus=None):
    """Overlapping Hadamard deviation with allantools' interface: ``(taus, dev, err, n)``; see ``stability``."""
    return _one_kind("ohdev", data, rate, data_type, taus)
