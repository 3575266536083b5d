"""Cross-spectral estimate on the LPSD plan: CSD, coherence and transfer function between series (``lcsd``).

CPU part: ``ref_lcsd``, the CPU reference built on the LPSD oracle's plan, segments, detrending and window: its
self-consistency (a series against itself or a scaled copy, single-segment rows) and physics on
white noise (the phase of a delay, the response of a short FIR filter, the coherence of independent noise), and the
argument checks that need no device.  GPU part (-m gpu): the CUDA kernels through the C ABI against ``ref_lcsd`` on the
option sets of the LPSD tests, the auto terms against ``lpsd``, the CTA and strided paths, determinism, launch count,
errors and the façade's ``calc_csd``.  Gates: densities within 1e-10 of the reference relative to sqrt(Sxx Syy) (fp64
throughout, the segment sums reordered), auto terms within 1e-13 of ``lpsd``'s psd (the same projections, summed per
segment rather than per group of eight).
"""
import numpy as np
import pytest

from oracle import post_oracle as po

SPEC_TOL = 1e-10
# the option sets of test_post.py::test_lpsd_matches_oracle
OPTION_SETS = [dict(), dict(order=-1), dict(order=1), dict(order=2), dict(win="hann", olap=0.5),
               dict(Jdes=60, Kdes=20, bmin=2.0, Lmin=32), dict(psll=120, olap=0.6)]


def _series(seed, n, fs):
    rng = np.random.RandomState(seed)
    t = np.arange(n) / fs
    return 0.7 + 1e-3 * np.cumsum(rng.randn(n)) + 0.05 * rng.randn(n) + 0.2 * np.sin(2 * np.pi * 0.123 * fs * t / 10)


def _pairs(n, fs, cx=2, cy=3):
    """x [cx, n], y [cy, n]: every y shares part of x[0], so the coherence is neither 0 nor 1."""
    xs = np.stack([_series(10 + a, n, fs) for a in range(cx)])
    ys = np.stack([0.5 * (b + 1) * xs[0] + _series(20 + b, n, fs) for b in range(cy)])
    return xs, ys


def ref_lcsd(x, y, fs, olap="default", bmin=1, Lmin=0, Jdes=500, Kdes=100, order=0, win="kaiser", psll=200.0):
    """CPU reference of the log-frequency cross-spectral estimate of x against y (LTPDA's log-frequency CSD / TF /
    coherence on the plan of ``po.lpsd``): the same plan, segment starts, detrending and window as ``po.lpsd``, its loop
    run on several series at once.

    For frequency row j and segment s of series u, A_{u,s} = sum_n w_n v_n e^{+i p_j n} is the detrended, windowed
    projection ``lpsd`` forms (the complex conjugate of the usual DFT X).  Then
        Sxy[a,b,j] = 2 / (fs S2_j) * (1 / K_j) * sum_s A_{x_a,s} conj(A_{y_b,s})
    is the one-sided CSD in scipy's convention, E[conj(X) Y]; Sxx, Syy are the same sum on one series -- bit for bit
    the ``psd`` of ``lpsd``.  Coherence coh = |Sxy|^2 / (Sxx Syy) (NaN where the denominator is 0; 1 to rounding where
    K_j = 1); transfer function (H1, the response of y to x) tf = Sxy / Sxx (NaN where Sxx is 0).  If y(t) = x(t - tau),
    arg tf = -2 pi f tau.

    x is [N] or [Cx, N], y is [N] or [Cy, N].  Returns a dict f, Sxx [Cx, nf], Syy [Cy, nf], Sxy, coh, tf [Cx, Cy, nf],
    enbw, K; a 1-D input drops its axis."""
    x = np.asarray(x, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    x1, y1 = x.ndim == 1, y.ndim == 1
    xs, ys = np.atleast_2d(x), np.atleast_2d(y)
    if xs.shape[1] != ys.shape[1]:
        raise ValueError("x and y must have the same length")
    ndata = xs.shape[1]
    series = np.concatenate([xs, ys])
    cx, cy = len(xs), len(ys)
    if olap == "default" or olap is None:
        olap = po.default_overlap(win, psll)
    f, r, m, L, K = po.ltf_plan(ndata, fs, olap, bmin, Lmin, Jdes, Kdes)
    nf = len(f)
    auto = np.zeros((cx + cy, nf))
    sxy = np.zeros((cx, cy, nf), dtype=np.complex128)
    enbw = np.zeros(nf)
    cache = {}
    for j in range(nf):
        l = int(L[j])
        if l not in cache:
            cache[l] = po.window(win, l, psll)
        w = cache[l]
        c = w * np.exp(2j * np.pi * m[j] / l * np.arange(l))
        tot = [0.0] * (cx + cy)
        cre = [[0.0] * cy for _ in range(cx)]
        cim = [[0.0] * cy for _ in range(cx)]
        for s in po.segment_starts(ndata, l, int(K[j])):
            a = [np.dot(c, po.detrend(series[u, s:s + l], order)) for u in range(cx + cy)]
            for u in range(cx + cy):
                tot[u] += a[u].real * a[u].real + a[u].imag * a[u].imag  # the sum lpsd forms
            for p in range(cx):
                for q in range(cy):
                    ar, ai, br, bi = a[p].real, a[p].imag, a[cx + q].real, a[cx + q].imag
                    cre[p][q] += ar * br + ai * bi
                    cim[p][q] += ai * br - ar * bi
        s2 = (w * w).sum()
        for u in range(cx + cy):
            auto[u, j] = 2.0 * (tot[u] / K[j]) / (fs * s2)
        for p in range(cx):
            for q in range(cy):
                sxy[p, q, j] = complex(2.0 * (cre[p][q] / K[j]) / (fs * s2), 2.0 * (cim[p][q] / K[j]) / (fs * s2))
        enbw[j] = fs * s2 / (w.sum() * w.sum())
    sxx, syy = auto[:cx], auto[cx:]
    den = sxx[:, None, :] * syy[None, :, :]
    coh = np.full(sxy.shape, np.nan)
    np.divide(np.abs(sxy) ** 2, den, out=coh, where=den != 0)
    tf = np.full(sxy.shape, np.nan + 1j * np.nan)
    np.divide(sxy, np.broadcast_to(sxx[:, None, :], sxy.shape), out=tf, where=sxx[:, None, :] != 0)
    if x1:
        sxx, sxy, coh, tf = sxx[0], sxy[0], coh[0], tf[0]
    if y1:
        syy, sxy, coh, tf = syy[0], sxy[..., 0, :], coh[..., 0, :], tf[..., 0, :]
    return {"f": f, "Sxx": sxx, "Syy": syy, "Sxy": sxy, "coh": coh, "tf": tf, "enbw": enbw, "K": K}


def _white(seed, n):
    return np.random.RandomState(seed).randn(n)


def _delayed(x, d):
    return np.concatenate([np.zeros(d), x[:-d]])


def _fir(x, h):
    return np.convolve(x, h)[:len(x)]


def _fir_response(h, f, fs):
    return np.polyval(np.asarray(h)[::-1], np.exp(-2j * np.pi * f / fs))


def _plan_L(n, fs, **kw):
    olap = kw.get("olap", po.default_overlap(kw.get("win", "kaiser"), kw.get("psll", 200.0)))
    return po.ltf_plan(n, fs, olap, kw.get("bmin", 1), kw.get("Lmin", 0), kw.get("Jdes", 500), kw.get("Kdes", 100))[3]


def _check_delay(out, n, fs, d, Jdes):
    """arg tf = -2 pi f d / fs where segments are long against the delay."""
    L = _plan_L(n, fs, Jdes=Jdes)
    sel = L >= 50 * d
    assert sel.sum() >= 20
    err = np.angle(out["tf"][sel] * np.exp(2j * np.pi * out["f"][sel] * d / fs))
    assert np.max(np.abs(err)) < 0.05


def _check_fir(out, h, fs):
    assert np.max(np.abs(out["tf"] - _fir_response(h, out["f"], fs))) < 0.05


def _check_independent(out, navs):
    sel = navs >= 100
    assert sel.sum() >= 20
    assert np.mean(out["coh"][sel]) < 0.02 and np.max(out["coh"][sel]) < 0.1


# ---------------------------------------------------------------------------------------------------------- CPU
def test_oracle_series_against_itself_and_a_scaled_copy():
    N, fs = 20000, 50.0
    x = _series(1, N, fs)
    out = ref_lcsd(x, x, fs, Jdes=120)
    f, _, psd, enbw, K = po.lpsd(x, fs, Jdes=120)
    assert np.array_equal(out["f"], f) and np.array_equal(out["K"], K) and np.array_equal(out["enbw"], enbw)
    assert np.array_equal(out["Sxx"], psd) and np.array_equal(out["Syy"], psd)
    assert np.array_equal(out["Sxy"].real, out["Sxx"]) and np.all(out["Sxy"].imag == 0)
    assert np.max(np.abs(out["coh"] - 1)) < 1e-12 and np.max(np.abs(out["tf"] - 1)) < 1e-14
    g = -2.5
    out = ref_lcsd(x, g * x, fs, Jdes=120)
    assert np.max(np.abs(out["tf"] / g - 1)) < 1e-12 and np.max(np.abs(out["coh"] - 1)) < 1e-12
    # batches: [Cx, N] against [Cy, N] is every pair of the 1-D estimates
    xs, ys = _pairs(3000, fs)
    full = ref_lcsd(xs, ys, fs, Jdes=60)
    assert full["Sxy"].shape == (2, 3, len(full["f"])) and full["Sxx"].shape == (2, len(full["f"]))
    one = ref_lcsd(xs[1], ys[2], fs, Jdes=60)
    assert one["Sxy"].shape == (len(full["f"]),)
    for k in ("Sxy", "coh", "tf"):
        assert np.array_equal(one[k], full[k][1, 2])
    with pytest.raises(ValueError):
        ref_lcsd(x, x[:-1], fs)


def test_oracle_single_segment_rows_are_fully_coherent():
    """With K = 1 the estimate has one segment: coherence 1 whatever the data."""
    N, fs = 20000, 50.0
    out = ref_lcsd(_white(1, N), _white(2, N), fs, Jdes=120)
    one = out["K"] == 1
    assert one.sum() >= 1
    assert np.max(np.abs(out["coh"][one] - 1)) < 1e-12


def test_oracle_delay_fir_and_independent_noise():
    N, fs, J = 20000, 50.0, 120
    x = _white(3, N)
    _check_delay(ref_lcsd(x, _delayed(x, 3), fs, Jdes=J), N, fs, 3, J)
    h = [0.5, 0.3, -0.2]
    _check_fir(ref_lcsd(x, _fir(x, h), fs, Jdes=J), h, fs)
    out = ref_lcsd(x, _white(4, N), fs, Jdes=J)
    _check_independent(out, out["K"])


def test_argument_errors_need_no_device():
    from deepfmkit_b200 import DeepFitObject, lcsd
    with pytest.raises(ValueError):
        lcsd(np.zeros(100), np.zeros(101), 1.0)
    with pytest.raises(ValueError):
        lcsd(np.zeros((2, 100)), np.zeros((3, 99)), 1.0)
    a, b = DeepFitObject(), DeepFitObject()
    a.fs, b.fs = 50.0, 25.0
    a.phi, b.phi = np.zeros(100), np.zeros(100)
    with pytest.raises(ValueError):
        a.calc_csd(b)
    b.fs, b.phi = 50.0, np.zeros(99)
    with pytest.raises(ValueError):
        a.calc_csd(b)


def test_entry_is_declared_and_bound():
    from deepfmkit_b200 import _lib
    assert "dfk_lcsd_dev" in _lib.SYMBOLS and _lib.ABI_VERSION == 6
    assert len(_lib.SYMBOLS["dfk_lcsd_dev"][1]) == 19


# ---------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def torch_mod():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _assert_matches_oracle(got, ref):
    assert np.array_equal(got["f"], ref["f"]) and np.array_equal(got["navs"], ref["K"])
    assert np.max(np.abs(got["Sxx"] / ref["Sxx"] - 1)) < SPEC_TOL
    assert np.max(np.abs(got["Syy"] / ref["Syy"] - 1)) < SPEC_TOL
    scale = np.sqrt(ref["Sxx"][:, None, :] * ref["Syy"][None, :, :])
    assert np.all(np.abs(got["Sxy"] - ref["Sxy"]) <= SPEC_TOL * scale)
    assert np.max(np.abs(got["coh"] - ref["coh"])) <= SPEC_TOL
    assert np.all(np.abs(got["tf"] - ref["tf"]) <= SPEC_TOL * np.sqrt(ref["Syy"][None, :, :] / ref["Sxx"][:, None, :]))
    assert np.max(np.abs(got["enbw"] / ref["enbw"] - 1)) < 1e-12


@pytest.mark.gpu
@pytest.mark.parametrize("kw", OPTION_SETS)
def test_lcsd_matches_oracle(torch_mod, kw):
    from deepfmkit_b200 import lcsd, lpsd
    N, fs = 6000, 50.0
    xs, ys = _pairs(N, fs)
    okw = dict(Jdes=120)
    okw.update(kw)
    got = lcsd(xs, ys, fs, **okw)
    assert got["Sxy"].dtype == np.complex128 and got["Sxy"].shape == (2, 3, len(got["f"]))
    _assert_matches_oracle(got, ref_lcsd(xs, ys, fs, **okw))
    # the auto terms are lpsd's psd of the same series
    for series, auto in ((xs, got["Sxx"]), (ys, got["Syy"])):
        psd = lpsd(series, fs, return_type="dict", **okw)["psd"]
        assert np.max(np.abs(auto / psd - 1)) < 1e-13


@pytest.mark.gpu
def test_lcsd_long_segments_strided_tensors_and_determinism(torch_mod):
    """CTA-per-group path (L >= 2048); a column of a row table read in place (stride 8); CUDA tensors and numpy give
    the same bits; a repeated call gives the same bits; exactly two launches per call."""
    from deepfmkit_b200 import _lib, lcsd, lpsd
    torch = torch_mod
    N, fs, J, K = 40000, 50.0, 40, 8
    xs, ys = _pairs(N, fs, cx=2, cy=1)
    opts = _lib.default_lpsd_opts()
    opts.jdes, opts.kdes = J, K
    assert int(np.max(_lib.lpsd_plan(N, fs, opts)["L"])) >= 2048
    got = lcsd(xs, ys, fs, Jdes=J, Kdes=K)
    _assert_matches_oracle(got, ref_lcsd(xs, ys, fs, Jdes=J, Kdes=K))
    psd = lpsd(xs, fs, Jdes=J, Kdes=K, return_type="dict")["psd"]
    assert np.max(np.abs(got["Sxx"] / psd - 1)) < 1e-13

    ctx = _lib.get_context(0)
    xd, yd = torch.from_numpy(xs).cuda(), torch.from_numpy(ys).cuda()
    on_dev = lcsd(xd, yd, fs, Jdes=J, Kdes=K)
    again = lcsd(xd, yd, fs, Jdes=J, Kdes=K)
    for k in ("f", "Sxx", "Syy", "Sxy", "coh", "tf", "enbw", "navs"):
        assert np.array_equal(on_dev[k], got[k], equal_nan=True), k
        assert np.array_equal(again[k], got[k], equal_nan=True), k

    # x[1] and y[0] as columns 2 and 5 of a [N, 8] row table, read in place
    rows = torch.zeros((N, 8), dtype=torch.float64, device="cuda")
    rows[:, 2] = xd[1]
    rows[:, 5] = yd[0]
    torch.cuda.synchronize()
    n0 = ctx.launch_count()
    col = ctx.lcsd_dev(rows.data_ptr() + 2 * 8, 1, 0, rows.data_ptr() + 5 * 8, 1, 0, N, 8, fs, opts)
    assert ctx.launch_count() - n0 == 2
    ref = lcsd(xs[1], ys[0], fs, Jdes=J, Kdes=K)
    assert np.array_equal(col["Sxx"][0], ref["Sxx"]) and np.array_equal(col["Syy"][0], ref["Syy"])
    assert np.array_equal(col["Sxy"][0, 0], ref["Sxy"])


@pytest.mark.gpu
def test_lcsd_physics_on_device(torch_mod):
    from deepfmkit_b200 import lcsd
    N, fs, J = 20000, 50.0, 120
    x = _white(3, N)
    _check_delay(lcsd(x, _delayed(x, 3), fs, Jdes=J), N, fs, 3, J)
    h = [0.5, 0.3, -0.2]
    _check_fir(lcsd(x, _fir(x, h), fs, Jdes=J), h, fs)
    out = lcsd(x, _white(4, N), fs, Jdes=J)
    _check_independent(out, out["navs"])
    # a series against itself: Sxy real and equal to Sxx, coherence and transfer function 1
    out = lcsd(x, x, fs, Jdes=J)
    assert np.array_equal(out["Sxy"].real, out["Sxx"]) and np.all(out["Sxy"].imag == 0)
    assert np.array_equal(out["Sxx"], out["Syy"])
    assert np.max(np.abs(out["coh"] - 1)) < 1e-12 and np.max(np.abs(out["tf"] - 1)) < 1e-14


@pytest.mark.gpu
def test_lcsd_errors_and_null_outputs(torch_mod):
    import ctypes
    from deepfmkit_b200 import _lib, lcsd
    torch = torch_mod
    N, fs = 3000, 50.0
    x = torch.from_numpy(_white(1, N)).cuda()
    with pytest.raises(ValueError):
        lcsd(x, x[:-1], fs)
    ctx = _lib.get_context(0)
    opts = _lib.default_lpsd_opts()
    p = x.data_ptr()
    with pytest.raises(RuntimeError, match="dfk_b200 error -1"):
        ctx.lcsd_dev(p, 0, N, p, 1, N, N, 1, fs, opts)
    with pytest.raises(RuntimeError, match="dfk_b200 error -1"):
        ctx.lcsd_dev(p, 1, N, p, 1, N, N, 0, fs, opts)
    lib = ctx.lib
    nf = ctypes.c_int32()
    cap = len(_lib.lpsd_plan(N, fs, opts)["f"])
    rc = lib.dfk_lcsd_dev(ctx._h, p, 1, N, p, 1, N, N, 1, fs, ctypes.byref(opts), cap - 1, ctypes.byref(nf),
                          None, None, None, None, None, None)
    assert rc == -1 and nf.value == cap  # DFK_ERR_ARG
    # every output may be NULL
    n0 = ctx.launch_count()
    rc = lib.dfk_lcsd_dev(ctx._h, p, 1, N, p, 1, N, N, 1, fs, ctypes.byref(opts), cap, ctypes.byref(nf),
                          None, None, None, None, None, None)
    assert rc == 0 and nf.value == cap and ctx.launch_count() - n0 == 2


@pytest.mark.gpu
def test_facade_calc_csd(torch_mod):
    """Two fitted channels through the façade: calc_csd is lcsd on their phases with the first fit's settings."""
    from deepfmkit_b200 import DeepFitFramework, DeepRawObject, lcsd
    from oracle import dfmi_oracle as orc
    dff = DeepFitFramework()
    fits = {}
    for label, seed in (("a", 4), ("b", 5)):
        x = orc.snr_signal(6.0, 200e3, 1000.0, 2.0, 40.0, seed=seed)
        dff.load_raw_object(DeepRawObject(data=x, f_samp=200e3, f_mod=1000.0, label=label))
        fits[label] = dff.fit(label, n=4)
    a, b = fits["a"], fits["b"]
    assert a.phi is not None and len(a.phi) == len(b.phi)
    a.Jdes, a.Kdes, a.order = 80, 30, 1  # settings are the calling object's
    got = a.calc_csd(b)
    ref = lcsd(a.phi, b.phi, a.fs, a.olap, a.bmin, a.Lmin, 80, 30, 1, a.win, a.psll)
    assert set(got) == {"f", "Sxx", "Syy", "Sxy", "coh", "tf", "enbw", "navs"}
    for k in got:
        assert np.array_equal(got[k], ref[k], equal_nan=True), k
    assert a.f is None and a.Sxx is None  # stores nothing
    b.fs = 2 * a.fs
    with pytest.raises(ValueError):
        a.calc_csd(b)
