"""Conditioned spectra on the LPSD plan (``lcsd_conditioned``): joint transfer functions, residual PSD and multiple
coherence of target series given a set of witnesses (multiple-input / single-output analysis).

CPU part: ``ref_lcsd_cond``, the CPU reference on the segments of ``ref_lcsd`` (same plan, segment starts, detrending
and window): per frequency row the Gram sums of the segment projections, then ``numpy.linalg`` solves.  Its physics
(two FIR paths and independent noise: H, Sres, mcoh), its agreement with ``ref_lcsd`` for one witness, the NaN rows
(duplicated witness, fewer segments than witnesses), and the argument checks that need no device.  GPU part (-m gpu):
the CUDA kernels through the C ABI against ``ref_lcsd_cond`` on the option sets of the LPSD tests, against ``lcsd`` on
the same series, one witness against ``lcsd``'s tf and coherence, determinism, the strided and CTA-per-group paths, the
witness limit, Cx = 8 x Cy = 256, the launch count, errors and ``calc_conditioned``.

Gates: every output within 1e-10 of the reference (the spectra relative to the scale of their entry, sqrt(S_aa S_bb);
H relative to sqrt(Syy / Sxx_aa); Sres relative to Syy; mcoh absolute), fp64 throughout with the sums reordered and a
Cholesky factorisation on the device against LU in numpy; Sxx, Sxy, Syy within 1e-12 of ``lcsd`` (the same projections
summed in another order).
"""
import numpy as np
import pytest

from oracle import post_oracle as po
from tests.test_cross_spectra import OPTION_SETS, _plan_L, ref_lcsd

SPEC_TOL = 1e-10
LCSD_TOL = 1e-12
PIVOT_TOL = 1e-10  # the device's singular-pivot threshold, relative to the diagonal of Sxx


def _detrend_rows(seg, order):
    """po.detrend on every row of seg [.., L] (least squares on the same centred basis)."""
    if order < 0:
        return seg
    if order == 0:
        return seg - seg.mean(axis=-1, keepdims=True)
    l = seg.shape[-1]
    u = np.arange(l, dtype=np.float64) - 0.5 * (l - 1)
    V = np.vander(u, order + 1)
    flat = seg.reshape(-1, l).T
    coef = np.linalg.lstsq(V, flat, rcond=None)[0]
    return (flat - V @ coef).T.reshape(seg.shape)


def ref_lcsd_cond(x, y, fs, olap="default", bmin=1, Lmin=0, Jdes=500, Kdes=100, order=0, win="kaiser", psll=200.0):
    """CPU reference of the conditioned spectra of targets y given witnesses x on the plan of ``po.lpsd``.

    For frequency row j the segments, detrending and window are those of ``ref_lcsd``; A_{u,s} = sum_n w_n v_n
    e^{+i p_j n} is the projection of segment s of series u and c_j = 2 / (fs S2_j K_j).  Then
        Sxx[a,b,j] = c_j sum_s A_{x_a,s} conj(A_{x_b,s}),  Sxy[a,t,j] = c_j sum_s A_{x_a,s} conj(A_{y_t,s}),
        Syy[t,j] = c_j sum_s |A_{y_t,s}|^2,  H[:,t,j] = Sxx^-1 Sxy[:,t],
        Sres[t,j] = Syy - Sxy[:,t]^H Sxx^-1 Sxy[:,t],  mcoh[t,j] = 1 - Sres / Syy (NaN where Syy = 0).
    H, Sres and mcoh are NaN where K_j < Cx or where a Cholesky pivot of Sxx is not above PIVOT_TOL times its
    diagonal entry.  x is [N] or [Cx, N], y is [N] or [Cy, N]; a 1-D y drops the Cy axis."""
    xs = np.atleast_2d(np.asarray(x, dtype=np.float64))
    y = np.asarray(y, dtype=np.float64)
    y1 = y.ndim == 1
    ys = np.atleast_2d(y)
    if xs.shape[1] != ys.shape[1]:
        raise ValueError("x and y must have the same length")
    ndata = xs.shape[1]
    series = np.concatenate([xs, ys])
    cx, cy = len(xs), len(ys)
    if olap == "default" or olap is None:
        olap = po.default_overlap(win, psll)
    f, r, m, L, K = po.ltf_plan(ndata, fs, olap, bmin, Lmin, Jdes, Kdes)
    nf = len(f)
    sxx = np.zeros((cx, cx, nf), dtype=np.complex128)
    sxy = np.zeros((cx, cy, nf), dtype=np.complex128)
    syy = np.zeros((cy, nf))
    h = np.full((cx, cy, nf), np.nan + 1j * np.nan)
    sres = np.full((cy, nf), np.nan)
    mcoh = np.full((cy, nf), np.nan)
    enbw = np.zeros(nf)
    for j in range(nf):
        l, k = int(L[j]), int(K[j])
        w = po.window(win, l, psll)
        c = w * np.exp(2j * np.pi * m[j] / l * np.arange(l))
        idx = po.segment_starts(ndata, l, k)[:, None] + np.arange(l)[None, :]
        A = _detrend_rows(series[:, idx], order) @ c  # [cx + cy, K]
        s2 = (w * w).sum()
        scale = 2.0 / (fs * s2 * k)
        G = A[:cx] @ A.conj().T  # [cx, cx + cy]
        sxx[:, :, j] = scale * G[:, :cx]
        sxx[range(cx), range(cx), j] = scale * np.sum(A[:cx].real ** 2 + A[:cx].imag ** 2, axis=1)
        sxy[:, :, j] = scale * G[:, cx:]
        syy[:, j] = scale * np.sum(A[cx:].real ** 2 + A[cx:].imag ** 2, axis=1)
        enbw[j] = fs * s2 / (w.sum() * w.sum())
        if k < cx:
            continue
        S = sxx[:, :, j]
        try:
            Lc = np.linalg.cholesky(S)
        except np.linalg.LinAlgError:
            continue
        if np.any(np.diag(Lc).real ** 2 <= PIVOT_TOL * np.diag(S).real):
            continue
        hj = np.linalg.solve(S, sxy[:, :, j])
        h[:, :, j] = hj
        sres[:, j] = syy[:, j] - np.sum(sxy[:, :, j].conj() * hj, axis=0).real
        with np.errstate(divide="ignore", invalid="ignore"):
            mcoh[:, j] = np.where(syy[:, j] != 0, 1.0 - sres[:, j] / syy[:, j], np.nan)
    out = {"f": f, "enbw": enbw, "K": K, "Sxx": sxx, "Syy": syy, "Sxy": sxy, "H": h, "Sres": sres, "mcoh": mcoh}
    if y1:
        for key in ("Syy", "Sres", "mcoh"):
            out[key] = out[key][0]
        for key in ("Sxy", "H"):
            out[key] = out[key][:, 0]
    return out


def _white(seed, n):
    return np.random.RandomState(seed).randn(n)


def _fir(x, h):
    return np.convolve(x, h)[:len(x)]


def _fir_response(h, f, fs):
    return np.polyval(np.asarray(h)[::-1], np.exp(-2j * np.pi * f / fs))


def _witness(seed, n):
    """A red (random-walk) plus white series with an offset, independent from seed to seed."""
    rng = np.random.RandomState(seed)
    return 0.05 * (seed % 7) + 1e-2 * np.cumsum(rng.randn(n)) + 0.5 * rng.randn(n)


def _miso(n, cx, cy, seed=0):
    """Witnesses [cx, n] and targets [cy, n]: each target a different FIR mix of every witness plus its own noise."""
    xs = np.stack([_witness(100 + seed + a, n) for a in range(cx)])
    ys = np.empty((cy, n))
    for t in range(cy):
        rng = np.random.RandomState(200 + seed + t)
        ys[t] = 0.3 * rng.randn(n)
        for a in range(cx):
            ys[t] += _fir(xs[a], rng.randn(3) / (1 + a))
    return xs, ys


# the MISO example of the issue: y = h1 * x1 + h2 * x2 + n
H1, H2, SIGMA_N = [0.5, 0.3, -0.2], [-0.4, 0.0, 0.25, 0.1], 0.3


def _two_paths(n, noise=True):
    x1, x2 = _white(11, n), _white(12, n)
    y = _fir(x1, H1) + _fir(x2, H2)
    if noise:
        y = y + SIGMA_N * _white(13, n)
    return np.stack([x1, x2]), y


def _check_residual(sres, sel, n, fs, Jdes):
    """Sres against the PSD of the white n, 2 sigma^2 / fs, on rows of K >= 100 segments of L >= 100 samples: each row
    within 20 %, their mean within 5 %.  Shorter segments are left out: there the window's main lobe (+-9 bins of the
    200 dB Kaiser window) spans a good part of the band, the filters' response changes across it, and the part of y
    that one complex gain per row cannot follow is left in Sres (a resolution bias, not noise)."""
    rows = sel & (_plan_L(n, fs, Jdes=Jdes) >= 100)
    assert rows.sum() >= 20
    ratio = sres[rows] / (2 * SIGMA_N ** 2 / fs)
    assert np.max(np.abs(ratio - 1)) < 0.2 and abs(np.mean(ratio) - 1) < 0.05


# ---------------------------------------------------------------------------------------------------------- CPU
def test_oracle_two_paths_response_residual_and_coherence():
    """H recovers both filter responses; Sres is the PSD of n (white: 2 sigma^2 / fs); mcoh is 1 without n."""
    N, fs, J = 20000, 50.0, 120
    xs, y = _two_paths(N)
    out = ref_lcsd_cond(xs, y, fs, Jdes=J)
    sel = out["K"] >= 100
    assert sel.sum() >= 20
    f = out["f"][sel]
    assert np.max(np.abs(out["H"][0, sel] - _fir_response(H1, f, fs))) < 0.05
    assert np.max(np.abs(out["H"][1, sel] - _fir_response(H2, f, fs))) < 0.05
    _check_residual(out["Sres"], sel, N, fs, J)
    # unit white witnesses: mcoh = g / (g + sigma^2), g = |H1|^2 + |H2|^2 (H1 vanishes at fs / 2)
    rows = sel & (_plan_L(N, fs, Jdes=J) >= 100)
    g = np.abs(_fir_response(H1, out["f"][rows], fs)) ** 2 + np.abs(_fir_response(H2, out["f"][rows], fs)) ** 2
    assert np.max(np.abs(out["mcoh"][rows] - g / (g + SIGMA_N ** 2))) < 0.05
    assert np.all(out["mcoh"][out["K"] >= 2] <= 1 + 1e-12)
    # without n, mcoh -> 1 as the resolution gets finer: what is left is the filters' response varying across the
    # window's main lobe, which falls about as 1 / L^2 (1e-5 at L = 3200)
    quiet = ref_lcsd_cond(xs, _two_paths(N, noise=False)[1], fs, Jdes=J)
    L = _plan_L(N, fs, Jdes=J)
    ok = (quiet["K"] >= 2) & (L >= 100)
    assert ok.sum() >= 20
    assert np.all(1 - quiet["mcoh"][ok] < 1 / L[ok]) and np.all(quiet["mcoh"][ok] <= 1 + 1e-12)
    assert np.all(1 - quiet["mcoh"][(quiet["K"] >= 2) & (L >= 2000)] < 1e-4)
    # a witness added cannot raise the residual: the multiple coherence is at least each pairwise coherence, and well
    # above it where the other path carries power
    ok = quiet["K"] >= 2
    for a in range(2):
        single = ref_lcsd(xs[a], _two_paths(N, noise=False)[1], fs, Jdes=J)
        assert np.all(single["coh"][ok] <= quiet["mcoh"][ok] + 1e-12)
        assert np.max(quiet["mcoh"][ok] - single["coh"][ok]) > 0.3


def test_oracle_one_witness_is_lcsd():
    """Cx = 1: H is lcsd's tf and Sres is Syy (1 - coh), to rounding."""
    N, fs, J = 6000, 50.0, 120
    xs, ys = _miso(N, 1, 3)
    out = ref_lcsd_cond(xs, ys, fs, Jdes=J)
    ref = ref_lcsd(xs[0], ys, fs, Jdes=J)
    assert np.array_equal(out["f"], ref["f"]) and np.array_equal(out["enbw"], ref["enbw"])
    assert np.max(np.abs(out["Sxx"][0, 0].real / ref["Sxx"] - 1)) < 1e-12 and np.all(out["Sxx"][0, 0].imag == 0)
    assert np.max(np.abs(out["Syy"] / ref["Syy"] - 1)) < 1e-12
    assert np.all(np.abs(out["Sxy"][0] - ref["Sxy"]) <= 1e-12 * np.sqrt(ref["Sxx"] * ref["Syy"]))
    assert np.all(np.abs(out["H"][0] - ref["tf"]) <= 1e-12 * np.sqrt(ref["Syy"] / ref["Sxx"]))
    assert np.all(np.abs(out["Sres"] - ref["Syy"] * (1 - ref["coh"])) <= 1e-12 * ref["Syy"])
    assert np.max(np.abs(out["mcoh"] - ref["coh"])) < 1e-12


def test_oracle_singular_rows_are_nan():
    """A duplicated witness makes every row singular; rows with fewer segments than witnesses are NaN too."""
    N, fs, J = 6000, 50.0, 120
    xs, ys = _miso(N, 3, 2)
    out = ref_lcsd_cond(xs, ys, fs, Jdes=J)
    few = out["K"] < 3
    assert few.sum() >= 1 and (~few).sum() >= 50
    for k in ("H", "Sres", "mcoh"):
        assert np.all(np.isnan(out[k][..., few])) and not np.any(np.isnan(out[k][..., ~few])), k
    assert not np.any(np.isnan(out["Sxx"])) and not np.any(np.isnan(out["Syy"]))
    dup = ref_lcsd_cond(np.stack([xs[0], xs[1], xs[0]]), ys, fs, Jdes=J)
    for k in ("H", "Sres", "mcoh"):
        assert np.all(np.isnan(dup[k])), k
    dep = ref_lcsd_cond(np.stack([xs[0], xs[1], 2 * xs[0] - 0.5 * xs[1]]), ys, fs, Jdes=J)
    assert np.all(np.isnan(dep["Sres"]))


def test_argument_errors_need_no_device():
    from deepfmkit_b200 import DeepFitObject, lcsd_conditioned
    with pytest.raises(ValueError):
        lcsd_conditioned(np.zeros(100), np.zeros(101), 1.0)
    with pytest.raises(ValueError):
        lcsd_conditioned(np.zeros((2, 100)), np.zeros((3, 99)), 1.0)
    with pytest.raises(ValueError):
        lcsd_conditioned(np.zeros((65, 100)), np.zeros(100), 1.0)
    with pytest.raises(ValueError):
        lcsd_conditioned(np.zeros((0, 100)), np.zeros(100), 1.0)
    a, b, c = DeepFitObject(), DeepFitObject(), DeepFitObject()
    a.fs, b.fs, c.fs = 50.0, 50.0, 25.0
    a.phi, b.phi, c.phi = np.zeros(100), np.zeros(100), np.zeros(100)
    with pytest.raises(ValueError):
        a.calc_conditioned([b, c])
    c.fs, c.phi = 50.0, np.zeros(99)
    with pytest.raises(ValueError):
        a.calc_conditioned([b, c])
    with pytest.raises(ValueError):
        a.calc_conditioned([])


def test_entry_is_declared_and_bound():
    from deepfmkit_b200 import _lib
    assert "dfk_lcsd_cond_dev" in _lib.SYMBOLS
    assert len(_lib.SYMBOLS["dfk_lcsd_cond_dev"][1]) == 22


# ---------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def torch_mod():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _expand_y(out):
    """A 1-D target result with its Cy axis restored."""
    if out["Syy"].ndim == 1:
        out = dict(out)
        for k in ("Syy", "Sres", "mcoh"):
            out[k] = out[k][None]
        for k in ("Sxy", "H"):
            out[k] = out[k][:, None]
    return out


def _assert_matches_oracle(got, ref, tol=SPEC_TOL):
    got, ref = _expand_y(got), _expand_y(ref)
    assert np.array_equal(got["f"], ref["f"]) and np.array_equal(got["navs"], ref["K"])
    assert np.max(np.abs(got["enbw"] / ref["enbw"] - 1)) < 1e-12
    dx = np.real(np.einsum("aaj->aj", ref["Sxx"]))
    assert np.all(np.abs(got["Sxx"] - ref["Sxx"]) <= tol * np.sqrt(dx[:, None, :] * dx[None, :, :]))
    assert np.all(np.imag(np.einsum("aaj->aj", got["Sxx"])) == 0)
    assert np.array_equal(got["Sxx"], np.conj(np.transpose(got["Sxx"], (1, 0, 2))))
    assert np.max(np.abs(got["Syy"] / ref["Syy"] - 1)) < tol
    assert np.all(np.abs(got["Sxy"] - ref["Sxy"]) <= tol * np.sqrt(dx[:, None, :] * ref["Syy"][None, :, :]))
    nan = np.isnan(ref["Sres"])
    for k in ("Sres", "mcoh"):
        assert np.array_equal(np.isnan(got[k]), nan), k
    assert np.array_equal(np.isnan(got["H"]), np.isnan(ref["H"]))
    ok = ~nan
    assert np.all(np.abs(got["Sres"][ok] - ref["Sres"][ok]) <= tol * ref["Syy"][ok])
    assert np.max(np.abs(got["mcoh"][ok] - ref["mcoh"][ok]), initial=0.0) <= tol
    hs = np.sqrt(ref["Syy"][None, :, :] / dx[:, None, :])
    okh = ~np.isnan(ref["H"])
    assert np.all(np.abs(got["H"] - ref["H"])[okh] <= tol * hs[okh])


@pytest.mark.gpu
@pytest.mark.parametrize("kw", OPTION_SETS)
def test_lcsd_conditioned_matches_oracle(torch_mod, kw):
    from deepfmkit_b200 import lcsd_conditioned
    N, fs = 6000, 50.0
    xs, ys = _miso(N, 2, 3)
    okw = dict(Jdes=120)
    okw.update(kw)
    got = lcsd_conditioned(xs, ys, fs, **okw)
    nf = len(got["f"])
    assert got["Sxx"].shape == (2, 2, nf) and got["H"].shape == (2, 3, nf) and got["Sres"].shape == (3, nf)
    assert got["H"].dtype == np.complex128 and got["Sxy"].dtype == np.complex128
    _assert_matches_oracle(got, ref_lcsd_cond(xs, ys, fs, **okw))


@pytest.mark.gpu
def test_spectra_agree_with_lcsd_and_one_witness_is_lcsd(torch_mod):
    """Sxx (every entry), Sxy and Syy are lcsd's on the same series; with one witness H is lcsd's tf and mcoh its
    coherence."""
    from deepfmkit_b200 import lcsd, lcsd_conditioned
    N, fs, J = 6000, 50.0, 120
    xs, ys = _miso(N, 3, 4)
    got = lcsd_conditioned(xs, ys, fs, Jdes=J)
    xx = lcsd(xs, xs, fs, Jdes=J)
    xy = lcsd(xs, ys, fs, Jdes=J)
    dx = xx["Sxx"]
    assert np.all(np.abs(got["Sxx"] - xx["Sxy"]) <= LCSD_TOL * np.sqrt(dx[:, None, :] * dx[None, :, :]))
    assert np.max(np.abs(got["Syy"] / xy["Syy"] - 1)) < LCSD_TOL
    assert np.all(np.abs(got["Sxy"] - xy["Sxy"]) <= LCSD_TOL * np.sqrt(dx[:, None, :] * xy["Syy"][None, :, :]))
    assert np.array_equal(got["f"], xy["f"]) and np.array_equal(got["navs"], xy["navs"])
    assert np.array_equal(got["enbw"], xy["enbw"])

    one = lcsd_conditioned(xs[1], ys, fs, Jdes=J)
    pair = lcsd(xs[1], ys, fs, Jdes=J)
    assert np.all(np.abs(one["H"][0] - pair["tf"]) <= LCSD_TOL * np.sqrt(pair["Syy"] / pair["Sxx"]))
    assert np.max(np.abs(one["mcoh"] - pair["coh"])) < LCSD_TOL
    assert np.all(np.abs(one["Sres"] - pair["Syy"] * (1 - pair["coh"])) <= LCSD_TOL * pair["Syy"])


@pytest.mark.gpu
def test_long_segments_strided_columns_determinism_and_launches(torch_mod):
    """CTA-per-group path (L >= 2048); witness and target columns of a row table read in place (stride 8); CUDA
    tensors and numpy give the same bits; a repeated call gives the same bits; exactly three launches per call."""
    from deepfmkit_b200 import _lib, lcsd_conditioned
    torch = torch_mod
    N, fs, J, K = 40000, 50.0, 40, 8
    xs, ys = _miso(N, 2, 1)
    opts = _lib.default_lpsd_opts()
    opts.jdes, opts.kdes = J, K
    assert int(np.max(_lib.lpsd_plan(N, fs, opts)["L"])) >= 2048
    got = lcsd_conditioned(xs, ys, fs, Jdes=J, Kdes=K)
    _assert_matches_oracle(got, ref_lcsd_cond(xs, ys, fs, Jdes=J, Kdes=K))

    xd, yd = torch.from_numpy(xs).cuda(), torch.from_numpy(ys).cuda()
    on_dev = lcsd_conditioned(xd, yd, fs, Jdes=J, Kdes=K)
    again = lcsd_conditioned(xd, yd, fs, Jdes=J, Kdes=K)
    for k in got:
        assert np.array_equal(on_dev[k], got[k], equal_nan=True), k
        assert np.array_equal(again[k], got[k], equal_nan=True), k

    # witnesses in columns 1 and 3, the target in column 6 of a [N, 8] row table
    rows = torch.zeros((N, 8), dtype=torch.float64, device="cuda")
    rows[:, 1] = xd[0]
    rows[:, 3] = xd[1]
    rows[:, 6] = yd[0]
    torch.cuda.synchronize()
    ctx = _lib.get_context(0)
    n0 = ctx.launch_count()
    col = ctx.lcsd_cond_dev(rows.data_ptr() + 1 * 8, 2, 2, rows.data_ptr() + 6 * 8, 1, 0, N, 8, fs, opts)
    assert ctx.launch_count() - n0 == 3
    for k in got:
        assert np.array_equal(col[k], got[k], equal_nan=True), k


@pytest.mark.gpu
def test_witness_limit_and_wide_targets(torch_mod):
    """Cx = 64 (the limit) against the reference, Cx = 65 refused by the function and the C ABI; Cx = 8 x Cy = 256."""
    from deepfmkit_b200 import _lib, lcsd_conditioned
    torch = torch_mod
    N, fs, J = 3000, 50.0, 60
    xs, ys = _miso(N, 64, 1)
    got = lcsd_conditioned(xs, ys[0], fs, Jdes=J)
    ref = ref_lcsd_cond(xs, ys[0], fs, Jdes=J)
    assert np.sum(ref["K"] >= 64) >= 10  # rows that can be solved
    _assert_matches_oracle(got, ref)
    x65 = np.vstack([xs, xs[:1]])
    with pytest.raises(ValueError):
        lcsd_conditioned(x65, ys[0], fs, Jdes=J)
    xd = torch.from_numpy(x65).cuda()
    ctx = _lib.get_context(0)
    with pytest.raises(RuntimeError, match="dfk_b200 error -1"):
        ctx.lcsd_cond_dev(xd.data_ptr(), 65, N, xd.data_ptr(), 1, N, N, 1, fs)

    xs, ys = _miso(N, 8, 256, seed=7)
    got = lcsd_conditioned(xs, ys, fs, Jdes=J)
    assert got["H"].shape == (8, 256, len(got["f"]))
    _assert_matches_oracle(got, ref_lcsd_cond(xs, ys, fs, Jdes=J))


@pytest.mark.gpu
def test_singular_rows_on_device(torch_mod):
    from deepfmkit_b200 import lcsd_conditioned
    N, fs, J = 6000, 50.0, 120
    xs, ys = _miso(N, 3, 2)
    dup = np.stack([xs[0], xs[1], xs[0]])
    got = lcsd_conditioned(dup, ys, fs, Jdes=J)
    for k in ("H", "Sres", "mcoh"):
        assert np.all(np.isnan(got[k])), k
    assert not np.any(np.isnan(got["Sxx"])) and not np.any(np.isnan(got["Sxy"]))
    got = lcsd_conditioned(xs, ys, fs, Jdes=J)
    few = got["navs"] < 3
    assert few.sum() >= 1
    for k in ("H", "Sres", "mcoh"):
        assert np.all(np.isnan(got[k][..., few])) and not np.any(np.isnan(got[k][..., ~few])), k


@pytest.mark.gpu
def test_physics_on_device(torch_mod):
    from deepfmkit_b200 import lcsd_conditioned
    N, fs, J = 20000, 50.0, 120
    xs, y = _two_paths(N)
    out = lcsd_conditioned(xs, y, fs, Jdes=J)
    sel = out["navs"] >= 100
    f = out["f"][sel]
    assert np.max(np.abs(out["H"][0, sel] - _fir_response(H1, f, fs))) < 0.05
    assert np.max(np.abs(out["H"][1, sel] - _fir_response(H2, f, fs))) < 0.05
    _check_residual(out["Sres"], sel, N, fs, J)


@pytest.mark.gpu
def test_errors_and_null_outputs(torch_mod):
    import ctypes
    from deepfmkit_b200 import _lib, lcsd_conditioned
    torch = torch_mod
    N, fs = 3000, 50.0
    x = torch.from_numpy(_white(1, N)).cuda()
    with pytest.raises(ValueError):
        lcsd_conditioned(x, x[:-1], fs)
    if torch.cuda.device_count() >= 2:
        with pytest.raises(ValueError):
            lcsd_conditioned(x, x.to("cuda:1"), fs)
    ctx = _lib.get_context(0)
    opts = _lib.default_lpsd_opts()
    p = x.data_ptr()
    for cx, cy, stride in ((0, 1, 1), (1, 0, 1), (1, 1, 0), (65, 1, 1), (64, 65535 - 63, 1)):
        with pytest.raises(RuntimeError, match="dfk_b200 error -1"):
            ctx.lcsd_cond_dev(p, cx, 0, p, cy, 0, N, stride, fs, opts)
    lib = ctx.lib
    nf = ctypes.c_int32()
    cap = len(_lib.lpsd_plan(N, fs, opts)["f"])
    nulls = [None] * 9
    rc = lib.dfk_lcsd_cond_dev(ctx._h, p, 1, N, p, 1, N, N, 1, fs, ctypes.byref(opts), cap - 1, ctypes.byref(nf), *nulls)
    assert rc == -1 and nf.value == cap  # DFK_ERR_ARG
    n0 = ctx.launch_count()
    rc = lib.dfk_lcsd_cond_dev(ctx._h, p, 1, N, p, 1, N, N, 1, fs, ctypes.byref(opts), cap, ctypes.byref(nf), *nulls)
    assert rc == 0 and nf.value == cap and ctx.launch_count() - n0 == 3


@pytest.mark.gpu
def test_facade_calc_conditioned(torch_mod):
    """Three fitted channels through the façade: calc_conditioned is lcsd_conditioned on their phases with the target
    fit's settings, and stores nothing."""
    from deepfmkit_b200 import DeepFitFramework, DeepRawObject, lcsd_conditioned
    from oracle import dfmi_oracle as orc
    dff = DeepFitFramework()
    fits = {}
    for label, seed in (("main", 4), ("w1", 5), ("w2", 6)):
        x = orc.snr_signal(6.0, 200e3, 1000.0, 2.0, 40.0, seed=seed)
        dff.load_raw_object(DeepRawObject(data=x, f_samp=200e3, f_mod=1000.0, label=label))
        fits[label] = dff.fit(label, n=4)
    main, w1, w2 = fits["main"], fits["w1"], fits["w2"]
    main.Jdes, main.Kdes, main.order = 80, 30, 1
    got = main.calc_conditioned([w1, w2])
    ref = lcsd_conditioned(np.stack([w1.phi, w2.phi]), main.phi, main.fs, main.olap, main.bmin, main.Lmin, 80, 30, 1,
                           main.win, main.psll)
    assert set(got) == {"f", "enbw", "navs", "Sxx", "Syy", "Sxy", "H", "Sres", "mcoh"}
    for k in got:
        assert np.array_equal(got[k], ref[k], equal_nan=True), k
    one = main.calc_conditioned(w1)
    assert one["Sxx"].shape == (1, 1, len(one["f"]))
    assert main.f is None and main.Sxx is None
