"""Time-domain witness subtraction (``wiener_subtract``): least-squares multi-input FIR filters and the cleaned
target series.

CPU part: ``ref_wiener``, the CPU reference, builds the explicit lagged design matrix on the M rows on which every tap
is inside the record and solves the loaded normal equations with numpy.  It is checked on its own (two FIR paths plus
white noise, the one-tap regression coefficient, causal against centred filters, a duplicated witness with and without
ridge), together with the argument checks that need no device.  GPU part (-m gpu): the CUDA kernels through the C ABI
against ``ref_wiener`` over shapes up to the 1024-unknown cap, strided columns, determinism and the launch count,
singular and ridge cases, NULL outputs, agreement with ``lcsd_conditioned``'s residual PSD, and witness subtraction of
laser-frequency noise from simulated and fitted channels.
"""
import numpy as np
import pytest

PIVOT_TOL = 1e-10  # the device's singular-pivot threshold, relative to the loaded diagonal entry


def ref_wiener(x, y, taps, lead=None, ridge=0.0):
    """CPU reference of ``wiener_subtract``: x [N] or [Cx, N], y [N] or [Cy, N]; the same dict, plus ``cond`` (the
    2-norm condition number of the loaded normal matrix) and ``G`` (that matrix)."""
    xs = np.atleast_2d(np.asarray(x, dtype=np.float64))
    y = np.asarray(y, dtype=np.float64)
    y1 = y.ndim == 1
    ys = np.atleast_2d(y)
    cx, n = xs.shape
    L = int(taps)
    k0 = (L - 1) // 2 if lead is None else int(lead)
    n0, M, nu = L - 1 - k0, n - L + 1, cx * L
    xt = xs - xs.mean(axis=1, keepdims=True)
    yt = ys - ys.mean(axis=1, keepdims=True)
    rows = np.arange(n0, n0 + M)
    # column (a, k) of the design matrix: x~_a[n + k0 - k]
    phi = np.stack([xt[a, rows + k0 - k] for a in range(cx) for k in range(L)], axis=1)
    Y = yt[:, rows].T  # [M, Cy]
    G = phi.T @ phi
    p = phi.T @ Y
    G = G + ridge * np.trace(G) / nu * np.eye(nu)
    singular = False
    try:
        Lc = np.linalg.cholesky(G)
        singular = bool(np.any(np.diag(Lc) ** 2 <= PIVOT_TOL * np.diag(G)))
    except np.linalg.LinAlgError:
        singular = True
    cy = len(ys)
    var_y = np.mean(Y ** 2, axis=0)
    if singular:
        h = np.full((nu, cy), np.nan)
    else:
        h = np.linalg.solve(G, p)
    res = (Y - phi @ h).T
    var_res = np.mean(res ** 2, axis=1)
    with np.errstate(divide="ignore", invalid="ignore"):
        explained = np.where(var_y != 0, 1.0 - var_res / var_y, np.nan)
    out = {"h": h.T.reshape(cy, cx, L), "offsets": k0 - np.arange(L), "n0": n0, "lead": k0, "residual": res,
           "var_y": var_y, "var_res": var_res, "explained": explained, "singular": singular,
           "cond": np.inf if singular else np.linalg.cond(G), "G": G}
    if y1:
        for k in ("h", "residual", "var_y", "var_res", "explained"):
            out[k] = out[k][0]
    return out


def _white(seed, n):
    return np.random.RandomState(seed).randn(n)


def _fir(x, h):
    return np.convolve(x, h)[:len(x)]


# two causal FIR paths (<= 9 taps) and white noise: y = h1 * x1 + h2 * x2 + n
H1, H2, SIGMA_N = [0.5, 0.3, -0.2, 0.1], [-0.4, 0.0, 0.25, 0.1, 0.0, 0.05, -0.1, 0.02, 0.03], 0.3


def _two_paths(n, noise=True):
    x1, x2 = _white(11, n), _white(12, n)
    y = _fir(x1, H1) + _fir(x2, H2)
    n_part = SIGMA_N * _white(13, n)
    return np.stack([x1, x2]), (y + n_part if noise else y), n_part


def _mixed(n, cx, cy, L, seed=0, walk=False):
    """Witnesses [cx, n] (white with offsets, or random walks) and targets [cy, n]: each target a random FIR mix of
    every witness (taps inside the model's window) plus its own white noise."""
    rng = np.random.RandomState(1000 + seed)
    xs = rng.randn(cx, n) + 0.1 * np.arange(cx)[:, None]
    if walk:
        xs = np.cumsum(xs, axis=1) * 1e-2
    ys = 0.2 * rng.randn(cy, n) + 1.5
    taps = min(L, 4)
    for t in range(cy):
        for a in range(cx):
            ys[t] += _fir(xs[a], rng.randn(taps) / (1 + a))
    return xs, ys


# ---------------------------------------------------------------------------------------------------------- CPU
def test_oracle_two_paths():
    """L = 16 with the centred lead: h recovers both responses at the offsets of a causal filter, the residual is the
    noise, and ``explained`` is the fraction of var_y not due to the noise."""
    N, L = 20000, 16
    xs, y, n_part = _two_paths(N)
    out = ref_wiener(xs, y, L)
    k0 = out["lead"]
    assert k0 == 7 and out["n0"] == 8 and np.array_equal(out["offsets"], 7 - np.arange(16))
    for a, hh in enumerate((H1, H2)):
        want = np.zeros(L)
        want[k0:k0 + len(hh)] = hh  # offset -j (tap k0 + j) carries h[j]
        assert np.max(np.abs(out["h"][a] - want)) < 0.01, a
    rows = slice(out["n0"], out["n0"] + N - L + 1)
    noise = n_part[rows] - n_part.mean()
    # the least-squares fit also removes the noise's projection on the n_u = 32 columns: rms sigma sqrt(n_u / M)
    assert np.sqrt(np.mean((out["residual"] - noise) ** 2)) < 2 * SIGMA_N * np.sqrt(2 * L / (N - L + 1))
    frac = np.mean(noise ** 2) / out["var_y"]
    assert abs(out["explained"] - (1 - frac)) < 2e-3
    assert not out["singular"]


def test_oracle_one_tap_is_the_regression_coefficient():
    N = 5000
    x, y = _white(1, N) + 3.0, 0.7 * _white(1, N) + 0.4 * _white(2, N) - 1.0
    out = ref_wiener(x, y, 1)
    assert out["n0"] == 0 and out["residual"].shape == (N,)
    xc, yc = x - x.mean(), y - y.mean()
    assert abs(out["h"][0, 0] - np.sum(xc * yc) / np.sum(xc * xc)) < 1e-12
    assert abs(out["var_y"] - np.var(y)) < 1e-12


def test_oracle_causal_and_centred_lead():
    """A delayed path is found by both the causal (lead 0) and the centred filter, at the tap of its offset; an
    advanced path only by the centred one."""
    N, L = 8000, 9
    x = _white(3, N)
    delayed = 0.7 * np.concatenate([np.zeros(3), x[:-3]]) + 0.1 * _white(4, N)
    causal, centred = ref_wiener(x, delayed, L, lead=0), ref_wiener(x, delayed, L)
    assert np.argmax(np.abs(causal["h"][0])) == 3 and abs(causal["h"][0, 3] - 0.7) < 0.01
    assert np.argmax(np.abs(centred["h"][0])) == 4 + 3 and abs(centred["h"][0, 7] - 0.7) < 0.01
    assert causal["offsets"][3] == -3 and centred["offsets"][7] == -3
    assert abs(causal["var_res"] - centred["var_res"]) < 1e-3 * causal["var_y"]
    advanced = 0.7 * np.concatenate([x[2:], np.zeros(2)]) + 0.1 * _white(4, N)
    causal, centred = ref_wiener(x, advanced, L, lead=0), ref_wiener(x, advanced, L)
    assert causal["explained"] < 0.05 and centred["explained"] > 0.95
    assert abs(centred["h"][0, 4 - 2] - 0.7) < 0.01


def test_oracle_duplicated_witness():
    """Two copies of a witness: singular with ridge 0; with ridge the copies get equal halves of the true filter."""
    N, L = 20000, 16
    xs, y, _ = _two_paths(N)
    dup = np.stack([xs[0], xs[0], xs[1]])
    out = ref_wiener(dup, y, L)
    assert out["singular"] and np.all(np.isnan(out["h"])) and np.all(np.isnan(out["residual"]))
    assert np.all(np.isnan(out["var_res"])) and np.isnan(out["explained"]) and np.isfinite(out["var_y"])
    good = ref_wiener(dup, y, L, ridge=1e-6)
    assert not good["singular"]
    assert np.max(np.abs(good["h"][0] - good["h"][1])) < 1e-9
    want = np.zeros(L)
    want[7:7 + len(H1)] = H1
    assert np.max(np.abs(good["h"][0] + good["h"][1] - want)) < 0.01


def test_argument_errors_need_no_device():
    from deepfmkit_b200 import DeepFitObject, wiener_subtract
    x, y = np.zeros((2, 100)), np.zeros(100)
    bad = [
        dict(witnesses=np.zeros(100), targets=np.zeros(101), taps=2),          # length mismatch
        dict(witnesses=np.zeros((65, 4000)), targets=y[:1].repeat(4000), taps=1),  # Cx > 64
        dict(witnesses=np.zeros((0, 100)), targets=y, taps=1),                  # Cx = 0
        dict(witnesses=x, targets=np.zeros((0, 100)), taps=1),                  # Cy = 0
        dict(witnesses=np.zeros((1, 2)), targets=np.zeros((65535, 2)), taps=1),  # Cx + Cy > 65535
        dict(witnesses=x, targets=y, taps=0),
        dict(witnesses=x, targets=y, taps=2.0),
        dict(witnesses=np.zeros((2, 5000)), targets=np.zeros(5000), taps=513),  # Cx L > 1024
        dict(witnesses=x, targets=y, taps=34),                                  # M = 67 < Cx L = 68
        dict(witnesses=x, targets=y, taps=4, lead=-1),
        dict(witnesses=x, targets=y, taps=4, lead=4),
        dict(witnesses=x, targets=y, taps=4, ridge=-1.0),
        dict(witnesses=x, targets=y, taps=4, ridge=np.nan),
        dict(witnesses=x, targets=y, taps=4, ridge=np.inf),
        dict(witnesses=np.zeros((2, 3, 100)), targets=y, taps=1),
    ]
    for kw in bad:
        with pytest.raises(ValueError):
            wiener_subtract(**kw)
    a, b, c = DeepFitObject(), DeepFitObject(), DeepFitObject()
    a.fs, b.fs, c.fs = 50.0, 50.0, 25.0
    a.phi, b.phi, c.phi = np.zeros(100), np.zeros(100), np.zeros(100)
    with pytest.raises(ValueError):
        a.subtract_witnesses([b, c], 3)
    c.fs, c.phi = 50.0, np.zeros(99)
    with pytest.raises(ValueError):
        a.subtract_witnesses([b, c], 3)
    with pytest.raises(ValueError):
        a.subtract_witnesses([], 3)
    with pytest.raises(ValueError):
        a.subtract_witnesses(b, 60)  # M = 41 < L = 60


def test_entry_is_declared_and_bound():
    from deepfmkit_b200 import _lib
    assert "dfk_wiener_dev" in _lib.SYMBOLS
    assert len(_lib.SYMBOLS["dfk_wiener_dev"][1]) == 18


def launches(nu, residual=True, var_res=True):
    """The launch count dfk_wiener_dev documents: 2 ceil(n_u / 64) + 4 (+1 with a residual or var_res, +1 for var_res)."""
    return 2 * (-(-nu // 64)) + 4 + int(residual or var_res) + int(var_res)


# ---------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def torch_mod():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


WELL_CONDITIONED = 1e3  # cond(G) of every white-witness system below except the square one at the cap (at most 3.2e2)


def _tolerances(ref, ill_conditioned):
    """The gates on h (relative to max|h|) and on the residual (relative to rms(y~)).

    A well-conditioned system (white witnesses; checked: cond(G) < WELL_CONDITIONED) gets the fixed 1e-9 gates.  A
    system marked ill-conditioned gets gates that grow with cond(G): a backward-stable solve of the normal equations has
    a forward error of about cond(G) eps in h and about sqrt(cond(G)) eps in the prediction (the error in h lies along
    the directions the witnesses barely excite), and the device and numpy round differently.  Three systems here are
    marked: random-walk witnesses (cond 2e7), the square system M = n_u at the 1024-unknown cap (a 1024 x 1024 random
    design matrix, cond 2e7) and a duplicated witness held apart only by the ridge (cond 2e6)."""
    c = ref["cond"]
    if not ill_conditioned:
        assert c < WELL_CONDITIONED, c
        return 1e-9, 1e-9
    return max(1e-9, 1e-13 * c), max(1e-9, 1e-12 * np.sqrt(c))


def _assert_matches(got, ref, ill_conditioned=False):
    tol_h, tol_e = _tolerances(ref, ill_conditioned)
    assert got["singular"] == ref["singular"] is False
    assert got["n0"] == ref["n0"] and got["lead"] == ref["lead"]
    assert np.array_equal(got["offsets"], ref["offsets"])
    assert got["h"].shape == ref["h"].shape
    assert np.max(np.abs(got["h"] - ref["h"])) <= tol_h * np.max(np.abs(ref["h"]))
    res = got["residual"]
    res = res.cpu().numpy() if hasattr(res, "cpu") else res
    assert res.shape == ref["residual"].shape
    rms_y = np.sqrt(np.atleast_1d(ref["var_y"]))
    err = np.abs(np.atleast_2d(res) - np.atleast_2d(ref["residual"]))
    assert np.all(err <= tol_e * rms_y[:, None])
    assert np.all(np.abs(got["var_y"] / ref["var_y"] - 1) < 1e-10)
    # var_res within 1e-10 relative; where almost nothing is left (M = n_u) the residual's own gate bounds it instead,
    # and for an ill-conditioned system the residual's error enters at first order
    dv = np.abs(got["var_res"] - ref["var_res"])
    slack = tol_e ** 2 * rms_y ** 2
    if ill_conditioned:
        slack = slack + 2 * tol_e * rms_y * np.sqrt(ref["var_res"])
    assert np.all(dv <= 1e-10 * ref["var_res"] + slack)
    assert np.all(np.abs(got["explained"] - ref["explained"]) <= dv / ref["var_y"] + 1e-12)


SHAPES = [  # (Cx, Cy, L, lead, N, random-walk witnesses, ill-conditioned)
    (1, 1, 1, None, 1000, False, False),
    (3, 2, 17, 0, 5001, False, False),
    (8, 2, 128, None, 20000, False, False),   # n_u = 1024, the cap
    (8, 1, 128, 100, 1151, False, True),      # n_u = 1024 and M = n_u exactly: a square random system
    (2, 1, 6, 2, 17, False, False),           # M = n_u exactly, tiny
    (64, 1, 16, None, 3001, False, False),
    (2, 300, 8, None, 4099, False, False),    # Cy = 300
    (5, 3, 21, 13, 10007, False, False),      # N a multiple of no tile size
    (4, 2, 12, None, 6000, True, True),       # random-walk witnesses
]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s[:5])) + ("w" if s[5] else ""))
def test_matches_oracle(torch_mod, shape):
    from deepfmkit_b200 import wiener_subtract
    cx, cy, L, lead, N, walk, ill = shape
    xs, ys = _mixed(N, cx, cy, L, seed=cx + cy + L, walk=walk)
    got = wiener_subtract(xs, ys, L, lead=lead)
    assert isinstance(got["residual"], np.ndarray) and got["residual"].shape == (cy, N - L + 1)
    _assert_matches(got, ref_wiener(xs, ys, L, lead=lead), ill_conditioned=ill)
    if cy == 1:
        one = wiener_subtract(xs, ys[0], L, lead=lead)
        assert one["h"].shape == (cx, L) and one["residual"].shape == (N - L + 1,)
        assert np.array_equal(one["h"], got["h"][0]) and np.array_equal(one["residual"], got["residual"][0])


@pytest.mark.gpu
def test_strided_columns_tensors_determinism_and_launches(torch_mod):
    """Witness and target columns of a [N, 8] row table read in place give the bits of contiguous copies; CUDA tensors
    and numpy give the same bits; a repeated call too; the launch count is the documented function of n_u."""
    from deepfmkit_b200 import _lib, wiener_subtract
    torch = torch_mod
    N, L, lead = 30011, 24, 5
    xs, ys = _mixed(N, 3, 2, L, seed=5)
    ctx = _lib.get_context(0)
    n0 = ctx.launch_count()
    got = wiener_subtract(xs, ys, L, lead=lead)
    assert ctx.launch_count() - n0 == launches(3 * L)
    _assert_matches(got, ref_wiener(xs, ys, L, lead=lead))
    xd, yd = torch.from_numpy(xs).cuda(), torch.from_numpy(ys).cuda()
    on_dev = wiener_subtract(xd, yd, L, lead=lead)
    again = wiener_subtract(xd, yd, L, lead=lead)
    assert isinstance(on_dev["residual"], torch.Tensor) and on_dev["residual"].is_cuda
    for k in ("h", "var_y", "var_res", "explained"):
        assert np.array_equal(on_dev[k], got[k]) and np.array_equal(again[k], got[k]), k
    assert np.array_equal(on_dev["residual"].cpu().numpy(), got["residual"])
    assert torch.equal(again["residual"], on_dev["residual"])

    rows = torch.zeros((N, 8), dtype=torch.float64, device="cuda")
    for c, v in zip((0, 2, 4, 5, 7), (xd[0], xd[1], xd[2], yd[0], yd[1])):
        rows[:, c] = v
    torch.cuda.synchronize()
    M = N - L + 1
    res = torch.full((2, M + 7), 123.0, dtype=torch.float64, device="cuda")
    col = ctx.wiener_dev(rows.data_ptr(), 3, 2, rows.data_ptr() + 5 * 8, 2, 2, N, 8, L, lead, 0.0, res.data_ptr(),
                         M + 7)
    for k in ("h", "var_y", "var_res"):
        assert np.array_equal(col[k], got[k]), k
    assert np.array_equal(res[:, :M].cpu().numpy(), got["residual"])
    assert torch.all(res[:, M:] == 123.0)


@pytest.mark.gpu
def test_singular_and_ridge_on_device(torch_mod):
    from deepfmkit_b200 import wiener_subtract
    N, L = 20000, 16
    xs, y, _ = _two_paths(N)
    dup = np.stack([xs[0], xs[0], xs[1]])
    out = wiener_subtract(dup, y, L)
    assert out["singular"]
    assert np.all(np.isnan(out["h"])) and np.all(np.isnan(out["residual"]))
    assert np.isnan(out["var_res"]) and np.isnan(out["explained"])
    assert np.isfinite(out["var_y"]) and abs(out["var_y"] / ref_wiener(dup, y, L)["var_y"] - 1) < 1e-10
    good = wiener_subtract(dup, y, L, ridge=1e-6)
    ref = ref_wiener(dup, y, L, ridge=1e-6)
    assert not good["singular"]
    _assert_matches(good, ref, ill_conditioned=True)
    assert np.max(np.abs(good["h"][0] - good["h"][1])) < 1e-9
    want = np.zeros(L)
    want[7:7 + len(H1)] = H1
    assert np.max(np.abs(good["h"][0] + good["h"][1] - want)) < 0.01


@pytest.mark.gpu
def test_null_outputs(torch_mod):
    """Filters only (no residual, no variances) and residual only, through Context.wiener_dev."""
    from deepfmkit_b200 import _lib, wiener_subtract
    torch = torch_mod
    N, L = 7000, 10
    xs, ys = _mixed(N, 2, 3, L, seed=9)
    full = wiener_subtract(xs, ys, L)
    xd, yd = torch.from_numpy(xs).cuda(), torch.from_numpy(ys).cuda()
    ctx = _lib.get_context(0)
    n0 = ctx.launch_count()
    only_h = ctx.wiener_dev(xd.data_ptr(), 2, N, yd.data_ptr(), 3, N, N, 1, L, (L - 1) // 2, variances=False)
    assert ctx.launch_count() - n0 == launches(2 * L, residual=False, var_res=False)
    assert np.array_equal(only_h["h"], full["h"]) and only_h["var_y"] is None and not only_h["singular"]
    M = N - L + 1
    res = torch.empty((3, M), dtype=torch.float64, device="cuda")
    n0 = ctx.launch_count()
    only_res = ctx.wiener_dev(xd.data_ptr(), 2, N, yd.data_ptr(), 3, N, N, 1, L, (L - 1) // 2, 0.0, res.data_ptr(), M,
                              filters=False, variances=False)
    assert ctx.launch_count() - n0 == launches(2 * L, residual=True, var_res=False)
    assert only_res["h"] is None
    assert np.array_equal(res.cpu().numpy(), full["residual"])


@pytest.mark.gpu
def test_c_abi_rejects_every_limit(torch_mod):
    """DFK_ERR_ARG for each limit, a bad lead or ridge, and a tap count so large that Cx L overflows int64."""
    from deepfmkit_b200 import _lib
    torch = torch_mod
    N = 4000
    x = torch.from_numpy(np.random.RandomState(3).randn(65, N)).cuda()
    p, ctx = x.data_ptr(), _lib.get_context(0)
    cases = [dict(Cx=65, L=1), dict(Cx=0, L=1), dict(Cy=0, L=1), dict(Cx=2, Cy=65534, L=1), dict(Cx=2, L=513),
             dict(Cx=1, L=0), dict(Cx=1, L=4, lead=4), dict(Cx=1, L=4, lead=-1), dict(Cx=1, L=4, ridge=-1.0),
             dict(Cx=1, L=4, ridge=float("nan")), dict(Cx=1, L=4, ridge=float("inf")), dict(Cx=4, L=2 ** 62),
             dict(Cx=8, L=128, N=1150), dict(Cx=1, L=4, stride=0)]
    for c in cases:
        kw = dict(Cx=1, Cy=1, N=N, L=1, lead=0, ridge=0.0, stride=1)
        kw.update(c)
        with pytest.raises(RuntimeError, match="dfk_b200 error -1"):
            ctx.wiener_dev(p, kw["Cx"], N, p, kw["Cy"], N, kw["N"], kw["stride"], kw["L"], kw["lead"], kw["ridge"],
                           filters=False, variances=False)


@pytest.mark.gpu
def test_agrees_with_lcsd_conditioned(torch_mod):
    """On the two-path case the residual's LPSD and lcsd_conditioned's Sres estimate the same white noise floor.  Each
    row's estimate has a relative standard deviation of about 1 / sqrt(K) (K = navs, fewer effective averages with the
    default overlap: counted as K / 2); the mean over rows is at least as good as its worst row, so the two means
    agree within 3 sqrt(2 / K_min + 2 / K_min') of each other."""
    from deepfmkit_b200 import _lib, lcsd_conditioned, lpsd, wiener_subtract
    N, L, fs, J = 200000, 16, 50.0, 200
    xs, y, _ = _two_paths(N)
    out = wiener_subtract(xs, y, L)
    _, _, psd, _, navs, plan = lpsd(out["residual"], fs, Jdes=J)
    cond = lcsd_conditioned(xs, y, fs, Jdes=J)
    opts = _lib.default_lpsd_opts()
    opts.jdes = J
    sel_r = (navs >= 1000) & (plan["L"] >= 100)
    sel_c = (cond["navs"] >= 1000) & (_lib.lpsd_plan(N, fs, opts)["L"] >= 100)
    assert sel_r.sum() >= 20 and sel_c.sum() >= 20
    a, b = np.mean(psd[sel_r]), np.mean(cond["Sres"][sel_c])
    tol = 3 * np.sqrt(2 / navs[sel_r].min() + 2 / cond["navs"][sel_c].min())
    assert abs(a / b - 1) < tol
    assert abs(a / (2 * SIGMA_N ** 2 / fs) - 1) < tol


def _fitted_pair(dm=6.0, seconds=2.0, scale=2e4):
    """A main channel (m = 12.6) and a witness (m = ``dm``) on the same laser, whose frequency noise is a random walk
    handed in through external_noise; both fitted (n = 4).  The witness depth stays inside the fitter's initial m grid
    (5..30): a shallower witness converges to another depth, and its phase then no longer scales with its arm-length
    mismatch.  Returns (main fit, witness fit, arm-length mismatch of main / witness)."""
    import deepfmkit_b200 as dfk
    from deepfmkit_b200 import physics
    laser = physics.LaserConfig()
    ifo = physics.InterferometerConfig()
    ifo.phi = 1.0
    dff = dfk.DeepFitFramework()
    main = physics.DFMIObject("main", laser, ifo, f_samp=200e3)
    dff.load_sim(main)
    wit = dff.create_witness_channel("main", "wit", m_witness=dm)
    n = int(seconds * main.f_samp)
    noise = {"laser_frequency": np.cumsum(np.random.RandomState(21).randn(n)) * scale}
    chans = physics.SignalGenerator().generate(main, seconds, mode="asd", witness_config=wit, external_noise=noise)
    dff.load_raw_object(chans["main"], "main")
    dff.load_raw_object(chans["witness"], "wit")
    fm, fw = dff.fit("main", n=4), dff.fit("wit", n=4)
    ratio = (ifo.meas_arml - ifo.ref_arml) / (wit.ifo.meas_arml - wit.ifo.ref_arml)
    return fm, fw, ratio


@pytest.mark.gpu
def test_physics_laser_frequency_noise(torch_mod):
    """Laser-frequency noise enters each channel's phase as 2 pi delta_f dl / c, so the witness predicts the main
    channel's phase noise with one tap, the ratio of the arm-length mismatches (its sign follows the fits' sign
    normalisation).  Gate: at least 99 % of the main phase's variance removed, and the zero-offset tap within 1 % of
    the ratio in magnitude, with every other tap below 2 % of it."""
    from deepfmkit_b200 import wiener_subtract
    fm, fw, ratio = _fitted_pair()
    assert np.std(fm.phi) > 0.01  # the noise is well above the fits' own scatter
    out = wiener_subtract(np.asarray(fw.phi), np.asarray(fm.phi), 5)
    assert out["explained"] > 0.99, out["explained"]
    k0 = out["lead"]
    h = out["h"][0]
    assert abs(abs(h[k0]) / abs(ratio) - 1) < 0.01, (h, ratio)
    assert np.all(np.abs(np.delete(h, k0)) < 0.02 * abs(ratio)), h


@pytest.mark.gpu
def test_facade_subtract_witnesses(torch_mod):
    from deepfmkit_b200 import wiener_subtract
    fm, fw, _ = _fitted_pair(seconds=1.0)
    got = fm.subtract_witnesses(fw, 3)
    ref = wiener_subtract(np.asarray(fw.phi)[None], np.asarray(fm.phi), 3)
    assert set(got) == {"h", "offsets", "n0", "lead", "residual", "var_y", "var_res", "explained", "singular"}
    for k in got:
        assert np.array_equal(got[k], ref[k]), k
    assert got["h"].shape == (1, 3) and got["residual"].shape == (len(fm.phi) - 2,)
    two = fm.subtract_witnesses([fw, fw], 3, ridge=1e-3)
    assert two["h"].shape == (2, 3) and not two["singular"]
    assert fm.f is None
