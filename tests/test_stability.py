"""Time-domain stability (``stability``, ``oadev`` / ``mdev`` / ``tdev`` / ``ohdev``, ``dfk_stability_dev``).

CPU: the numpy reference ``ref_stability`` (every term from window sums, no running sums) against brute-force loops
over the definitions, the identities between kinds, the expected Allan variance of white and random-walk series, the
host build of the double-double core (tests/host/stability_harness.cpp) against exact integer arithmetic on grid series
whose running sums pass 2^53 grid steps, and the argument checks.  GPU: agreement with the reference and the exact
values, bit-identity across batching, strides, input kinds, repeats and tau lists, the edge cases, the launch count
and the fit object's method."""
import ctypes
import math
import os
import subprocess
import tempfile
from fractions import Fraction

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KINDS = ("oadev", "mdev", "tdev", "ohdev")


# ---------------------------------------------------------------------------------------------------------------------
# reference
def _counts(Nx, m):
    return {"oadev": Nx - 2 * m, "mdev": Nx - 3 * m + 1, "tdev": Nx - 3 * m + 1, "ohdev": Nx - 3 * m}


def ref_m(Nx, fs, taus, kinds):
    """The averaging factors of a call, by the rules written out: the tau rule's m values inside at least one
    requested kind's range."""
    if isinstance(taus, str):
        if taus == "octave":
            cand = [2 ** k for k in range(int(math.floor(math.log2(Nx))) + 1)]
        elif taus == "decade":
            cand = [f * 10 ** k for k in range(int(math.floor(math.log10(Nx))) + 1) for f in (1, 2, 4)]
        else:
            cand = list(range(1, Nx + 1))
    else:
        cand = sorted({max(1, int(round(t * fs))) for t in taus})
    return np.array([m for m in cand if max(_counts(Nx, m)[k] for k in kinds) >= 1], dtype=np.int64)


def _win(a, m, n):
    """The first n window sums of length m of a (n <= 0: none)."""
    if n <= 0:
        return np.zeros(0)
    return np.lib.stride_tricks.sliding_window_view(a[:n + m - 1], m).sum(axis=-1)


def ref_stability(x, fs, kinds=KINDS, taus="octave", data_type="phase"):
    """numpy reference in ``stability``'s layout.  Every difference is formed from window sums of the input: for
    'freq' data the second difference of x at offset m is (W[i+m] - W[i]) / fs with W the length-m window sums of y,
    the third (W[i+2m] - 2 W[i+m] + W[i]) / fs, and mdev's term the length-m window sum of the second differences."""
    x = np.atleast_2d(np.asarray(x, dtype=np.float64))
    C, N = x.shape
    freq = data_type == "freq"
    Nx = N + 1 if freq else N
    ms = ref_m(Nx, fs, taus, kinds)
    out = {"taus": ms / fs, "m": ms}
    dev = {k: np.full((C, ms.size), np.nan) for k in KINDS}
    for c in range(C):
        v = x[c]
        for t, m in enumerate(ms):
            m = int(m)
            tau = m / fs
            cnt = _counts(Nx, m)
            na, nm, nh = cnt["oadev"], cnt["mdev"], cnt["ohdev"]
            if freq:
                W = _win(v, m, N - m + 1)
                a = (W[m:m + na] - W[:na]) / fs if na > 0 else np.zeros(0)
                h = (W[2 * m:2 * m + nh] - 2 * W[m:m + nh] + W[:nh]) / fs if nh > 0 else np.zeros(0)
            else:
                a = v[2 * m:2 * m + na] - 2 * v[m:m + na] + v[:na] if na > 0 else np.zeros(0)
                h = (v[3 * m:3 * m + nh] - 3 * v[2 * m:2 * m + nh] + 3 * v[m:m + nh] - v[:nh]) if nh > 0 else np.zeros(0)
            md = _win(a, m, nm)
            if na > 0:
                dev["oadev"][c, t] = np.sqrt(np.sum(a * a) / (2 * tau * tau * na))
            if nm > 0:
                dev["mdev"][c, t] = np.sqrt(np.sum(md * md) / (2 * m * m * tau * tau * nm))
                dev["tdev"][c, t] = tau * dev["mdev"][c, t] / np.sqrt(3)
            if nh > 0:
                dev["ohdev"][c, t] = np.sqrt(np.sum(h * h) / (6 * tau * tau * nh))
    for k in kinds:
        n = np.array([max(0, _counts(Nx, int(m))[k]) for m in ms], dtype=np.int64)
        out[k], out[k + "_n"] = dev[k], n
        with np.errstate(invalid="ignore", divide="ignore"):
            out[k + "_err"] = np.where(n > 0, dev[k] / np.sqrt(np.maximum(n, 1)), np.nan)
    return out


def brute_stability(v, fs, m, data_type):
    """The definitions as loops: x and S as running sums in Python floats (math.fsum), then each sum term by term."""
    v = [float(a) for a in v]
    x = [math.fsum(v[:n]) / fs for n in range(len(v) + 1)] if data_type == "freq" else v
    Nx = len(x)
    S = [math.fsum(x[:k]) for k in range(Nx + 1)]
    tau = m / fs
    res = {}
    n = Nx - 2 * m
    res["oadev"] = math.sqrt(sum((x[i + 2 * m] - 2 * x[i + m] + x[i]) ** 2 for i in range(n)) / (2 * tau ** 2 * n)) \
        if n > 0 else math.nan
    n = Nx - 3 * m + 1
    res["mdev"] = math.sqrt(sum((S[j + 3 * m] - 3 * S[j + 2 * m] + 3 * S[j + m] - S[j]) ** 2 for j in range(n))
                            / (2 * m * m * tau ** 2 * n)) if n > 0 else math.nan
    res["tdev"] = tau * res["mdev"] / math.sqrt(3)
    n = Nx - 3 * m
    res["ohdev"] = math.sqrt(sum((x[i + 3 * m] - 3 * x[i + 2 * m] + 3 * x[i + m] - x[i]) ** 2 for i in range(n))
                             / (6 * tau ** 2 * n)) if n > 0 else math.nan
    return res


def _close(a, b, tol):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape, (a.shape, b.shape)
    assert np.array_equal(np.isnan(a), np.isnan(b))
    ok = ~np.isnan(b)
    rel = np.abs(a[ok] - b[ok]) / np.abs(b[ok])
    assert rel.size == 0 or rel.max() <= tol, rel.max()


TAU_RULES = ["octave", "decade", "all", [0.5, 1.0, 1.0, 2.6, 7.0, 30.0]]


@pytest.mark.parametrize("data_type", ["phase", "freq"])
@pytest.mark.parametrize("taus", TAU_RULES, ids=["octave", "decade", "all", "explicit"])
def test_reference_equals_brute_force(data_type, taus):
    rs = np.random.RandomState(3)
    N, fs = 41, 2.0
    v = np.cumsum(rs.randn(N)) + 0.3 * rs.randn(N)
    ref = ref_stability(v, fs, KINDS, taus, data_type)
    from deepfmkit_b200.spectra import _stability_m
    Nx = N + (data_type == "freq")
    assert np.array_equal(ref["m"], _stability_m(Nx, fs, taus, KINDS))
    assert ref["m"].size > 0
    for t, m in enumerate(ref["m"]):
        b = brute_stability(v, fs, int(m), data_type)
        for k in KINDS:
            got = ref[k][0, t]
            assert (math.isnan(got) and math.isnan(b[k])) or abs(got / b[k] - 1) < 1e-9, (k, m, got, b[k])


def test_tau_rules():
    from deepfmkit_b200.spectra import _stability_m
    assert list(_stability_m(1000, 1.0, "octave", ("oadev",))) == [1, 2, 4, 8, 16, 32, 64, 128, 256]
    assert list(_stability_m(1000, 1.0, "octave", ("mdev",))) == [1, 2, 4, 8, 16, 32, 64, 128, 256]
    assert list(_stability_m(1000, 1.0, "decade", ("oadev",))) == [1, 2, 4, 10, 20, 40, 100, 200, 400]
    assert list(_stability_m(1000, 1.0, "decade", ("ohdev",))) == [1, 2, 4, 10, 20, 40, 100, 200]
    assert list(_stability_m(10, 1.0, "all", ("oadev", "ohdev"))) == [1, 2, 3, 4]
    assert list(_stability_m(10, 4.0, [0.1, 0.26, 0.24, 1.0, 100.0], ("oadev",))) == [1, 4]
    for Nx in (3, 7, 1000, 4096):
        for rule in TAU_RULES:
            for kinds in (KINDS, ("oadev",), ("ohdev",), ("mdev", "tdev")):
                assert np.array_equal(_stability_m(Nx, 3.0, rule, kinds), ref_m(Nx, 3.0, rule, kinds))


def test_identities():
    rs = np.random.RandomState(11)
    for data_type in ("phase", "freq"):
        v = rs.randn(3, 5000)
        ref = ref_stability(v, 10.0, KINDS, "octave", data_type)
        assert ref["m"][0] == 1
        assert np.allclose(ref["mdev"][:, 0], ref["oadev"][:, 0], rtol=1e-13, atol=0)
        assert np.allclose(ref["tdev"], ref["taus"] * ref["mdev"] / np.sqrt(3), rtol=1e-15, atol=0, equal_nan=True)


@pytest.mark.parametrize("model", ["white", "random_walk"])
def test_expected_allan_variance(model):
    """White y of variance s^2: AVAR = s^2 / m.  A random walk of y with step variance q: AVAR = q (2 m^2 + 1) / (6 m).
    Averaged over 16 series of 1.5e5 samples (rate 1), within 3 per cent for m = 1 .. 64."""
    rs = np.random.RandomState(5 if model == "white" else 6)
    C, N, s2 = 16, 150_000, 2.5
    e = rs.randn(C, N) * np.sqrt(s2)
    y = e if model == "white" else np.cumsum(e, axis=1)
    ref = ref_stability(y, 1.0, ("oadev",), [1, 2, 4, 8, 16, 32, 64], "freq")
    m = ref["m"].astype(np.float64)
    want = s2 / m if model == "white" else s2 * (2 * m * m + 1) / (6 * m)
    ratio = np.mean(ref["oadev"] ** 2, axis=0) / want
    assert np.all(np.abs(ratio - 1) < 0.03), ratio


# ---------------------------------------------------------------------------------------------------------------------
# exact values on grid series
GRID_N = 1 << 17
GRID_M = 2 ** np.arange(15)


def grid_series():
    """Two 'freq' series on integer grids whose running sums pass 2^53 grid steps, even after the mean is removed:
    a drift plus noise (grid 2^-20) and a random walk (grid 2^-30).  Returns {name: (integer list, grid step)}."""
    rs = np.random.RandomState(7)
    k = np.arange(GRID_N)
    drift = (1 << 24) * k + rs.randint(-(1 << 12), 1 << 12, GRID_N)
    walk = np.cumsum(rs.randint(-(1 << 30), 1 << 30, GRID_N))
    return {"drift": ([int(v) for v in drift], 2.0 ** -20), "walk": ([int(v) for v in walk], 2.0 ** -30)}


def exact_stability(yi, ms, g):
    """'freq' deviations [4, n_m] (rate 1) of the series yi * g, from running sums and differences in Python integers;
    the only roundings are the float of an exact fraction and the square root."""
    X = np.concatenate([[0], np.cumsum(np.array(yi, dtype=object))])
    S = np.concatenate([[0], np.cumsum(X)])
    Nx = len(X)
    out = np.full((4, len(ms)), np.nan)
    for t, m in enumerate(int(m) for m in ms):
        na, nm, nh = Nx - 2 * m, Nx - 3 * m + 1, Nx - 3 * m
        if na > 0:
            d = X[2 * m:2 * m + na] - 2 * X[m:m + na] + X[:na]
            out[0, t] = math.sqrt(Fraction(int(np.dot(d, d)), 2 * m * m * na)) * g
        if nm > 0:
            d = S[3 * m:3 * m + nm] - 3 * S[2 * m:2 * m + nm] + 3 * S[m:m + nm] - S[:nm]
            out[1, t] = math.sqrt(Fraction(int(np.dot(d, d)), 2 * nm)) / (m * m) * g
            out[2, t] = m * out[1, t] / math.sqrt(3)
        if nh > 0:
            d = X[3 * m:3 * m + nh] - 3 * X[2 * m:2 * m + nh] + 3 * X[m:m + nh] - X[:nh]
            out[3, t] = math.sqrt(Fraction(int(np.dot(d, d)), 6 * m * m * nh)) * g
    return out


def cumsum_route(y, ms):
    """The host route as allantools computes it: phase = fp64 cumsum of the mean-removed series, then the
    differences (mdev by allantools' running form).  [4, n_m] like exact_stability."""
    x = np.concatenate([[0.0], np.cumsum(y - y.mean())])
    Nx = x.size
    out = np.full((4, len(ms)), np.nan)
    for t, m in enumerate(int(m) for m in ms):
        na, nh = Nx - 2 * m, Nx - 3 * m
        d = x[2 * m:2 * m + na] - 2 * x[m:m + na] + x[:na]
        out[0, t] = np.sqrt(np.sum(d * d) / (2 * m * m * na))
        d = x[3 * m:3 * m + nh] - 3 * x[2 * m:2 * m + nh] + 3 * x[m:m + nh] - x[:nh]
        out[3, t] = np.sqrt(np.sum(d * d) / (6 * m * m * nh))
        v = np.sum(x[2 * m:3 * m] - 2 * x[m:2 * m] + x[:m])
        va = v + np.cumsum(x[3 * m:3 * m + nh] - 3 * x[2 * m:2 * m + nh] + 3 * x[m:m + nh] - x[:nh])
        out[1, t] = np.sqrt((v * v + np.sum(va * va)) / (2.0 * m ** 4 * (nh + 1)))
        out[2, t] = m * out[1, t] / np.sqrt(3)
    return out


@pytest.fixture(scope="module")
def grid_cases():
    cases = {}
    for name, (yi, g) in grid_series().items():
        y = np.array(yi, dtype=np.float64) * g
        assert all(int(a) == b for a, b in zip(y / g, yi))  # the grid values are exact in fp64
        cases[name] = (y, exact_stability(yi, GRID_M, g))
    return cases


@pytest.fixture(scope="module")
def stab_core():
    out = os.path.join(tempfile.mkdtemp(prefix="dfk_stab_"), "libstab.so")
    src = os.path.join(ROOT, "tests", "host", "stability_harness.cpp")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-x", "c++", "-fPIC", "-shared", "-ffp-contract=off", "-mfma",
                           "-o", out, src])
    lib = ctypes.CDLL(out)
    vp = ctypes.c_void_p
    lib.sh_stability.argtypes = [vp, ctypes.c_int64, ctypes.c_int, vp, ctypes.c_int, ctypes.c_double, vp, vp]

    def run(y, ms, data_type="freq", fs=1.0):
        y, ms = np.ascontiguousarray(y, dtype=np.float64), np.ascontiguousarray(ms, dtype=np.int64)
        dev, n = np.zeros((4, ms.size)), np.zeros((4, ms.size), dtype=np.int64)
        lib.sh_stability(y.ctypes.data, y.size, int(data_type == "freq"), ms.ctypes.data, ms.size, float(fs),
                         dev.ctypes.data, n.ctypes.data)
        return dev, n
    return run


@pytest.mark.parametrize("name", ["drift", "walk"])
def test_host_core_is_exact_where_cumsum_is_not(grid_cases, stab_core, name):
    y, ex = grid_cases[name]
    miss = np.max(np.abs(cumsum_route(y, GRID_M) / ex - 1))
    assert miss >= 1e-9, miss  # the case has teeth: the fp64 route loses the differences
    dev, n = stab_core(y, GRID_M)
    assert np.max(np.abs(dev / ex - 1)) <= 1e-13, np.abs(dev / ex - 1).max(axis=1)


def test_host_core_matches_reference(stab_core):
    rs = np.random.RandomState(2)
    for data_type in ("phase", "freq"):
        v = np.cumsum(rs.randn(20000)) + 5.0
        ref = ref_stability(v, 7.0, KINDS, "octave", data_type)
        dev, n = stab_core(v, ref["m"], data_type, 7.0)
        for i, k in enumerate(KINDS):
            _close(dev[i], ref[k][0], 1e-11)
            assert np.array_equal(n[i], ref[k + "_n"])


# ---------------------------------------------------------------------------------------------------------------------
# arguments
BAD_CALLS = [dict(kinds=()), dict(kinds=("oadev", "adev")), dict(kinds="allan"), dict(taus="log10"),
             dict(taus=[]), dict(taus=[1.0, -2.0]), dict(taus=[np.nan]), dict(taus=[[1.0, 2.0]]), dict(taus=["a"]),
             dict(data_type="frequency"), dict(data_type=None), dict(fs=0.0), dict(fs=np.inf), dict(fs=-1.0),
             dict(x=np.zeros(2)), dict(x=np.zeros(1), data_type="freq"), dict(x=np.zeros((2, 3, 10))),
             dict(x=np.zeros((0, 10))), dict(x=np.zeros(10), taus=[100.0]), dict(x=np.zeros(5), kinds="ohdev",
                                                                                   taus=[2.0])]


@pytest.mark.parametrize("kw", BAD_CALLS)
def test_argument_errors_before_device_work(monkeypatch, kw):
    from deepfmkit_b200 import _lib, stability

    def no_device(*a, **k):
        raise AssertionError("device work before the argument check")
    monkeypatch.setattr(_lib, "get_context", no_device)
    kw = dict(kw)
    x = kw.pop("x", np.zeros(100))
    fs = kw.pop("fs", 1.0)
    with pytest.raises(ValueError):
        stability(x, fs, **kw)


def test_entry_is_declared_and_bound():
    from deepfmkit_b200 import _lib
    with open(os.path.join(ROOT, "include", "dfk_b200.h")) as f:
        assert "int dfk_stability_dev(" in f.read()
    assert len(_lib.SYMBOLS["dfk_stability_dev"][1]) == 13
    import deepfmkit_b200 as dfk
    for name in ("stability", "oadev", "mdev", "tdev", "ohdev"):
        assert name in dfk.__all__ and callable(getattr(dfk, name))
    assert callable(dfk.DeepFitObject.calc_stability)


def launches(kinds, data_type):
    """The launch count dfk_stability_dev documents."""
    return 2 + (3 if data_type == "freq" else 1) + (3 if {"mdev", "tdev"} & set(kinds) else 0)


# ---------------------------------------------------------------------------------------------------------------------
# GPU
@pytest.fixture(scope="module")
def torch_mod():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _same(a, b, kinds=KINDS):
    assert np.array_equal(a["m"], b["m"]) and np.array_equal(a["taus"], b["taus"])
    for k in kinds:
        for s in ("", "_err", "_n"):
            assert np.array_equal(a[k + s], b[k + s], equal_nan=True), k + s


@pytest.mark.gpu
@pytest.mark.parametrize("data_type", ["phase", "freq"])
@pytest.mark.parametrize("taus", TAU_RULES, ids=["octave", "decade", "all", "explicit"])
def test_matches_reference(torch_mod, data_type, taus):
    from deepfmkit_b200 import stability
    rs = np.random.RandomState(17)
    N = 600 if taus == "all" else 30011
    v = np.cumsum(rs.randn(3, N), axis=1) + 0.5 * rs.randn(3, N) + 1e3
    got = stability(v, 4.0, KINDS, taus, data_type)
    ref = ref_stability(v, 4.0, KINDS, taus, data_type)
    assert np.array_equal(got["m"], ref["m"]) and np.allclose(got["taus"], ref["taus"], rtol=0, atol=0)
    for k in KINDS:
        _close(got[k], ref[k], 1e-11)
        _close(got[k + "_err"], ref[k + "_err"], 1e-11)
        assert np.array_equal(got[k + "_n"], ref[k + "_n"])
    assert np.allclose(got["tdev"], got["taus"] * got["mdev"] / np.sqrt(3), rtol=1e-15, atol=0, equal_nan=True)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["drift", "walk"])
def test_exact_on_grid_series(torch_mod, grid_cases, name):
    from deepfmkit_b200 import stability
    y, ex = grid_cases[name]
    got = stability(y, 1.0, KINDS, [float(m) for m in GRID_M], "freq")
    assert np.array_equal(got["m"], GRID_M)
    for i, k in enumerate(KINDS):
        assert np.max(np.abs(got[k] / ex[i] - 1)) <= 1e-13, (k, np.abs(got[k] / ex[i] - 1).max())


@pytest.mark.gpu
def test_hadamard_ignores_drift(torch_mod):
    from deepfmkit_b200 import stability
    rs = np.random.RandomState(4)
    N = 100_000
    y = rs.randn(N)
    a = 1e-3
    base = stability(y, 1.0, ("oadev", "ohdev"), data_type="freq")
    drift = stability(y + a * np.arange(N), 1.0, ("oadev", "ohdev"), data_type="freq")
    _close(drift["ohdev"], base["ohdev"], 1e-12)
    assert np.all(drift["oadev"][-4:] > 2 * base["oadev"][-4:])


@pytest.mark.gpu
def test_bit_identity(torch_mod):
    """A channel alone and in a batch of 256; a stride-8 column of a row table and a contiguous copy; a tensor and
    numpy; a repeated call; one tau alone and inside the octave list."""
    torch = torch_mod
    from deepfmkit_b200 import stability
    rs = np.random.RandomState(9)
    N = 50_007
    batch = np.cumsum(rs.randn(256, N), axis=1) + rs.randn(256, N)
    for data_type in ("phase", "freq"):
        whole = stability(batch, 50.0, data_type=data_type)
        one = stability(batch[137], 50.0, data_type=data_type)
        for k in KINDS:
            assert np.array_equal(one[k], whole[k][137], equal_nan=True)
        table = torch.zeros((N, 8), dtype=torch.float64, device="cuda")
        table[:, 2] = torch.from_numpy(batch[137]).cuda()
        col = stability(table[:, 2], 50.0, data_type=data_type)
        assert table[:, 2].stride() == (8,)
        _same(col, one)
        _same(stability(torch.from_numpy(batch[137]).cuda(), 50.0, data_type=data_type), one)
        _same(stability(batch[137], 50.0, data_type=data_type), one)
        for t, m in enumerate(one["m"]):
            alone = stability(batch[137], 50.0, taus=[m / 50.0], data_type=data_type)
            assert np.array_equal(alone["m"], [m])
            for k in KINDS:
                assert np.array_equal(alone[k], one[k][t:t + 1], equal_nan=True), (k, m)


@pytest.mark.gpu
def test_edge_cases(torch_mod):
    from deepfmkit_b200 import mdev, oadev, ohdev, stability, tdev
    rs = np.random.RandomState(1)
    # a NaN sample poisons its own channel only, for both data types and wherever it falls
    v = rs.randn(4, 5000)
    v[1, 2500] = np.nan
    v[3, 0] = np.nan
    for data_type in ("phase", "freq"):
        got = stability(v, 1.0, taus="all", data_type=data_type)
        ref = ref_stability(v[[0, 2]], 1.0, KINDS, "all", data_type)
        for k in KINDS:
            assert np.all(np.isnan(got[k][[1, 3]]))
            _close(got[k][[0, 2]], ref[k], 1e-11)
    # m inside oadev's range but outside mdev's and ohdev's: NaN and n = 0 there
    x = rs.randn(10)
    got = stability(x, 1.0, taus="all")
    assert list(got["m"]) == [1, 2, 3, 4]
    assert list(got["oadev_n"]) == [8, 6, 4, 2] and list(got["mdev_n"]) == [8, 5, 2, 0]
    assert list(got["ohdev_n"]) == [7, 4, 1, 0]
    assert np.all(np.isfinite(got["oadev"])) and np.isnan(got["mdev"][3]) and np.isnan(got["tdev"][3])
    assert np.isnan(got["ohdev"][3]) and np.isnan(got["ohdev_err"][3])
    _close(got["ohdev"][:3], ref_stability(x, 1.0, KINDS, "all")["ohdev"][0, :3], 1e-11)
    # Nx = 3: three phase points, or two frequency samples
    for data, dt in ((np.array([0.0, 1.0, 5.0]), "phase"), (np.array([1.0, 4.0]), "freq")):
        got = stability(data, 1.0, data_type=dt)
        ref = ref_stability(data, 1.0, KINDS, "octave", dt)
        assert list(got["m"]) == [1] and got["oadev_n"][0] == 1 and got["mdev_n"][0] == 1 and got["ohdev_n"][0] == 0
        for k in KINDS:
            _close(got[k], ref[k][0], 1e-15)
    # one long series
    y = rs.randn(1_800_000)
    got = stability(y, 50.0, data_type="freq")
    ref = ref_stability(y, 50.0, KINDS, [m / 50.0 for m in got["m"][::4]], "freq")
    for k in KINDS:
        _close(got[k][::4], ref[k][0], 1e-11)
    # the one-kind forms
    for fn, k in ((oadev, "oadev"), (mdev, "mdev"), (tdev, "tdev"), (ohdev, "ohdev")):
        taus, dev, err, n = fn(x, rate=2.0)
        alone = stability(x, 2.0, kinds=(k,))
        assert np.array_equal(taus, alone["taus"]) and np.array_equal(dev, alone[k])
        assert np.array_equal(err, alone[k + "_err"], equal_nan=True) and np.array_equal(n, alone[k + "_n"])


@pytest.mark.gpu
def test_launch_count(torch_mod):
    torch = torch_mod
    from deepfmkit_b200 import _lib
    ctx = _lib.get_context(0)
    v = torch.from_numpy(np.random.RandomState(0).randn(3, 10_000)).cuda()
    ms = np.array([1, 2, 4, 3000], dtype=np.int64)
    for data_type, code in (("phase", _lib.STAB_PHASE), ("freq", _lib.STAB_FREQ)):
        for mask in range(1, 16):
            kinds = [k for k in KINDS if mask & _lib.STAB_BITS[k]]
            n0 = ctx.launch_count()
            dev, n = ctx.stability_dev(v.data_ptr(), 10_000, 1, 3, 10_000, 1.0, code, mask, ms)
            assert ctx.launch_count() - n0 == launches(kinds, data_type), (data_type, kinds)
            for i, k in enumerate(KINDS):  # slots of kinds not requested are left as they were
                assert np.all(np.isnan(dev[i])) if k not in kinds else np.all(np.isfinite(dev[i][:, 0]))


@pytest.mark.gpu
def test_c_abi_rejects_bad_arguments(torch_mod):
    torch = torch_mod
    from deepfmkit_b200 import _lib
    ctx = _lib.get_context(0)
    v = torch.zeros(100, dtype=torch.float64, device="cuda")
    ok = dict(v_ptr=v.data_ptr(), N=100, stride=1, C=1, ld_c=100, fs=1.0, data_type=0, kinds=1, m=[1])
    for bad in (dict(v_ptr=None), dict(C=0), dict(stride=0), dict(N=2), dict(N=1, data_type=1), dict(kinds=0),
                dict(kinds=16), dict(data_type=2), dict(m=[1, 0]), dict(m=[]), dict(fs=0.0)):
        kw = {**ok, **bad}
        with pytest.raises(RuntimeError, match="error -1"):
            ctx.stability_dev(**kw)


@pytest.mark.gpu
def test_facade_calc_stability(torch_mod):
    from deepfmkit_b200 import stability
    from tests.test_wiener import _fitted_pair
    fm, _, _ = _fitted_pair(seconds=1.0)
    got = fm.calc_stability()
    _same(got, stability(fm.phi, fm.fs, data_type="freq"))
    two = fm.calc_stability(column="amp", kinds=("oadev",), taus="decade")
    _same(two, stability(fm.amp, fm.fs, kinds=("oadev",), taus="decade", data_type="freq"), kinds=("oadev",))
    assert fm.f is None
