"""Per-buffer parameter uncertainties of the NLS readout: s^2 (J^T J)^-1 at each fitted row, s^2 = ssq / (2N - 4).

CPU: the host build of dfk::fit_covariance against the oracle's 4x4 J^T J, its degenerate cases, and the options the
covariance does not support.  GPU: dfk_lm_cov, every _cov record entry (rows bit-identical to the plain entry,
covariance bit-identical to dfk_lm_cov on the same harmonic vectors), launch counts, calibration against the scatter
of a Monte-Carlo sweep and the Cramer-Rao bound, and the fitter / facade columns.
"""
import ctypes
import os
import subprocess
import tempfile

import numpy as np
import pytest

from oracle import dfmi_oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
c_double_p = ctypes.POINTER(ctypes.c_double)

# fixtures that carry harmonic vectors and the reference's fitted rows
FIXTURES = ["cfg1_quickstart", "cfg2_1mhz", "cfg3_channel", "deep_mod_n62", "fallback_m16", "pathological_m3", "low_snr",
            "drift_phi_slow", "full_cfg1", "full_cfg2_first", "cfg5_crlb"]
BLOCK = [(0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2), (3, 3)]  # covariance row entries 0..6 in the 4x4 matrix
DIAG = {0: 0, 3: 1, 5: 2, 6: 3}  # entry -> parameter index of the diagonal entries


def _ptr(a):
    return a.ctypes.data_as(c_double_p)


def fixture_qi_rows(golden, name):
    """(N, qi [nfit, 2N], rows [nfit, 8]) of a golden fixture: the reference's harmonic vectors and fitted rows."""
    g = golden(name)
    qi = np.ascontiguousarray(g["qi"].reshape(-1, g["qi"].shape[-1]))
    ref = (g["rows"] if name == "cfg5_crlb" else g["rows_seq"]).reshape(-1, 7)
    rows = np.zeros((len(ref), 8))
    rows[:, :7] = ref
    return qi.shape[1] // 2, qi, rows


def oracle_cov(N, qi, row):
    """The oracle's full 4x4 s^2 inv(J^T J) at the row's parameters, and s^2."""
    s2 = row[5] / (2 * N - 4)
    _, jtj, _ = orc.model_state(N, qi, row[:4])
    return np.linalg.inv(jtj) * s2, s2


def assert_cov_gates(N, qi, rows, cov):
    """Diagonal within 1e-10 relative, block off-diagonals within 1e-10 sqrt(C_ii C_jj), s^2 bit-equal, and the oracle's
    psi cross terms (not stored) at most 1e-10 of sqrt(C_psipsi C_ii)."""
    for f in range(len(rows)):
        ref, s2 = oracle_cov(N, qi[f], rows[f])
        assert cov[f, 7] == s2, (f, cov[f, 7], s2)
        d = np.diag(ref)
        for k, (i, j) in enumerate(BLOCK):
            tol = 1e-10 * (abs(ref[i, i]) if i == j else np.sqrt(d[i] * d[j]))
            assert abs(cov[f, k] - ref[i, j]) <= tol, (f, k, cov[f, k], ref[i, j])
        for i in range(3):
            assert abs(ref[3, i]) <= 1e-10 * np.sqrt(d[3] * d[i]) and abs(ref[i, 3]) <= 1e-10 * np.sqrt(d[3] * d[i])


# ---------------------------------------------------------------------------------------------------
# CPU: the host build of the core
@pytest.fixture(scope="module")
def cov_core():
    out = os.path.join(tempfile.mkdtemp(prefix="dfk_cov_"), "libcov.so")
    src = os.path.join(ROOT, "tests", "host", "cov_harness.cpp")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-x", "c++", "-fPIC", "-shared", "-ffp-contract=off", "-mfma",
                           "-o", out, src])
    lib = ctypes.CDLL(out)
    lib.hh_fit_covariance.argtypes = [ctypes.c_int, ctypes.c_longlong, c_double_p, c_double_p, ctypes.c_int, c_double_p]

    def run(N, qi, rows):
        qi = np.ascontiguousarray(qi, dtype=np.float64).reshape(len(rows), 2 * N)
        rows = np.ascontiguousarray(rows, dtype=np.float64)
        cov = np.full((len(rows), 8), -123.0)
        lib.hh_fit_covariance(N, len(rows), _ptr(qi), _ptr(rows), rows.shape[1], _ptr(cov))
        return cov
    return run


@pytest.mark.parametrize("name", FIXTURES)
def test_host_core_vs_oracle(cov_core, golden, name):
    N, qi, rows = fixture_qi_rows(golden, name)
    assert_cov_gates(N, qi, rows, cov_core(N, qi, rows))


def _model_qi(N, p):
    """Noise-free harmonic vector of the model at p (fit.py:111-114)."""
    from scipy.special import jv
    a, m, phi, psi = p
    j = np.arange(1, N + 1)
    env = a * np.cos(phi + j * np.pi / 2) * jv(j, m)
    return np.concatenate([env * np.cos(j * psi), -env * np.sin(j * psi)])


def test_host_core_degenerate_cases(cov_core):
    p = [1.1, 6.0, 0.3, 0.2]
    rng = np.random.RandomState(3)
    N = 10
    qi = _model_qi(N, p) + 1e-4 * rng.standard_normal(2 * N)
    row = np.array(p + [0.0, 2.5e-7, 0.0, 5.0])
    # a = 0: the amplitude column vanishes, so does the psi column (its entries carry a): only s^2 survives
    c = cov_core(N, qi, np.array([[0.0, 6.0, 0.3, 0.2, 0.0, 2.5e-7, 0.0, 0.0]]))[0]
    assert np.all(np.isnan(c[:7])) and c[7] == 2.5e-7 / 16
    # 2N - 4 <= 0: nothing to estimate the noise from
    for n in (1, 2):
        c = cov_core(n, qi[:2 * n], row[None, :])[0]
        assert np.all(np.isnan(c)), (n, c)
    # a non-finite parameter
    for k in range(4):
        for bad in (np.nan, np.inf):
            r = row.copy()
            r[k] = bad
            assert np.all(np.isnan(cov_core(N, qi, r[None, :])[0])), (k, bad)
    # noise-free input: zeros, not -0
    c = cov_core(N, _model_qi(N, p), np.array([p + [0.0, 0.0, 0.0, 0.0]]))[0]
    assert np.all(c == 0.0) and not np.any(np.signbit(c))
    # the largest harmonic count: finite, and the oracle's numbers
    N = 64
    p = [1.0, 30.0, -0.4, 0.1]
    qi = _model_qi(N, p) + 1e-5 * rng.standard_normal(2 * N)
    rows = np.array([p + [0.0, orc.residual_ssq(N, qi, np.array(p)), 0.0, 0.0]])
    c = cov_core(N, qi, rows)
    assert np.all(np.isfinite(c)) and np.all(c[0, [0, 3, 5, 6, 7]] > 0)
    assert_cov_gates(N, qi[None, :], rows, c)
    c = cov_core(N, _model_qi(N, p), np.array([p + [0.0, 0.0, 0.0, 0.0]]))[0]
    assert np.all(c == 0.0)


def test_unsupported_uncertainty_options_raise():
    """The EKF and the multi-GPU sweep have no covariance: asking for one is an error, before any device work."""
    from deepfmkit_b200 import DeepRawObject, EKFFitter
    from deepfmkit_b200.montecarlo import nls_sweep_sharded
    raw = DeepRawObject(data=np.ones(8000), f_samp=200e3, f_mod=1000)
    with pytest.raises(ValueError, match="NLS"):
        EKFFitter({"n": 20}).fit(raw, uncertainties=True)
    with pytest.raises(ValueError, match="single-GPU"):
        nls_sweep_sharded([6.0], 10, uncertainties=True)


# ---------------------------------------------------------------------------------------------------
# GPU
@pytest.fixture(scope="module")
def torch_mod():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


@pytest.fixture(scope="module")
def ctx(torch_mod):
    from deepfmkit_b200 import _lib
    c = _lib.Context(0)
    yield c
    c.close()


def dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).cuda()


def lm_cov(torch, ctx, qi, rows, N):
    """dfk_lm_cov on device tensors (or host arrays) -> host [nfit, 8]."""
    qi_d, rows_d = (t if isinstance(t, torch.Tensor) else dev(torch, t) for t in (qi, rows))
    n = rows_d.numel() // 8
    cov = torch.empty((n, 8), dtype=torch.float64, device="cuda")
    ctx.lm_cov(qi_d.data_ptr(), n, N, rows_d.data_ptr(), cov.data_ptr())
    ctx.synchronize()
    return cov.cpu().numpy()


def demod(torch, ctx, xd, nbuf, R, N, w0):
    qi = torch.empty((nbuf, 2 * N), dtype=torch.float64, device="cuda")
    dc = torch.empty(nbuf, dtype=torch.float64, device="cuda")
    ctx.demod(xd.data_ptr(), nbuf, R, N, w0, qi.data_ptr(), dc.data_ptr())
    return qi


@pytest.mark.gpu
@pytest.mark.parametrize("name", FIXTURES)
def test_standalone_entry_vs_oracle(torch_mod, ctx, golden, name):
    N, qi, rows = fixture_qi_rows(golden, name)
    assert_cov_gates(N, qi, rows, lm_cov(torch_mod, ctx, qi, rows, N))


def _record(golden, name):
    """(x, R, N, w0) of a golden record."""
    from tests.test_oracle_golden import _signal_from_meta
    g = golden(name)
    if name.startswith("drift"):
        m, fs, fm, secs, trial, amp_n, aamp, af = g["meta"]
        x, _ = orc.asd_signal(m, fs, fm, secs, trial=int(trial), amp_n=amp_n, arml_mod_amp=aamp, arml_mod_f=af)
        N = g["qi"].shape[1] // 2
        R = len(x) // len(g["qi"])
    else:
        meta = g["meta"]
        x = g["x"] if "x" in g.files else _signal_from_meta(meta)
        fs, fm, N = meta[1], meta[2], int(meta[9])
        R = int(fs / fm * meta[8])
    return np.ascontiguousarray(x[: (len(x) // R) * R]), R, N, orc.rad_per_sample(fs, fm)


def _dev_pair(torch, ctx, xd, nbuf, R, N, w0, seeded, init=(1.6, 6.0, 0.0, 0.0)):
    """Rows of dfk_nls_fit_dev, rows and cov of dfk_nls_fit_cov_dev, and the launches each issued."""
    rows0 = torch.empty((nbuf, 8), dtype=torch.float64, device="cuda")
    rows1 = torch.empty_like(rows0)
    cov = torch.empty_like(rows0)
    n0 = ctx.launch_count()
    ctx.nls_fit_dev(xd.data_ptr(), nbuf, R, N, w0, init, seeded, None, rows0.data_ptr())
    n1 = ctx.launch_count()
    ctx.nls_fit_dev(xd.data_ptr(), nbuf, R, N, w0, init, seeded, None, rows1.data_ptr(), cov_ptr=cov.data_ptr())
    n2 = ctx.launch_count()
    ctx.synchronize()
    return rows0.cpu().numpy(), rows1, cov.cpu().numpy(), n1 - n0, n2 - n1


@pytest.mark.gpu
@pytest.mark.parametrize("seeded", [0, 1, 3, -1])
@pytest.mark.parametrize("name", ["cfg1_quickstart", "drift_phi_slow"])
def test_record_entry_matches_standalone(torch_mod, ctx, golden, name, seeded):
    x, R, N, w0 = _record(golden, name)
    nbuf = len(x) // R
    xd = dev(torch_mod, x)
    rows0, rows1, cov, l0, l1 = _dev_pair(torch_mod, ctx, xd, nbuf, R, N, w0, seeded)
    assert np.array_equal(rows0.view(np.int64), rows1.cpu().numpy().view(np.int64))
    assert l1 == l0 + 1
    qi = demod(torch_mod, ctx, xd, nbuf, R, N, w0)
    ref = lm_cov(torch_mod, ctx, qi, rows1, N)
    assert np.array_equal(cov.view(np.int64), ref.view(np.int64))
    ok = rows0[:, 6] < 2
    assert ok.sum() >= nbuf // 2
    assert_cov_gates(N, qi.cpu().numpy()[ok], rows0[ok], cov[ok])


@pytest.mark.gpu
def test_direct_path_record(torch_mod, ctx):
    """f_mod off the sample grid: the record takes the direct (non-folding) lock-in."""
    from deepfmkit_b200 import _lib
    fs, fm, n, N = 200e3, 1234.5, 20, 10
    R = int(fs / fm * n)
    w0 = 2 * np.pi * fm / fs
    assert _lib.demod_path(R, w0) == 0
    nbuf = 40
    xd = torch_mod.empty(nbuf * R, dtype=torch_mod.float64, device="cuda")
    ctx.synth_snr_dev(xd.data_ptr(), nbuf * R, 1, fs, fm, 6.0, snr_db=40.0, seed=11)
    rows0, rows1, cov, l0, l1 = _dev_pair(torch_mod, ctx, xd, nbuf, R, N, w0, True)
    assert np.array_equal(rows0.view(np.int64), rows1.cpu().numpy().view(np.int64)) and l1 == l0 + 1
    qi = demod(torch_mod, ctx, xd, nbuf, R, N, w0)
    assert np.array_equal(cov.view(np.int64), lm_cov(torch_mod, ctx, qi, rows1, N).view(np.int64))
    assert_cov_gates(N, qi.cpu().numpy(), rows0, cov)


@pytest.mark.gpu
def test_batch_with_per_channel_guess(torch_mod, ctx):
    from deepfmkit_b200 import nls_fit_batch
    R, N, bpc = 4000, 10, 12
    w0 = orc.rad_per_sample(200e3, 1000.0)
    ms = np.array([4.0, 6.0, 9.0, 13.0])
    x = np.stack([orc.snr_signal(float(m), 200e3, 1000.0, bpc * R / 200e3, 40.0, seed=c, phi0=0.4 * c)[: bpc * R]
                  for c, m in enumerate(ms)])
    rows0 = nls_fit_batch(x, 200e3, 1000.0, 20, init_m=ms)
    rows, cov = nls_fit_batch(x, 200e3, 1000.0, 20, init_m=ms, return_cov=True)
    assert cov.shape == (4, bpc, 8)
    assert np.array_equal(rows0.view(np.int64), rows.view(np.int64))
    qi = demod(torch_mod, ctx, dev(torch_mod, x), 4 * bpc, R, N, w0)
    ref = lm_cov(torch_mod, ctx, qi, rows.reshape(-1, 8), N)
    assert np.array_equal(cov.reshape(-1, 8).view(np.int64), ref.view(np.int64))
    assert np.all(rows[..., 6] == 0)
    assert_cov_gates(N, qi.cpu().numpy(), rows.reshape(-1, 8), cov.reshape(-1, 8))


@pytest.mark.gpu
def test_time_major_batch(torch_mod, ctx):
    from deepfmkit_b200 import nls_fit_batch
    R, N, bpc, C = 4000, 10, 6, 8
    w0 = orc.rad_per_sample(200e3, 1000.0)
    x = np.stack([orc.snr_signal(6.0, 200e3, 1000.0, bpc * R / 200e3, 40.0, seed=c, phi0=0.7 * c)[: bpc * R]
                  for c in range(C)], 1)  # [T, C]
    xd = dev(torch_mod, x)
    rows0 = nls_fit_batch(xd, 200e3, 1000.0, 20, time_major=True, return_tensor=True)
    rows, cov = nls_fit_batch(xd, 200e3, 1000.0, 20, time_major=True, return_tensor=True, return_cov=True)
    assert isinstance(cov, torch_mod.Tensor) and tuple(cov.shape) == (C, bpc, 8)
    assert torch_mod.equal(rows0, rows)
    qi = torch_mod.empty((C * bpc, 2 * N), dtype=torch_mod.float64, device="cuda")
    dc = torch_mod.empty(C * bpc, dtype=torch_mod.float64, device="cuda")
    ctx.demod_tm(xd.data_ptr(), bpc, C, R, N, w0, qi.data_ptr(), dc.data_ptr())
    ref = lm_cov(torch_mod, ctx, qi, rows, N)
    assert np.array_equal(cov.cpu().numpy().reshape(-1, 8).view(np.int64), ref.view(np.int64))


@pytest.mark.gpu
@pytest.mark.parametrize("pinned", [False, True])
def test_host_entry_over_slabs(torch_mod, ctx, golden, pinned):
    x, R, N, w0 = _record(golden, "full_cfg1")
    nbuf = len(x) // R
    if pinned:
        xp = torch_mod.empty(len(x), dtype=torch_mod.float64, pin_memory=True)
        xp.numpy()[:] = x
        x = xp.numpy()
    slab = 180  # buffers per slab: 500 buffers span three slabs
    ctx.set_host_slab_bytes(slab * R * 8)
    try:
        n0 = ctx.launch_count()
        rows0 = ctx.nls_fit_host(x, R, N, w0, [1.6, 6.0, 0.0, 0.0], seeded=True)
        n1 = ctx.launch_count()
        cov = np.empty((nbuf, 8))
        rows = ctx.nls_fit_host(x, R, N, w0, [1.6, 6.0, 0.0, 0.0], seeded=True, cov_out=cov)
        n2 = ctx.launch_count()
    finally:
        ctx.set_host_slab_bytes(0)
    assert np.array_equal(rows0.view(np.int64), rows.view(np.int64))
    assert n2 - n1 == (n1 - n0) + (nbuf + slab - 1) // slab
    qi = demod(torch_mod, ctx, dev(torch_mod, x), nbuf, R, N, w0).cpu().numpy()
    assert_cov_gates(N, qi, rows, cov)


@pytest.mark.gpu
def test_sweep_entry(torch_mod, ctx):
    from deepfmkit_b200 import _lib
    ms, nt, R, N = np.array([3.0, 6.0, 12.0]), 5000, 200, 15
    rows0 = torch_mod.empty((3, nt, 8), dtype=torch_mod.float64, device="cuda")
    rows = torch_mod.empty_like(rows0)
    cov = torch_mod.empty_like(rows0)
    kw = dict(phi0=0.3, snr_db=40.0, seed=7)
    n0 = ctx.launch_count()
    ctx.nls_sweep_dev(ms, nt, 0, nt, R, N, 200e3, 1000.0, rows0.data_ptr(), **kw)
    n1 = ctx.launch_count()
    ctx.nls_sweep_dev(ms, nt, 0, nt, R, N, 200e3, 1000.0, rows.data_ptr(), cov_ptr=cov.data_ptr(), **kw)
    n2 = ctx.launch_count()
    assert n2 - n1 == n1 - n0 + 1
    assert torch_mod.equal(rows0, rows)
    qi = torch_mod.empty((3, nt, 2 * N), dtype=torch_mod.float64, device="cuda")
    dc = torch_mod.empty((3, nt), dtype=torch_mod.float64, device="cuda")
    for i, m in enumerate(ms):
        ctx.sweep_demod_dev(nt, 0, R, N, 200e3, 1000.0, float(m), qi[i].data_ptr(), dc[i].data_ptr(), phi0=0.3,
                            snr_db=40.0, seed=7 + i * nt)
    ref = lm_cov(torch_mod, ctx, qi, rows, N)
    assert np.array_equal(cov.cpu().numpy().reshape(-1, 8).view(np.int64), ref.view(np.int64))
    r = rows.cpu().numpy().reshape(-1, 8)
    sel = np.arange(0, len(r), 97)
    assert_cov_gates(N, qi.cpu().numpy().reshape(-1, 2 * N)[sel], r[sel], cov.cpu().numpy().reshape(-1, 8)[sel])
    assert _lib.COV_STRIDE == 8


@pytest.mark.gpu
def test_predicted_errors_are_calibrated(torch_mod):
    """The predicted sigma of every parameter matches the scatter of 20 000 realisations, and at phi0 = 0 the bound."""
    from deepfmkit_b200 import nls_sweep
    out = nls_sweep([3.0, 6.0, 12.0], 20000, phi0=0.3, uncertainties=True, seed=3)
    for name in ("amp", "m", "phi", "psi"):
        ratio = out[f"{name}_err_rms"] / out[f"{name}_std"]
        assert np.all(np.abs(ratio - 1) < 0.03), (name, ratio)
    out = nls_sweep([6.0], 20000, phi0=0.0, uncertainties=True, seed=4, return_rows=True)
    assert abs(out["m_err_rms"][0] / out["crlb_sigma_m"][0] - 1) < 0.03
    assert out["cov"].shape == (1, 20000, 8) and out["rows"].shape == (1, 20000, 8)
    ok = out["rows"][0, :, 6] == 0
    assert np.isclose(out["m_err_rms"][0], np.sqrt(np.mean(out["cov"][0, ok, 3])), rtol=1e-2)


@pytest.mark.gpu
def test_fitter_columns(torch_mod, ctx):
    import pandas as pd
    from deepfmkit_b200 import DeepRawObject, StandardNLSFitter
    from deepfmkit_b200.fitters import RESULT_COLUMNS
    x = orc.snr_signal(6.0, 200e3, 1000, 0.5, 40.0, seed=2, phi0=0.3)
    R, N, w0 = 4000, 10, orc.rad_per_sample(200e3, 1000.0)
    nbuf = len(x) // R
    fitter = StandardNLSFitter({"n": 20})
    # host route
    raw = DeepRawObject(data=pd.DataFrame(x, columns=["ch0"]), f_samp=200e3, f_mod=1000)
    plain = fitter.fit(raw)
    assert list(plain.columns) == RESULT_COLUMNS
    assert [str(t) for t in plain.dtypes] == ["float64"] * 6 + ["int64"]
    df = fitter.fit(raw, uncertainties=True)
    assert list(df.columns) == RESULT_COLUMNS + ["amp_err", "m_err", "phi_err", "psi_err"]
    assert all(str(df[c].dtype) == "float64" for c in ("amp_err", "m_err", "phi_err", "psi_err"))
    pd.testing.assert_frame_equal(df[RESULT_COLUMNS], plain, check_exact=True)
    qi = demod(torch_mod, ctx, dev(torch_mod, x[: nbuf * R]), nbuf, R, N, w0).cpu().numpy()
    rows = np.zeros((nbuf, 8))
    rows[:, :7] = plain.to_numpy(dtype=float)
    for f in range(nbuf):
        ref, _ = oracle_cov(N, qi[f], rows[f])
        got = df.loc[f, ["amp_err", "m_err", "phi_err", "psi_err"]].to_numpy(dtype=float)
        assert np.all(np.abs(got ** 2 - np.diag(ref)) <= 1e-10 * np.diag(ref)), f
    # device-record route: the square roots of dfk_nls_fit_cov_dev's entries 0, 3, 5 and 6 on the same schedule
    xd = dev(torch_mod, x)
    draw = DeepRawObject(device_data=xd, f_samp=200e3, f_mod=1000)
    dplain = fitter.fit(draw)
    ddf = fitter.fit(draw, uncertainties=True)
    pd.testing.assert_frame_equal(ddf[RESULT_COLUMNS], dplain, check_exact=True)
    chunks = os.cpu_count() or 1
    rows_d = torch_mod.empty((nbuf, 8), dtype=torch_mod.float64, device="cuda")
    cov_d = torch_mod.empty_like(rows_d)
    ctx.nls_fit_dev(xd.data_ptr(), nbuf, R, N, w0, [1.6, 6.0, 0.0, 0.0], chunks, None, rows_d.data_ptr(),
                    cov_ptr=cov_d.data_ptr())
    cov = cov_d.cpu().numpy()
    for c, k in (("amp_err", 0), ("m_err", 3), ("phi_err", 5), ("psi_err", 6)):
        assert np.array_equal(ddf[c].to_numpy(), np.sqrt(cov[:, k])), c


@pytest.mark.gpu
def test_facade_uncertainties(torch_mod, tmp_path):
    import pandas as pd
    from deepfmkit_b200 import DeepFitFramework, DeepRawObject

    class _Laser:
        df = 1.5e9

    class _Sim:
        label = "ch"
        laser = _Laser()
        fit_n = 20

    x = orc.snr_signal(6.0, 200e3, 1000, 0.3, 40.0, seed=1)
    outs = {}
    for flag in (False, True):
        raw = DeepRawObject(data=pd.DataFrame(x, columns=["ch0"]), f_samp=200e3, f_mod=1000, label="ch")
        raw.sim = _Sim()
        dff = DeepFitFramework()
        dff.load_raw_object(raw)
        dff.sims["ch"] = raw.sim
        fobj = dff.fit("ch", uncertainties=flag) if flag else dff.fit("ch")
        dff.to_txt(str(tmp_path) + f"/{int(flag)}_")
        outs[flag] = (dff.fits_df["ch_nls"], fobj, open(str(tmp_path) + f"/{int(flag)}_ch_nls.txt", "rb").read())
    df0, f0, t0 = outs[False]
    df1, f1, t1 = outs[True]
    assert t0 == t1
    assert list(df1.columns) == list(df0.columns[:7]) + ["amp_err", "m_err", "phi_err", "psi_err", "tau", "tau_err"]
    assert np.array_equal(df1["tau_err"].to_numpy(), df1["m_err"].to_numpy() / (2 * np.pi * 1.5e9))
    for c in ("amp_err", "m_err", "phi_err", "psi_err", "tau_err"):
        assert getattr(f0, c) is None
        assert np.array_equal(getattr(f1, c), df1[c].to_numpy()), c
    assert np.array_equal(f1.tau, f0.tau)
    # without a simulation tau and its error are zero, as the reference forms tau
    raw = DeepRawObject(data=pd.DataFrame(x, columns=["ch0"]), f_samp=200e3, f_mod=1000, label="nosim")
    dff = DeepFitFramework()
    dff.load_raw_object(raw)
    fobj = dff.fit("nosim", n=20, uncertainties=True)
    assert np.all(fobj.tau_err == 0.0) and np.all(dff.fits_df["nosim_nls"]["tau_err"] == 0.0)
