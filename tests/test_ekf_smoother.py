"""EKF fixed-interval (Rauch-Tung-Striebel) smoother: dfk_ekf_smooth_dev / ekf_smooth / EKFFitter.fit(smooth=True).

CPU: the numpy reference ref_ekf_rts against a batch least-squares solve of the linearised model, the host build of
the smoother core (tests/host/smooth_harness.cpp) against the reference on the full_ekf_8ch records, the core's
invariants, and the argument errors.  GPU: filtered outputs bit-identical to dfk_ekf_dev, smoothed outputs against
the host core and the reference (also deep in time with a carried state, where the checked replay runs), bit-identity
over the checkpoint interval, channels per warp and runs, calibration against the truth on records drawn from the
model, and the edges (NaN samples, short windows, launch count, fitter and facade).
"""
import ctypes
import os
import subprocess
import tempfile
from multiprocessing import Pool

import numpy as np
import pytest

from oracle import dfmi_oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
c_double_p = ctypes.POINTER(ctypes.c_double)
F_SAMP, F_MOD = 200e3, 1000.0
Q_DEFAULT = np.asarray(orc.EKF_Q_DIAG, dtype=float)
# host core against the numpy reference over 2e5 steps: measured 1.4e-13 (states) and 1.6e-13 relative (variances)
STATE_TOL = 1e-11
VAR_RTOL = 1e-9


def _ptr(a):
    return a.ctypes.data_as(c_double_p)


def _tri(i, j):
    return i * 5 - (i * (i - 1)) // 2 + (j - i)


def _tri_of(P):
    return np.array([P[i, j] for i in range(5) for j in range(i, 5)])


def _full_of(tri):
    P = np.zeros((5, 5))
    for i in range(5):
        for j in range(i, 5):
            P[i, j] = P[j, i] = tri[_tri(i, j)]
    return P


# ---------------------------------------------------------------------------------------------------------------------
# numpy reference
def ref_ekf_forward(z, x0, P0, q, r, k0=0):
    """The oracle's filter (ekf_track's loop: full matrices, simple-form update) storing, per step k, x_f[k], P_f[k],
    the predicted state the measurement was linearised at and the Jacobian row H_k."""
    z = np.asarray(z, dtype=float)
    T = len(z)
    state = np.array(x0, dtype=float)
    cov = np.array(P0, dtype=float)
    qm = np.diag(q)
    w_m = 2 * np.pi * F_MOD
    t_axis = (int(k0) + np.arange(T)) / F_SAMP
    xf, Pf, xbar, H = np.empty((T, 5)), np.empty((T, 5, 5)), np.empty((T, 5)), np.empty((T, 5))
    for k in range(T):
        cov = cov + qm
        a, m, phi, psi, dc = state
        theta = w_m * t_axis[k] + psi
        arg = phi + m * np.cos(theta)
        s_arg = np.sin(arg)
        h = np.array([np.cos(arg), -a * s_arg * np.cos(theta), -a * s_arg, a * m * s_arg * np.sin(theta), 1.0])
        xbar[k], H[k] = state, h
        innov = z[k] - (a * np.cos(arg) + dc)
        ph = cov @ h
        s = h @ ph + r
        gain = ph / s
        state = state + gain * innov
        cov = cov - np.outer(gain, h @ cov)
        xf[k], Pf[k] = state, cov
    return xf, Pf, xbar, H


def ref_rts(xf, Pf, q):
    """The RTS recursion with numpy.linalg: G = P_f Pp^-1 by a batched solve, then the backward pass."""
    T = len(xf)
    Pp = Pf + np.diag(q)
    G = np.linalg.solve(np.swapaxes(Pp, 1, 2), np.swapaxes(Pf, 1, 2)).swapaxes(1, 2)
    xs, Ps = np.empty_like(xf), np.empty_like(Pf)
    xs[-1], Ps[-1] = xf[-1], Pf[-1]
    for k in range(T - 2, -1, -1):
        xs[k] = xf[k] + G[k] @ (xs[k + 1] - xf[k])
        Ps[k] = Pf[k] + G[k] @ (Ps[k + 1] - Pp[k]) @ G[k].T
    return xs, Ps


def ref_ekf_rts(z, x0, P0, q, r, k0=0):
    """(x_s, P_s, x_f, P_f) at every step of the window."""
    xf, Pf, _, _ = ref_ekf_forward(z, x0, P0, q, r, k0)
    xs, Ps = ref_rts(xf, Pf, q)
    return xs, Ps, xf, Pf


def _snap(a, R):
    n = len(a) // R
    return a[R - 1:n * R:R]


def _ref_snapshots(args):
    z, x0, P0, q, r, k0, R = args
    xs, Ps, xf, Pf = ref_ekf_rts(z, x0, P0, q, r, k0)
    d = lambda P: np.diagonal(_snap(P, R), axis1=1, axis2=2).copy()  # noqa: E731
    return _snap(xs, R), d(Ps), _snap(xf, R), d(Pf)


# ---------------------------------------------------------------------------------------------------------------------
# host core
@pytest.fixture(scope="module")
def core():
    out = os.path.join(tempfile.mkdtemp(prefix="dfk_smooth_"), "libsmooth.so")
    src = os.path.join(ROOT, "tests", "host", "smooth_harness.cpp")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-x", "c++", "-fPIC", "-shared", "-ffp-contract=off", "-mfma",
                           "-o", out, src])
    lib = ctypes.CDLL(out)
    lib.sh_smooth.argtypes = [c_double_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, ctypes.c_double,
                              ctypes.c_double, c_double_p, c_double_p, c_double_p, ctypes.c_double, ctypes.c_int64,
                              c_double_p, c_double_p, c_double_p, c_double_p]

    def run(z, R, x0, P0, q, r, B=1024, k0=0):
        """(xs, vs, xf, vf) at the snapshots, [nbuf, 5] each; P0 a full 5x5 matrix."""
        z = np.ascontiguousarray(z, dtype=np.float64)
        nbuf = len(z) // R
        outs = [np.full((nbuf, 5), -1.0) for _ in range(4)]
        lib.sh_smooth(_ptr(z), len(z), R, k0, F_SAMP, F_MOD, _ptr(np.asarray(x0, dtype=float)), _ptr(_tri_of(P0)),
                      _ptr(np.asarray(q, dtype=float)), float(r), B, *[_ptr(o) for o in outs])
        return tuple(outs)
    return run


def _default_prior(z):
    return np.array([1.6, 6.0, 0.0, 0.0, np.mean(z)]), np.eye(5), Q_DEFAULT, float(np.var(z))


def _full_ekf_records(golden):
    g = golden("full_ekf_8ch")
    return [orc.snr_signal(6.0, F_SAMP, F_MOD, 1.0, 40.0, seed=int(c), phi0=2 * np.pi * c / 4096) for c in g["channels"]]


# ---- 1. the reference is the batch solve -----------------------------------------------------------------------------
def test_reference_equals_batch_solve():
    """RTS over the filter's x_f, P_f is the posterior of the linear-Gaussian problem: prior x_0 ~ N(x0, P0 + Q) (the
    filter's first prediction), increments x_k - x_(k-1) ~ N(0, Q), and the measurement linearised at the filter's
    predicted states, y_k = z_k - h(xbar_k) + H_k xbar_k = H_k x_k + v_k, v_k ~ N(0, r).  Solved here as one dense
    1000-unknown system; means and covariance blocks agree to rounding (an identity, not an approximation)."""
    z = orc.snr_signal(6.0, F_SAMP, F_MOD, 0.001, 30.0, seed=11)
    T = len(z)
    assert T == 200
    x0, P0, q, r = _default_prior(z)
    xf, Pf, xbar, H = ref_ekf_forward(z, x0, P0, q, r)
    xs, Ps = ref_rts(xf, Pf, q)
    n = 5 * T
    lam, eta = np.zeros((n, n)), np.zeros(n)
    pi = np.linalg.inv(P0 + np.diag(q))
    lam[:5, :5] += pi
    eta[:5] += pi @ x0
    qi = np.diag(1.0 / q)
    for k in range(1, T):
        a, b = slice(5 * k - 5, 5 * k), slice(5 * k, 5 * k + 5)
        lam[a, a] += qi
        lam[b, b] += qi
        lam[a, b] -= qi
        lam[b, a] -= qi
    for k in range(T):
        a, m, phi, psi, dc = xbar[k]
        theta = 2 * np.pi * F_MOD * (k / F_SAMP) + psi
        hx = a * np.cos(phi + m * np.cos(theta)) + dc
        y = z[k] - hx + H[k] @ xbar[k]
        b = slice(5 * k, 5 * k + 5)
        lam[b, b] += np.outer(H[k], H[k]) / r
        eta[b] += H[k] * y / r
    # cond(lam) ~ 1e9 (Q^-1 = 1e8 beside 1/r ~ 2): rounding alone moves either solution by up to cond eps |x|
    bound = np.linalg.cond(lam) * np.finfo(float).eps
    cov = np.linalg.inv(lam)
    mean = np.linalg.solve(lam, eta)
    mean_dev = np.max(np.abs(mean.reshape(T, 5) - xs))
    blocks = np.stack([cov[5 * k:5 * k + 5, 5 * k:5 * k + 5] for k in range(T)])
    scale = np.sqrt(np.einsum("kii,kjj->kij", blocks, blocks))
    cov_dev = np.max(np.abs(blocks - Ps) / scale)
    # the RTS means solve the normal equations as well as the direct solve does
    res_rts = np.linalg.norm(lam @ xs.ravel() - eta) / np.linalg.norm(eta)
    res_dir = np.linalg.norm(lam @ mean - eta) / np.linalg.norm(eta)
    print(f"batch solve vs RTS over {T} steps (cond eps = {bound:.1e}): means {mean_dev:.2e}, covariances "
          f"{cov_dev:.2e} of sqrt(C_ii C_jj); normal-equation residuals {res_rts:.1e} (RTS), {res_dir:.1e} (solve)")
    assert mean_dev < bound * np.max(np.abs(xs)), (mean_dev, bound)
    assert cov_dev < bound, (cov_dev, bound)
    assert res_rts < 10 * res_dir, (res_rts, res_dir)


# ---- 2. host core against the reference ------------------------------------------------------------------------------
def test_core_vs_reference(core, golden):
    """The host-compiled core (ekf_step + rts_step, checkpointed as on the device) against ref_ekf_rts on the
    full_ekf_8ch channels' 2e5-step records (R = 4000: 50 snapshots each).  Gates: states STATE_TOL absolute,
    variances VAR_RTOL relative, each at least 10x the deviation measured here (printed)."""
    recs = _full_ekf_records(golden)
    R = 4000
    jobs = [(z, *_default_prior(z), 0, R) for z in recs]
    with Pool(min(len(jobs), os.cpu_count() or 1)) as pool:
        refs = pool.map(_ref_snapshots, jobs)
    dx = dv = dxf = dvf = 0.0
    for z, (xs_r, vs_r, xf_r, vf_r) in zip(recs, refs):
        xs, vs, xf, vf = core(z, R, *_default_prior(z))
        dx = max(dx, np.max(np.abs(xs - xs_r)))
        dv = max(dv, np.max(np.abs(vs - vs_r) / vs_r))
        dxf = max(dxf, np.max(np.abs(xf - xf_r)))
        dvf = max(dvf, np.max(np.abs(vf - vf_r) / vf_r))
    print(f"core vs reference: smoothed states {dx:.2e}, variances {dv:.2e} rel; filtered {dxf:.2e}, {dvf:.2e} rel")
    assert dx < STATE_TOL and dxf < STATE_TOL, (dx, dxf)
    assert dv < VAR_RTOL and dvf < VAR_RTOL, (dv, dvf)


# ---- 3. invariants of the core ---------------------------------------------------------------------------------------
def test_core_invariants(core, golden):
    """Last snapshot (T % R == 0): smoothed = filtered, bit for bit.  Smoothed variances <= filtered ones to rounding.
    Every checkpoint interval B gives the same bits (the replay from a checkpoint is the forward run)."""
    z = _full_ekf_records(golden)[0][:40_000]
    R = 200
    prior = _default_prior(z)
    base = core(z, R, *prior, B=1024)
    xs, vs, xf, vf = base
    assert np.array_equal(xs[-1], xf[-1]) and np.array_equal(vs[-1], vf[-1])
    assert np.all(vs <= vf * (1 + 1e-12)), np.max(vs / vf)
    assert np.all(vs[:-1] < vf[:-1])  # every earlier snapshot gains from later data
    for B in (32, 96, 4096, 40_000, 65_536):
        got = core(z, R, *prior, B=B)
        assert all(np.array_equal(a, b) for a, b in zip(got, base)), B


# ---- 4. argument errors ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kw,msg", [(dict(block=48), "block"), (dict(block=-32), "block"), (dict(block=1.5), "block"),
                                    (dict(k0=100), "k0"), (dict(k0=-200), "k0"), (dict(k0=200), "carried state"),
                                    (dict(state=np.zeros((2, 32))), "state"), (dict(state=np.zeros((3, 31))), "state"),
                                    (dict(k0=200, state=np.zeros(32)), "state")])
def test_argument_errors_before_device_work(monkeypatch, kw, msg):
    from deepfmkit_b200 import _lib, ekf_smooth

    def no_device(*a, **k):
        raise AssertionError("device work before the argument check")
    monkeypatch.setattr(_lib, "get_context", no_device)
    with pytest.raises(ValueError, match=msg):
        ekf_smooth(np.zeros((3, 1000)), F_SAMP, F_MOD, 1, **kw)


# =====================================================================================================================
# GPU
from tests.test_gpu_variants import EKF_C, EKF_EXPLICIT, EKF_R, EKF_T, REPLAY_CASES, REPLAY_R, _replay_inputs  # noqa: E402,E501


@pytest.fixture(scope="module")
def bank():
    """test_gpu_variants' 67-channel bank (12 123 samples: ragged last tile and buffer) under default and explicit
    options."""
    rng = np.random.RandomState(67)
    ms, phis = rng.uniform(3.0, 12.0, EKF_C), rng.uniform(-3.0, 3.0, EKF_C)
    z = np.stack([orc.snr_signal(ms[c], F_SAMP, F_MOD, 0.07, 40.0, seed=300 + c, phi0=phis[c])[:EKF_T]
                  for c in range(EKF_C)])
    rng = np.random.RandomState(68)
    ms, phis = rng.uniform(5.95, 6.05, EKF_C), rng.uniform(0.1, 0.2, EKF_C)
    ze = np.stack([orc.snr_signal(ms[c], F_SAMP, F_MOD, 0.07, 40.0, seed=400 + c, phi0=phis[c])[:EKF_T]
                   for c in range(EKF_C)])
    return {"default": z, "explicit": ze}


def _prior(z, opt):
    """The device's prior for a channel: the explicit options in full, or the defaults with the record's mean and
    variance."""
    if opt == "default":
        return _default_prior(z)
    e = EKF_EXPLICIT
    return (np.array([e["init_a"], e["init_m"], e["init_phi"], e["init_psi"], e["init_dc"]]), np.diag(e["p0_diag"]),
            np.asarray(e["q_diag"]), e["r_val"])


def _ctx_smooth(z, layout, opts, block=0, k0=0, state=None):
    """dfk_ekf_smooth_dev on a [C, T] host record laid out channel- or time-major; every output as numpy."""
    import torch
    from deepfmkit_b200 import _lib
    ctx = _lib.get_context(0)
    C, T = z.shape
    if layout == "cm":
        zd, ld_t, ld_c = torch.from_numpy(np.ascontiguousarray(z)).cuda(), 1, T
    else:
        zd, ld_t, ld_c = torch.from_numpy(np.ascontiguousarray(z.T)).cuda(), C, 1
    nbuf = T // EKF_R
    out = {k: torch.full((C, nbuf, w), -1.0, dtype=torch.float64, device="cuda")
           for k, w in (("rows", 8), ("var", 5), ("filtered", 8), ("filtered_var", 5))}
    ctx.ekf_smooth_dev(zd.data_ptr(), T, C, ld_t, ld_c, EKF_R, F_SAMP, F_MOD, opts, k0, state, block,
                       *[out[k].data_ptr() for k in ("rows", "var", "filtered", "filtered_var")])
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items()}


def _ctx_filter(z, layout, opts):
    import torch
    from deepfmkit_b200 import _lib
    ctx = _lib.get_context(0)
    C, T = z.shape
    if layout == "cm":
        zd, ld_t, ld_c = torch.from_numpy(np.ascontiguousarray(z)).cuda(), 1, T
    else:
        zd, ld_t, ld_c = torch.from_numpy(np.ascontiguousarray(z.T)).cuda(), C, 1
    rows = torch.full((C, T // EKF_R, 8), -1.0, dtype=torch.float64, device="cuda")
    ctx.ekf_dev(zd.data_ptr(), T, C, ld_t, ld_c, EKF_R, F_SAMP, F_MOD, opts, rows.data_ptr())
    torch.cuda.synchronize()
    return rows.cpu().numpy()


@pytest.fixture(scope="module")
def smooth_runs(bank):
    """The smoother and the filter on the bank: default and explicit options (test_gpu_variants' EKF_EXPLICIT: initial
    state, P0, Q, r and dc), channel- and time-major."""
    from tests.test_gpu_variants import _ekf_opts
    out = {}
    for opt, z in bank.items():
        opts = _ekf_opts(EKF_EXPLICIT if opt == "explicit" else None)
        for layout in ("cm", "tm"):
            out[opt, layout] = _ctx_smooth(z, layout, opts)
            out[opt, layout, "ekf_dev"] = _ctx_filter(z, layout, opts)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("opt", ["default", "explicit"])
def test_filtered_outputs_bit_identical(bank, smooth_runs, core, opt):
    """The forward kernel's rows are dfk_ekf_dev's bit for bit in both layouts (the same step, tiles and replay
    decision); its variances are the host core's diag P_f within the host-core gates."""
    z = bank[opt]
    for layout in ("cm", "tm"):
        assert np.array_equal(smooth_runs[opt, layout]["filtered"], smooth_runs[opt, layout, "ekf_dev"]), layout
    worst = [0.0, 0.0]
    got = smooth_runs[opt, "cm"]
    for c in range(0, EKF_C, 6):
        _, _, xf, vf = core(z[c], EKF_R, *_prior(z[c], opt))
        worst[0] = max(worst[0], np.max(np.abs(got["filtered"][c, :, :5] - xf)))
        worst[1] = max(worst[1], np.max(np.abs(got["filtered_var"][c] - vf) / vf))
    print(f"filtered ({opt}) vs host core: states {worst[0]:.2e}, variances {worst[1]:.2e} relative")
    assert worst[0] < STATE_TOL and worst[1] < VAR_RTOL, worst


@pytest.mark.gpu
@pytest.mark.parametrize("opt", ["default", "explicit"])
def test_smoothed_vs_core_and_reference(bank, smooth_runs, core, opt):
    """Smoothed rows and variances within the host-core gates of the host core and of ref_ekf_rts."""
    z = bank[opt]
    chans = list(range(0, EKF_C, 6)) + [EKF_C - 1]
    jobs = [(z[c], *_prior(z[c], opt), 0, EKF_R) for c in chans]
    with Pool(min(len(jobs), os.cpu_count() or 1)) as pool:
        refs = pool.map(_ref_snapshots, jobs)
    got = smooth_runs[opt, "cm"]
    if opt == "explicit":  # (the default options take dc and r from statistics summed in a layout's own order)
        assert all(np.array_equal(got[k], smooth_runs[opt, "tm"][k]) for k in got)
    assert np.all(got["rows"][:, :, 5] == 0) and np.all(got["rows"][:, :, 6] == 1) and np.all(got["rows"][:, :, 7] == 0)
    dev = {"core": [0.0, 0.0], "ref": [0.0, 0.0]}
    for c, (xs_r, vs_r, _, _) in zip(chans, refs):
        xs_c, vs_c, _, _ = core(z[c], EKF_R, *_prior(z[c], opt))
        for key, (xs, vs) in (("core", (xs_c, vs_c)), ("ref", (xs_r, vs_r))):
            dev[key][0] = max(dev[key][0], np.max(np.abs(got["rows"][c, :, :5] - xs)))
            dev[key][1] = max(dev[key][1], np.max(np.abs(got["var"][c] - vs) / vs))
    print(f"smoothed ({opt}) vs core: {dev['core'][0]:.2e}, {dev['core'][1]:.2e} rel; "
          f"vs reference: {dev['ref'][0]:.2e}, {dev['ref'][1]:.2e} rel")
    for key in dev:
        assert dev[key][0] < STATE_TOL and dev[key][1] < VAR_RTOL, (key, dev[key])


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["crossing", "one_hour"])
def test_smoothed_deep_in_time_with_carried_state(core, case):
    """A window starting at k0 from a carried state (x, full covariance, r) where the carrier angle reaches 1e6 inside
    the window ('crossing') or is past it throughout ('one_hour'), so the checked replay runs in both passes: the
    filtered rows are dfk_ekf_stream_dev's bit for bit, the carried state is not written, and the smoothed rows and
    variances match the host core run from the same state at the same k0."""
    import torch
    from deepfmkit_b200 import _lib, ekf_smooth
    z, state, kw = _replay_inputs(*REPLAY_CASES[case])
    k0, T = kw["k0"], len(z)
    sd = torch.from_numpy(state[None, :].copy()).cuda()
    got = ekf_smooth(z[None, :], F_SAMP, F_MOD, REPLAY_R // 200, k0=k0, state=sd, return_tensor=True)
    got = {k: v.cpu().numpy()[0] for k, v in got.items()}
    assert np.array_equal(sd.cpu().numpy()[0], state)
    ctx = _lib.get_context(0)
    zd = torch.from_numpy(z[None, :].copy()).cuda()
    rows = torch.empty((1, T // REPLAY_R, 8), dtype=torch.float64, device="cuda")
    ctx.ekf_stream_dev(zd.data_ptr(), T, 1, 1, T, REPLAY_R, F_SAMP, F_MOD, None, k0, sd.data_ptr(), rows.data_ptr())
    torch.cuda.synchronize()
    assert np.array_equal(got["filtered"], rows.cpu().numpy()[0])
    xs, vs, xf, vf = core(z, REPLAY_R, state[:5], _full_of(state[5:20]), Q_DEFAULT, state[30], k0=k0)
    dx, dv = np.max(np.abs(got["rows"][:, :5] - xs)), np.max(np.abs(got["var"] - vs) / vs)
    dxf, dvf = np.max(np.abs(got["filtered"][:, :5] - xf)), np.max(np.abs(got["filtered_var"] - vf) / vf)
    print(f"{case}: smoothed vs core {dx:.2e}, {dv:.2e} rel; filtered {dxf:.2e}, {dvf:.2e} rel")
    # 'crossing' inherits the filter's own deviation near |w_m t| = 1e6, where one ulp of the carrier angle is 1.2e-10
    # rad (test_gpu_variants.test_ekf_checked_replay_vs_oracle): measured on a B200, 1.4e-11 in the filtered and
    # 1.4e-11 in the smoothed states; 'one_hour' 1.1e-14 in both
    tol = 2e-10 if case == "crossing" else STATE_TOL
    assert dxf < tol and dx < tol and dv < VAR_RTOL and dvf < VAR_RTOL, (dx, dv, dxf, dvf)


@pytest.mark.gpu
def test_bit_identity_over_block_cpw_and_runs(bank):
    """Checkpoint interval B in {32, 96, 4096, >= T}, DFK_EKF_CPW in {1, ..., 32} and repeated runs: the same bits.
    The last snapshot of a window with T % R == 0 equals the filtered one."""
    from deepfmkit_b200 import _lib, ekf_smooth
    z = bank["default"]
    base = ekf_smooth(z, F_SAMP, F_MOD, 20, block=32)
    same = lambda a: all(np.array_equal(a[k], base[k]) for k in base)  # noqa: E731
    for B in (96, 4096, 12_128, 65_536):
        assert same(ekf_smooth(z, F_SAMP, F_MOD, 20, block=B)), B
    for cpw in (1, 2, 4, 8, 16, 32):
        with _lib.dev_overrides(DFK_EKF_CPW=cpw):
            assert same(ekf_smooth(z, F_SAMP, F_MOD, 20)), cpw
    assert same(ekf_smooth(z, F_SAMP, F_MOD, 20, block=32))
    even = ekf_smooth(z[:, :12_000], F_SAMP, F_MOD, 20)
    assert np.array_equal(even["rows"][:, -1], even["filtered"][:, -1])
    assert np.array_equal(even["var"][:, -1], even["filtered_var"][:, -1])


@pytest.mark.gpu
def test_statistics_on_model_records():
    """128 channels x 40 000 samples drawn from the filter's own model: a random walk with the filter's Q starting at
    the filter's initial state, measurement noise of variance r.  The smoothed mean-squared error of phi and psi is
    <= the filtered one at every row, and over the interior rows (away from both ends) the mean smoothed variance is
    within [0.8, 1.25] of the empirical MSE."""
    from deepfmkit_b200 import ekf_smooth
    C, T, R, r = 128, 40_000, 200, 1e-2
    rng = np.random.RandomState(2026)
    x0 = np.array([1.0, 6.0, 0.3, 0.1, 1.0])
    truth = x0 + np.cumsum(rng.randn(C, T, 5) * np.sqrt(Q_DEFAULT), axis=1)
    t = np.arange(T) / F_SAMP
    a, m, phi, psi, dc = np.moveaxis(truth, 2, 0)
    z = a * np.cos(phi + m * np.cos(2 * np.pi * F_MOD * t + psi)) + dc + np.sqrt(r) * rng.randn(C, T)
    got = ekf_smooth(z, F_SAMP, F_MOD, 1, init_a=x0[0], init_m=x0[1], init_phi=x0[2], init_psi=x0[3], R_val=r,
                     P0_diag=[1e-4] * 5)
    snap = truth[:, R - 1::R]
    for name, i in (("phi", 2), ("psi", 3)):
        mse_s = np.mean((got["rows"][:, :, i] - snap[:, :, i]) ** 2, axis=0)
        mse_f = np.mean((got["filtered"][:, :, i] - snap[:, :, i]) ** 2, axis=0)
        assert np.all(mse_s <= mse_f), (name, np.flatnonzero(mse_s > mse_f))
        inner = slice(20, -20)
        ratio = np.mean(got["var"][:, inner, i]) / np.mean(mse_s[inner])
        per_row = np.mean(got["var"][:, inner, i], axis=0) / mse_s[inner]
        print(f"{name}: smoothed/filtered MSE {np.mean(mse_s[inner] / mse_f[inner]):.3f}, mean smoothed variance / MSE "
              f"{ratio:.3f} (per row {per_row.min():.2f} .. {per_row.max():.2f})")
        assert 0.8 <= ratio <= 1.25, (name, ratio)


@pytest.mark.gpu
def test_nan_sample_poisons_its_channel_backwards_only(bank):
    """A NaN sample at t = 6001 in one channel (explicit options, so no statistic sees it): that channel's smoothed rows
    and variances at the snapshot before t are NaN (and the later ones, since the filter is NaN from t on); its filtered
    row before t and every output of the other channels are those of the clean record bit for bit."""
    from tests.test_gpu_variants import _ekf_opts
    opts = _ekf_opts(EKF_EXPLICIT)
    z = bank["explicit"][:8].copy()
    clean = _ctx_smooth(z, "cm", opts)
    z[3, 6_001] = np.nan
    got = _ctx_smooth(z, "cm", opts)
    others = [c for c in range(8) if c != 3]
    for k in clean:
        assert np.array_equal(got[k][others], clean[k][others]), k
    assert np.all(np.isnan(got["rows"][3, :, :5])) and np.all(np.isnan(got["var"][3]))
    assert np.array_equal(got["filtered"][3, :1], clean["filtered"][3, :1])  # snapshot 0 at sample 3999
    assert np.array_equal(got["filtered_var"][3, :1], clean["filtered_var"][3, :1])
    assert np.all(np.isnan(got["filtered"][3, 1:, :5]))


@pytest.mark.gpu
def test_short_window_writes_nothing():
    """T < R: no rows, nothing written, status OK (the library is asked directly with sentinel-filled outputs)."""
    import torch
    from deepfmkit_b200 import _lib
    ctx = _lib.get_context(0)
    zd = torch.ones((2, 3999), dtype=torch.float64, device="cuda")
    out = torch.full((16,), 7.0, dtype=torch.float64, device="cuda")
    ctx.ekf_smooth_dev(zd.data_ptr(), 3999, 2, 1, 3999, 4000, F_SAMP, F_MOD, None, 0, None, 0, out.data_ptr(),
                       out.data_ptr(), out.data_ptr(), out.data_ptr())
    torch.cuda.synchronize()
    assert torch.all(out == 7.0)


_NAMES_SCRIPT = """
import numpy as np, torch
from deepfmkit_b200 import _lib
from oracle import dfmi_oracle as orc
from tests.test_gpu_variants import launched_kernels
ctx = _lib.Context(0)
z = torch.from_numpy(np.stack([orc.snr_signal(6.0, 200e3, 1000.0, 0.05, 40.0, seed=c) for c in range(8)])).cuda()
C, T = z.shape
rows = torch.empty((C, T // 4000, 8), dtype=torch.float64, device="cuda")
_, names = launched_kernels(lambda: ctx.ekf_smooth_dev(z.data_ptr(), T, C, 1, T, 4000, 200e3, 1000.0, None, 0, None, 0,
                                                       rows.data_ptr()))
print("\\n".join(sorted(n.split("(")[0] for n in names)))
"""


@pytest.mark.gpu
def test_launch_count_and_kernels(bank):
    """Statistics (default options, channel-major: one launch), forward, backward: three launches; two with r and dc
    given.  The kernel names come from torch.profiler in a process of its own: with a profiler session here, the later
    sessions of test_gpu_variants in the same pytest process saw no kernels at all on a B200."""
    import sys
    import torch
    from deepfmkit_b200 import _lib
    ctx = _lib.get_context(0)
    z = torch.from_numpy(bank["default"]).cuda()
    C, T = z.shape
    rows = torch.empty((C, T // EKF_R, 8), dtype=torch.float64, device="cuda")
    opts = _lib.default_ekf_opts()
    for want in (3, 2):
        n0 = ctx.launch_count()
        ctx.ekf_smooth_dev(z.data_ptr(), T, C, 1, T, EKF_R, F_SAMP, F_MOD, opts, 0, None, 0, rows.data_ptr())
        ctx.synchronize()
        assert ctx.launch_count() - n0 == want, want
        opts.r_val, opts.init_dc = 1e-3, 1.0
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    out = subprocess.run([sys.executable, "-c", _NAMES_SCRIPT], cwd=ROOT, env=env, capture_output=True, text=True,
                         timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    names = {n.replace(" ", "") for n in out.stdout.split()}
    for k in ("channel_stats_kernel", "ekf_smooth_forward_kernel", "ekf_smooth_backward_kernel"):
        assert any(n.endswith("dfk::" + k) for n in names), (k, names)


@pytest.mark.gpu
def test_fitter_and_facade(bank):
    """EKFFitter.fit(smooth=True) on a host record and on a device record gives ekf_smooth's rows; the facade passes
    smooth through and adds tau; uncertainties=True still raises."""
    import pandas as pd
    import torch
    from deepfmkit_b200 import DeepFitFramework, DeepRawObject, EKFFitter, ekf_smooth
    z = bank["default"][5]
    ref = ekf_smooth(z[None, :], F_SAMP, F_MOD, 20)["rows"][0]
    host = EKFFitter({"n": 20}).fit(DeepRawObject(data=z, f_samp=F_SAMP, f_mod=F_MOD), smooth=True)
    assert list(host.columns) == ["amp", "m", "phi", "psi", "dc", "ssq", "fitok"]
    assert np.array_equal(host.to_numpy(dtype=float)[:, :5], ref[:, :5])
    raw = DeepRawObject(data=z, f_samp=F_SAMP, f_mod=F_MOD)
    raw.device_data = torch.from_numpy(z).cuda()
    dev = EKFFitter({"n": 20}).fit(raw, smooth=True)
    assert np.array_equal(dev.to_numpy(dtype=float), host.to_numpy(dtype=float))
    with pytest.raises(ValueError):
        EKFFitter({"n": 20}).fit(raw, smooth=True, uncertainties=True)

    class _Laser:
        df = 1.5e9

    class _Sim:
        label = "ch"
        laser = _Laser()
        fit_n = 20

    r = DeepRawObject(data=pd.DataFrame(z, columns=["ch0"]), f_samp=F_SAMP, f_mod=F_MOD, label="ch")
    r.sim = _Sim()
    dff = DeepFitFramework()
    dff.load_raw_object(r)
    dff.sims["ch"] = r.sim
    fobj = dff.fit("ch", method="ekf", smooth=True)
    df = dff.fits_df["ch_ekf"]
    assert np.array_equal(df[["amp", "m", "phi", "psi", "dc"]].to_numpy(), ref[:, :5])
    assert np.array_equal(df["tau"].to_numpy(), df["m"].to_numpy() / (2 * np.pi * 1.5e9))
    assert np.array_equal(fobj.phi, ref[:, 2])
