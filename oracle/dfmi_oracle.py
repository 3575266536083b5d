"""numpy restatement of the DFMI readout hot path (TEST INFRASTRUCTURE, see oracle/__init__.py).

Every function cites the reference lines it follows (paths relative to the
upstream repo mdovale/DeepFMKit).  The arithmetic is kept in the same
operation order as the reference so that the oracle reproduces the reference's
numbers to the last bit wherever numpy/scipy evaluate the same expressions;
``tests/test_oracle_golden.py`` pins that against fixtures minted from the
unmodified reference.

Layout conventions (identical to the reference):
  * a record is a 1-D fp64 array; buffer ``b`` is ``x[b*R:(b+1)*R]``;
  * the harmonic vector is ``qi = [Q_1..Q_N, I_1..I_N]`` with Q the cosine and
    I the sine lock-in mean, normalised by 1/R;
  * the parameter vector is ``[amp, m, phi, psi]``;
  * a result row is ``(amp, m, phi, psi, dc, ssq, fitok)``.
"""
from __future__ import annotations

import math
import os
from dataclasses import dataclass, replace

import numpy as np
from scipy.special import jv

ROW_COLUMNS = ("amp", "m", "phi", "psi", "dc", "ssq", "fitok")

# fit.py:222 -- the damping ladder is fixed and restarted at every outer step.
LAMBDA_LADDER = (0.0, 1e-7, 1e-5, 1e-3, 1e-1, 1, 10, 100)


@dataclass(frozen=True)
class Tunables:
    """Module-level knobs of the reference solver (fit.py:5-16)."""

    max_lma_steps: int = 100
    conv_improve: float = 1e-9
    conv_param: float = 1e-9
    fitok_threshold: float = 1e-3
    m_grid_min: float = 5.0
    m_grid_max: float = 30.0
    m_grid_step: float = 0.5
    bessel_amp_threshold: float = 0.05
    sincos_amp_threshold: float = 0.1


DEFAULT_TUNABLES = Tunables()


# --------------------------------------------------------------------------- #
# buffer geometry                                                              #
# --------------------------------------------------------------------------- #
def buffer_geometry(n_samples: int, f_samp: float, f_mod: float, n: int):
    """(R, fs, nbuf) exactly as fitters.py:81-83 / core.py:416-418."""
    R = int(f_samp / f_mod * n)
    fs = f_samp / R
    nbuf = int(n_samples / R)
    return R, fs, nbuf


def rad_per_sample(f_samp: float, f_mod: float) -> float:
    """w0 of fitters.py:39,376,434 (left-to-right evaluation matters for the last bit)."""
    return 2.0 * np.pi * f_mod / f_samp


# --------------------------------------------------------------------------- #
# demodulation: fit.py:18-66 + the mean() loops of fitters.py:45-49            #
# --------------------------------------------------------------------------- #
def lockin_means(buf: np.ndarray, w0: float, nh: int) -> np.ndarray:
    """Harmonic vector of one buffer: mean(x*cos(k*w0*t)), mean(x*sin(k*w0*t)), k=1..nh.

    The time index restarts at zero for every buffer (fit.py:55) and the angle
    is formed as ``((k)*w0)*t`` in fp64 (fit.py:59).
    """
    buf = np.asarray(buf)
    t = np.arange(len(buf))
    qi = np.zeros(2 * nh)
    for h in range(nh):
        angle = (h + 1) * w0 * t
        qi[h] = (buf * np.cos(angle)).mean()
        qi[h + nh] = (buf * np.sin(angle)).mean()
    return qi


# --------------------------------------------------------------------------- #
# harmonic model, Jacobian, normal equations: fit.py:68-150                    #
# --------------------------------------------------------------------------- #
def model_state(nh: int, qi: np.ndarray, p: np.ndarray):
    """Return (ssq, JTJ[4,4], g[4]) at parameter vector p = [a, m, phi, psi]."""
    a, m, phi, psi = p
    order = np.arange(1, nh + 1)
    quarter = np.cos(phi + order * np.pi / 2.0)  # fit.py:100
    cpsi = np.cos(order * psi)
    spsi = np.sin(order * psi)
    bes = jv(order, m)  # fit.py:106
    dbes = 0.5 * (jv(order - 1, m) - jv(order + 1, m))  # fit.py:108

    envelope = a * quarter * bes  # fit.py:111
    mq = envelope * cpsi
    mi = -envelope * spsi  # fit.py:114 (the line above it in the reference is dead)

    res = np.concatenate([qi[:nh] - mq, qi[nh:] - mi])
    ssq = np.dot(res, res)

    jac = np.zeros((2 * nh, 4))
    if a != 0:  # fit.py:126 -- the amplitude column stays zero at a == 0
        jac[:nh, 0] = mq / a
        jac[nh:, 0] = mi / a
    dm = a * quarter * dbes  # fit.py:131
    jac[:nh, 1] = dm * cpsi
    jac[nh:, 1] = -dm * spsi
    dphi = a * np.cos(phi + order * np.pi / 2.0 + np.pi / 2.0) * bes  # fit.py:137-138
    jac[:nh, 2] = dphi * cpsi
    jac[nh:, 2] = -dphi * spsi
    jac[:nh, 3] = envelope * -spsi * order  # fit.py:143
    jac[nh:, 3] = -envelope * cpsi * order  # fit.py:144

    return ssq, jac.T @ jac, jac.T @ res


def residual_ssq(nh: int, qi: np.ndarray, p: np.ndarray) -> float:
    """Sum of squared residuals only (fit.py:152-167)."""
    a, m, phi, psi = p
    order = np.arange(1, nh + 1)
    envelope = a * np.cos(phi + order * np.pi / 2.0) * jv(order, m)
    mq = envelope * np.cos(order * psi)
    mi = -envelope * np.sin(order * psi)
    res = np.concatenate([qi[:nh] - mq, qi[nh:] - mi])
    return np.dot(res, res)


def damped_step(lam: float, jtj: np.ndarray, g: np.ndarray) -> np.ndarray:
    """Solve (JTJ + lam*diag(JTJ)) dp = g; an exactly singular system yields dp = 0 (fit.py:169-206)."""
    lhs = jtj + lam * np.diag(np.diag(jtj))
    try:
        return np.linalg.solve(lhs, g)
    except np.linalg.LinAlgError:
        return np.zeros(4)


@dataclass
class LMCounters:
    """Work counters used for the FP64 flop accounting of the LM kernel (SURVEY 8d)."""

    n_state: int = 0
    n_ssq: int = 0
    n_solve: int = 0
    n_grid: int = 0


def lm_descend(nh: int, qi: np.ndarray, p0: np.ndarray, tun: Tunables = DEFAULT_TUNABLES,
               counters: LMCounters | None = None):
    """Levenberg-Marquardt loop of fit.py:208-258. Returns (p, ssq)."""
    p = np.array(p0, dtype=float)
    ssq, jtj, g = model_state(nh, qi, p)
    if counters:
        counters.n_state += 1
    for _ in range(tun.max_lma_steps):
        p_prev = p.copy()
        best_ssq, best_p = ssq, p
        for lam in LAMBDA_LADDER:
            dp = damped_step(lam, jtj, g)
            if counters:
                counters.n_solve += 1
            if np.linalg.norm(dp) < 1e-15:  # fit.py:230
                continue
            trial = p + dp
            trial_ssq = residual_ssq(nh, qi, trial)
            if counters:
                counters.n_ssq += 1
            if trial_ssq < best_ssq:  # first strictly better damping wins (fit.py:240-243)
                best_ssq, best_p = trial_ssq, trial
                break
        if best_ssq >= ssq:  # fit.py:246
            break
        p = best_p
        ssq, jtj, g = model_state(nh, qi, p)
        if counters:
            counters.n_state += 1
        moved = np.linalg.norm(p - p_prev)
        if (ssq - best_ssq) < tun.conv_improve and moved < tun.conv_param:  # fit.py:255
            break
    return p, ssq


def grid_seed(nh: int, qi: np.ndarray, tun: Tunables = DEFAULT_TUNABLES) -> np.ndarray:
    """Fallback initialiser: scan m on a grid with psi = 0, estimate phi and a linearly (fit.py:260-320).

    With psi_try = 0 the sine-half weights are -J*sin(0) = -0.0, so only the
    cosine half of qi can pass the Bessel threshold; the sine-half branches
    are kept for fidelity.
    """
    best_ssq = 9e99
    best = np.zeros(4)
    psi_try = 0.0
    order = np.arange(1, nh + 1)
    q_part, i_part = qi[:nh], qi[nh:]
    for m_try in np.arange(tun.m_grid_min, tun.m_grid_max + tun.m_grid_step, tun.m_grid_step):
        wq = jv(order, m_try) * np.cos(order * psi_try)
        wi = jv(order, m_try) * -np.sin(order * psi_try)
        s_sum = c_sum = 0.0
        n_s = n_c = 0
        for h in range(nh):
            quad = int(order[h] % 4)
            for val, w in ((q_part[h], wq[h]), (i_part[h], wi[h])):
                if abs(w) > tun.bessel_amp_threshold:
                    r = val / w
                    if quad == 0:
                        c_sum += r; n_c += 1
                    elif quad == 1:
                        s_sum -= r; n_s += 1
                    elif quad == 2:
                        c_sum -= r; n_c += 1
                    else:
                        s_sum += r; n_s += 1
        if n_s == 0 or n_c == 0:
            continue
        phi_try = np.arctan2(s_sum / n_s, c_sum / n_c)
        lut = np.array([math.cos(phi_try), -math.sin(phi_try), -math.cos(phi_try), math.sin(phi_try)])
        a_sum, n_a = 0.0, 0
        for h in range(nh):
            f = lut[order[h] % 4]
            for val, w in ((q_part[h], wq[h]), (i_part[h], wi[h])):
                if abs(w) > tun.bessel_amp_threshold and abs(f) > tun.sincos_amp_threshold:
                    a_sum += val / (f * w)
                    n_a += 1
        if n_a == 0:
            continue
        cand = np.array([a_sum / n_a, m_try, phi_try, psi_try])
        cand_ssq = residual_ssq(nh, qi, cand)
        if cand_ssq < best_ssq:
            best_ssq, best = cand_ssq, cand
    return best


def fit_harmonics(nh: int, qi: np.ndarray, p0: np.ndarray, tun: Tunables = DEFAULT_TUNABLES,
                  counters: LMCounters | None = None):
    """One full fit (fit.py:322-362). Returns (status, p, ssq); status 0/1/2 as in the reference."""
    p, ssq = lm_descend(nh, qi, p0, tun, counters)
    if ssq < tun.fitok_threshold:
        status = 0
    else:
        seed = grid_seed(nh, qi, tun)
        if counters:
            counters.n_grid += 1
        if np.any(seed):
            p2, ssq2 = lm_descend(nh, qi, seed, tun, counters)
            if ssq2 < ssq:
                p, ssq = p2, ssq2
        status = 1 if ssq < tun.fitok_threshold else 2
    if p[0] < 0:  # fit.py:352-357
        p[0] *= -1
        p[2] += np.pi
    if p[1] < 0:
        p[1] *= -1
        p[2] += np.pi
    p[2] = (p[2] + np.pi) % (2 * np.pi) - np.pi  # fit.py:360; psi is left unwrapped
    return status, p, ssq


# --------------------------------------------------------------------------- #
# per-record drivers: fitters.py:13-60, 370-447                                #
# --------------------------------------------------------------------------- #
def nls_chain(bufs: np.ndarray, nh: int, w0: float, guess, tun: Tunables = DEFAULT_TUNABLES,
              counters: LMCounters | None = None) -> np.ndarray:
    """Warm-start chain over the rows of ``bufs`` (fitters.py:42-58 / 378-392). Returns rows[nbuf,7]."""
    guess = np.array(guess, dtype=float)
    rows = np.zeros((bufs.shape[0], 7))
    for b in range(bufs.shape[0]):
        qi = lockin_means(bufs[b], w0, nh)
        status, p, ssq = fit_harmonics(nh, qi, guess, tun, counters)
        guess = p
        rows[b] = (p[0], p[1], p[2], p[3], np.mean(bufs[b]), ssq, status)
    return rows


def nls_fit(x: np.ndarray, f_samp: float, f_mod: float, n: int, nh: int = 10,
            init_a: float = 1.6, init_m: float = 6.0, init_psi: float = 0.0,
            schedule: str = "sequential", n_chunks: int | None = None,
            tun: Tunables = DEFAULT_TUNABLES, counters: LMCounters | None = None) -> np.ndarray:
    """StandardNLSFitter.fit restated (fitters.py:330-428).

    schedule:
      'sequential' -- one warm-start chain over all buffers (parallel=False, fitters.py:370-393);
      'seeded'     -- buffer 0 first, then ``n_chunks`` chains over np.array_split(buffers[1:])
                      each seeded from buffer 0's result (parallel=True, fitters.py:395-428);
      'gpu'        -- 'seeded' with one buffer per chain, i.e. the reference's own schedule at
                      n_cores >= nbuf-1; this is the schedule the CUDA path implements.
    """
    x = np.asarray(x, dtype=float).ravel()
    R, _, nbuf = buffer_geometry(len(x), f_samp, f_mod, n)
    if nbuf == 0:
        return np.zeros((0, 7))
    w0 = rad_per_sample(f_samp, f_mod)
    bufs = x[: nbuf * R].reshape(nbuf, R)
    seed = np.array([init_a, init_m, 0.0, init_psi])
    if schedule == "sequential":
        return nls_chain(bufs, nh, w0, seed, tun, counters)
    first = nls_chain(bufs[:1], nh, w0, seed, tun, counters)
    if nbuf == 1:
        return first
    if schedule == "gpu":
        n_chunks = nbuf - 1
    elif n_chunks is None:
        n_chunks = os.cpu_count()
    n_chunks = min(n_chunks, nbuf)
    rows = [first]
    for chunk in np.array_split(bufs[1:], n_chunks):
        if chunk.size:
            rows.append(nls_chain(chunk, nh, w0, first[0, :4], tun, counters))
    return np.concatenate(rows, axis=0)


def _pool_job(args):
    chunk, nh, w0, guess = args
    return nls_chain(chunk, nh, w0, guess)


def nls_fit_pool(x: np.ndarray, f_samp: float, f_mod: float, n: int, nh: int = 10,
                 init_a: float = 1.6, init_m: float = 6.0, init_psi: float = 0.0,
                 n_procs: int | None = None) -> np.ndarray:
    """The reference's multiprocessing schedule (fitters.py:395-428) with a real process pool.

    Used only to time the CPU baseline on the host cores; numerically identical
    to ``nls_fit(schedule='seeded', n_chunks=n_procs)``.
    """
    from multiprocessing import Pool

    x = np.asarray(x, dtype=float).ravel()
    R, _, nbuf = buffer_geometry(len(x), f_samp, f_mod, n)
    if nbuf == 0:
        return np.zeros((0, 7))
    w0 = rad_per_sample(f_samp, f_mod)
    bufs = x[: nbuf * R].reshape(nbuf, R)
    n_procs = min(n_procs or os.cpu_count(), nbuf)
    first = nls_chain(bufs[:1], nh, w0, np.array([init_a, init_m, 0.0, init_psi]))
    if nbuf == 1:
        return first
    jobs = [(c, nh, w0, first[0, :4]) for c in np.array_split(bufs[1:], n_procs) if c.size]
    with Pool(n_procs) as pool:
        parts = pool.map(_pool_job, jobs)
    return np.concatenate([first] + parts, axis=0)


# --------------------------------------------------------------------------- #
# time-domain EKF: fitters.py:214-320                                          #
# --------------------------------------------------------------------------- #
EKF_P0_DIAG = (1.0, 1.0, 1.0, 1.0, 1.0)
EKF_Q_DIAG = (1e-8, 1e-8, 1e-6, 1e-6, 1e-8)


def ekf_track(x: np.ndarray, f_samp: float, f_mod: float, n: int,
              init_a: float = 1.6, init_m: float = 6.0, init_phi: float = 0.0, init_psi: float = 0.0,
              p0_diag=EKF_P0_DIAG, q_diag=EKF_Q_DIAG, r_val: float | None = None,
              init_dc: float | None = None, k0: int = 0, init_cov=None) -> np.ndarray:
    """5-state random-walk EKF with scalar measurement, state snapshot every R samples.

    State [a, m, phi, psi, dc]; time is absolute, t_k = k / f_samp (fitters.py:263).
    Returns rows[nbuf,7] with ssq = 0 and fitok = 1 (fitters.py:313-318).
    k0 and init_cov are not reference options either: x is then the part of a longer record that starts at sample k0
    (t_k = (k0 + k) / f_samp), and the filter resumes from the full 5x5 covariance init_cov instead of diag(p0_diag),
    which is how a continuation slab of the GPU's streamed entry point is checked.
    """
    z = np.asarray(x, dtype=float).ravel()
    R, _, nbuf = buffer_geometry(len(z), f_samp, f_mod, n)
    # init_dc is not a reference option: it lets tests of the slab-wise GPU entry point start the filter from the
    # first slab's mean, as that entry point does (the reference always uses the whole record's mean).
    state = np.array([init_a, init_m, init_phi, init_psi, np.mean(z) if init_dc is None else init_dc])
    cov = np.diag(p0_diag).astype(float) if init_cov is None else np.array(init_cov, dtype=float).reshape(5, 5)
    q_mat = np.diag(q_diag).astype(float)
    if r_val is None:
        r_val = np.var(z)
    r_mat = np.array([[r_val]])
    eye = np.eye(5)
    w_m = 2 * np.pi * f_mod
    t_axis = (int(k0) + np.arange(len(z))) / f_samp
    snaps = np.zeros((nbuf, 5))
    for k in range(len(z)):
        cov = eye @ cov @ eye.T + q_mat  # fitters.py:276 (F = I)
        a, m, phi, psi, dc = state
        theta = w_m * t_axis[k] + psi
        arg = phi + m * np.cos(theta)
        pred = a * np.cos(arg) + dc
        s_arg = np.sin(arg)
        h_row = np.array([[np.cos(arg), -a * s_arg * np.cos(theta), -a * s_arg,
                           +a * m * s_arg * np.sin(theta), 1.0]])
        innov = z[k] - pred
        s_mat = h_row @ cov @ h_row.T + r_mat
        gain = (cov @ h_row.T) @ np.linalg.inv(s_mat)
        state = state + (gain @ innov.reshape(1, 1)).flatten()
        cov = (eye - gain @ h_row) @ cov  # simple form, not Joseph (fitters.py:302)
        if (k + 1) % R == 0:
            idx = (k + 1) // R - 1
            if idx < nbuf:
                snaps[idx] = state
    rows = np.zeros((nbuf, 7))
    rows[:, :5] = snaps
    rows[:, 6] = 1.0
    return rows


# --------------------------------------------------------------------------- #
# 'snr'-mode synthetic input: physics.py:475-530, helpers.py:10-14             #
# --------------------------------------------------------------------------- #
SPEED_OF_LIGHT = 299792458.0  # scipy.constants.c


def effective_m(m_target: float, ref_arml: float = 0.1, meas_arml: float = 0.3) -> float:
    """Round trip m -> laser.df -> DFMIObject.m (helpers.py:10-14, physics.py:291-295)."""
    opd = np.abs(meas_arml - ref_arml)
    df = (m_target * SPEED_OF_LIGHT) / (2 * np.pi * opd)
    delta_l = meas_arml - ref_arml
    return 2 * np.pi * df * delta_l / SPEED_OF_LIGHT


def laser_df(m_target: float, ref_arml: float = 0.1, meas_arml: float = 0.3) -> float:
    return (m_target * SPEED_OF_LIGHT) / (2 * np.pi * np.abs(meas_arml - ref_arml))


def snr_signal(m_target: float, f_samp: float, f_mod: float, n_seconds: float, snr_db: float,
               seed: int = 0, amp: float = 1.0, visibility: float = 1.0,
               phi0: float = 0.0, psi0: float = 0.0) -> np.ndarray:
    """y = A(1 + C cos(phi0 + m cos(w_m t + psi0))) + sigma*randn, MT19937 seeded by trial number."""
    n = int(n_seconds * f_samp)
    t = np.arange(n) / f_samp
    m = effective_m(m_target)
    w_mod = 2 * np.pi * f_mod
    clean = amp * (1 + visibility * np.cos(phi0 + m * np.cos(w_mod * t + psi0)))
    ac = clean - np.mean(clean)
    noise_power = np.mean(ac ** 2) / 10 ** (snr_db / 10.0)
    rng = np.random.RandomState(seed=seed)
    return clean + rng.randn(len(clean)) * np.sqrt(noise_power)


def asd_signal(m_target: float, f_samp: float, f_mod: float, n_seconds: float, trial: int = 0,
               amp_n: float = 0.0, df_n: float = 0.0, arml_mod_amp: float = 0.0, arml_mod_f: float = 5.0,
               arml_mod_psi: float = 0.0, phi0: float = 0.0, psi0: float = 0.0, amp: float = 1.0,
               visibility: float = 1.0, wavelength: float = 1.064e-6, ref_arml: float = 0.1,
               meas_arml: float = 0.3, dynamic: bool = True, df: float = None, external_noise: dict = None):
    """'asd'-mode record of the reference's exact physical model (physics.py:423-440, 557-611, 615-722).

    Only the white noise sources (``amp_n``, ``df_n``: ``RandomState(1 + 4*trial).normal``, amplitude drawn before
    df, physics.py:581-597) are restated; the coloured ones (``f_n``, ``arml_mod_n``) need ``pyplnoise``, a
    third-party generator that is absent from the reference checkout and from this image.  ``external_noise``
    (physics.py:430-434) replaces all internal draws by given series -- keys 'laser_frequency', 'amplitude', 'df',
    'armlength', missing ones zero -- which is how those two sources can still be exercised.
    The arm-length modulation makes the interferometric phase walk: the record drifting fits are tested on.
    Returns (signal, ground-truth phase).
    """
    n = int(n_seconds * f_samp)
    t = np.arange(n) / f_samp
    if df is None:
        df = laser_df(m_target, ref_arml, meas_arml)
    noise_f = noise_arm = 0.0
    if external_noise:
        noise_amp = external_noise.get("amplitude", 0.0)
        noise_df = external_noise.get("df", 0.0)
        noise_f = external_noise.get("laser_frequency", 0.0)
        noise_arm = external_noise.get("armlength", 0.0)
    else:
        rng = np.random.RandomState(seed=1 + trial * 4)  # physics.py:577-580
        noise_amp = rng.normal(scale=amp_n * np.sqrt(f_samp / 2.0), size=n) if amp_n != 0.0 else 0.0
        noise_df = rng.normal(scale=df_n * np.sqrt(f_samp / 2.0), size=n) if df_n != 0.0 else 0.0
    omega_mod = 2 * np.pi * f_mod
    g = np.cos(omega_mod * t + psi0)  # default waveform_func (physics.py:44)
    peak = np.max(np.abs(g))
    g = g / peak if peak != 0 else np.zeros_like(g)
    dt = t[1] - t[0]
    fs = 1 / dt
    phi_mod = (2 * np.pi / fs) * np.cumsum((df + noise_df) * g)  # physics.py:675
    tau_r = ref_arml / SPEED_OF_LIGHT
    tau_m = meas_arml / SPEED_OF_LIGHT
    if not dynamic:
        path = phi0 * wavelength / (2 * np.pi)
    else:
        path = (arml_mod_amp * np.sin(2 * np.pi * arml_mod_f * t + arml_mod_psi) + noise_arm
                + phi0 * wavelength / (2 * np.pi))
    tau_dl = path / SPEED_OF_LIGHT
    pm_meas = np.interp(t - (tau_m + tau_dl), t, phi_mod)
    pm_ref = np.interp(t - tau_r, t, phi_mod)
    f0 = (SPEED_OF_LIGHT / wavelength) + noise_f
    carrier = (2 * np.pi * f0) * ((tau_m + tau_dl) - tau_r)
    phase = carrier + (pm_meas - pm_ref)
    signal = (amp + noise_amp) * (1 + visibility * np.cos(phase))
    truth = (2 * np.pi * SPEED_OF_LIGHT / wavelength) * ((tau_m + tau_dl) - tau_r)
    if np.isscalar(truth):
        truth = np.full_like(t, truth, dtype=float)
    return signal, truth


# --------------------------------------------------------------------------- #
# CRLB of m (helpers.py:16-45) -- used only for the "<= 1% of sigma" clause    #
# --------------------------------------------------------------------------- #
def crlb_sigma_m(m_true: float, nh: int, snr_db: float, buffer_size: int) -> float:
    noise_td = 0.5 / 10 ** (snr_db / 10.0)
    var_iq = noise_td / (2 * buffer_size)
    _, jtj, _ = model_state(nh, np.zeros(2 * nh), np.array([1.0, m_true, 0.0, 0.0]))
    try:
        return float(np.sqrt(np.linalg.inv(jtj)[1, 1] * var_iq))
    except np.linalg.LinAlgError:
        return float("nan")


def with_tunables(**kw) -> Tunables:
    return replace(DEFAULT_TUNABLES, **kw)
