"""Pin the CPU oracle against fixtures minted from the unmodified reference (tests/golden/make_golden.py)."""
import numpy as np
import pytest

from oracle import dfmi_oracle as orc

NLS_CASES = ["cfg1_quickstart", "cfg2_1mhz", "cfg3_channel", "deep_mod_n62", "fallback_m16",
             "pathological_m3", "low_snr"]


def _signal_from_meta(meta):
    m, f_samp, f_mod, n_seconds, snr_db, trial, phi, psi = meta[:8]
    return orc.snr_signal(m, f_samp, f_mod, n_seconds, snr_db, seed=int(trial), phi0=phi, psi0=psi)


@pytest.mark.parametrize("name", NLS_CASES)
def test_synth_matches_reference_physics(golden, name):
    g = golden(name)
    x = _signal_from_meta(g["meta"])
    assert np.array_equal(x[:16], g["x_head"])
    assert np.array_equal(x[-16:], g["x_tail"])
    assert x.sum() == g["x_sum"][0] and np.abs(x).sum() == g["x_sum"][1]
    if "x" in g.files:
        assert np.array_equal(x, g["x"])


@pytest.mark.parametrize("name", NLS_CASES)
def test_demod_bit_exact(golden, name):
    g = golden(name)
    meta = g["meta"]
    x = g["x"] if "x" in g.files else _signal_from_meta(meta)
    f_samp, f_mod, n, nh = meta[1], meta[2], int(meta[8]), int(meta[9])
    R, _, nbuf = orc.buffer_geometry(len(x), f_samp, f_mod, n)
    w0 = orc.rad_per_sample(f_samp, f_mod)
    for b in range(min(nbuf, 4)):
        qi = orc.lockin_means(x[b * R:(b + 1) * R], w0, nh)
        assert np.array_equal(qi, g["qi"][b])


@pytest.mark.parametrize("name", NLS_CASES)
def test_nls_rows_bit_exact(golden, name):
    g = golden(name)
    meta = g["meta"]
    x = g["x"] if "x" in g.files else _signal_from_meta(meta)
    f_samp, f_mod, n, nh, n_cores = meta[1], meta[2], int(meta[8]), int(meta[9]), int(meta[10])
    kw = dict(init_a=meta[11], init_m=meta[12], init_psi=meta[13])
    seq = orc.nls_fit(x, f_samp, f_mod, n, nh, schedule="sequential", **kw)
    assert np.array_equal(seq, g["rows_seq"])
    if len(g["rows_par"]):
        par = orc.nls_fit(x, f_samp, f_mod, n, nh, schedule="seeded", n_chunks=n_cores, **kw)
        assert np.array_equal(par, g["rows_par"])


def test_expected_flags_in_fixtures(golden):
    assert set(golden("cfg1_quickstart")["rows_seq"][:, 6]) == {0.0}
    assert 1.0 in set(golden("fallback_m16")["rows_seq"][:, 6])
    assert 2.0 in set(golden("pathological_m3")["rows_seq"][:, 6])


def test_gpu_schedule_within_gate_of_reference(golden):
    """Every buffer seeded from buffer 0 (the CUDA schedule) stays within 1e-8 of the reference chain."""
    for name in ("cfg1_quickstart", "cfg3_channel", "low_snr"):
        g = golden(name)
        meta = g["meta"]
        x = g["x"] if "x" in g.files else _signal_from_meta(meta)
        rows = orc.nls_fit(x, meta[1], meta[2], int(meta[8]), int(meta[9]), schedule="gpu",
                           init_a=meta[11], init_m=meta[12], init_psi=meta[13])
        ref = g["rows_seq"]
        assert np.array_equal(rows[:, 6], ref[:, 6])
        assert np.max(np.abs(rows[:, :4] - ref[:, :4])) < 1e-8
        assert np.array_equal(rows[:, 4], ref[:, 4])


def test_cfg5_rows(golden):
    g = golden("cfg5_crlb")
    for a, m in enumerate(g["ms"]):
        for t in range(int(g["trials"])):
            x = orc.snr_signal(float(m), 200e3, 1000, 1 / 1000, 40.0, seed=t)
            row = orc.nls_fit(x, 200e3, 1000, 1, 15, init_m=float(m))[0]
            assert np.array_equal(row, g["rows"][a, t])


def test_solver_units(golden):
    g = golden("solver_units")
    nh = int(g["nh"])
    for c in range(len(g["params"])):
        ssq, jtj, grad = orc.model_state(nh, g["data"][c], g["params"][c])
        assert ssq == g["ssq"][c]
        assert np.array_equal(jtj.flatten(), g["jtj"][c])
        assert np.array_equal(grad, g["grad"][c])
        assert orc.residual_ssq(nh, g["data"][c], g["params"][c]) == g["ssq_only"][c]
        for li, lam in enumerate(orc.LAMBDA_LADDER):
            assert np.array_equal(orc.damped_step(lam, jtj, grad), g["steps"][c, li])
        assert np.array_equal(orc.grid_seed(nh, g["data"][c]), g["seeds"][c])
        st, p, s = orc.fit_harmonics(nh, g["data"][c].copy(), np.array([1.6, 6.0, 0.0, 0.0]))
        assert st == g["fit_status"][c] and s == g["fit_ssq"][c] and np.array_equal(p, g["fit_p"][c])
        assert np.array_equal(orc.grid_seed(nh, g["clean_qi"][c]), g["clean_seed"][c])
        st, p, s = orc.fit_harmonics(nh, g["clean_qi"][c].copy(), np.array([1.6, 6.0, 0.0, 0.0]))
        assert st == g["clean_status"][c] and s == g["clean_ssq"][c] and np.array_equal(p, g["clean_p"][c])


def ekf_kwargs(g):
    kw = {}
    rename = {"P0_diag": "p0_diag", "Q_diag": "q_diag", "R_val": "r_val"}
    for k, v in zip(g["kw_keys"], g["kw_vals"]):
        v = v[~np.isnan(v)]
        kw[rename.get(str(k), str(k))] = float(v[0]) if v.size == 1 else v
    return kw


@pytest.mark.parametrize("name", ["ekf_default", "ekf_offset"])
def test_ekf_full_record_bit_exact(golden, name):
    g = golden(name)
    rows = orc.ekf_track(g["x"], 200e3, 1000.0, 20, **ekf_kwargs(g))
    assert np.array_equal(rows, g["rows"])


@pytest.mark.parametrize("name", ["ekf_default", "ekf_offset"])
def test_ekf_resume_options_at_their_defaults_are_bit_exact(golden, name):
    """k0 = 0 and init_cov = None (or the same diagonal given as a full matrix) leave the filter the reference's."""
    g = golden(name)
    kw = ekf_kwargs(g)
    rows = orc.ekf_track(g["x"], 200e3, 1000.0, 20, k0=0, init_cov=None, **kw)
    assert np.array_equal(rows, g["rows"])
    cov = np.diag(kw.get("p0_diag", orc.EKF_P0_DIAG))
    rows = orc.ekf_track(g["x"], 200e3, 1000.0, 20, init_cov=cov, **kw)
    assert np.array_equal(rows, g["rows"])


def test_crlb_helper_is_finite():
    s = orc.crlb_sigma_m(6.0, 10, 40.0, 4000)
    assert 1e-5 < s < 1e-2


# ---- full-size fixtures (tests/golden/make_golden_full.py) -------------------------------------------------------
def _full_signal(g):
    m, f_samp, f_mod, secs, snr, trial, phi, psi = g["meta"][:8]
    x = orc.snr_signal(m, f_samp, f_mod, secs, snr, seed=int(trial), phi0=phi, psi0=psi)
    assert np.array_equal(x[:16], g["x_head"]) and np.array_equal(x[-16:], g["x_tail"])
    assert x.sum() == g["x_sum"][0] and np.abs(x).sum() == g["x_sum"][1]
    return x


def test_full_cfg1_all_500_buffers_bit_exact(golden):
    g = golden("full_cfg1")
    x = _full_signal(g)
    assert np.array_equal(orc.nls_fit(x, 200e3, 1000.0, 20, 10, schedule="sequential"), g["rows_seq"])
    assert np.array_equal(orc.nls_fit(x, 200e3, 1000.0, 20, 10, schedule="seeded", n_chunks=int(g["meta"][10])),
                          g["rows_par"])
    assert len(g["rows_seq"]) == 500


@pytest.mark.parametrize("name", ["full_cfg2_first", "full_cfg2_last", "full_cfg3_c37"])
def test_full_slab_prefix_bit_exact(golden, name):
    """A prefix of the sequential chain is the chain of the prefix: pin the first 40 buffers of the long fixtures."""
    g = golden(name)
    x = _full_signal(g)
    f_samp, n, nh = g["meta"][1], int(g["meta"][8]), int(g["meta"][9])
    R = int(f_samp / 1000.0 * n)
    rows = orc.nls_fit(x[: 40 * R], f_samp, 1000.0, n, nh, schedule="sequential")
    assert np.array_equal(rows, g["rows_seq"][:40])
    w0 = orc.rad_per_sample(f_samp, 1000.0)
    for b in (0, 39, len(g["qi"]) - 1):
        assert np.array_equal(orc.lockin_means(x[b * R:(b + 1) * R], w0, nh), g["qi"][b])


def test_full_cfg5_subset_bit_exact(golden):
    g = golden("full_cfg5")
    assert g["rows"].shape == (19, 1000, 7)
    for a, m in enumerate(g["ms"]):
        for t in (0, 1, 499, 999):
            x = orc.snr_signal(float(m), 200e3, 1000.0, 1e-3, 40.0, seed=t)
            assert np.array_equal(orc.nls_fit(x, 200e3, 1000.0, 1, 15, init_m=float(m))[0], g["rows"][a, t])


@pytest.mark.parametrize("name", ["drift_phi_1um", "drift_phi_slow"])
def test_drifting_records_bit_exact(golden, name):
    """'asd'-mode physics restated by the oracle (bit-equal record) and all three reference schedules on it."""
    g = golden(name)
    m, fs, fm, secs, trial, amp_n, aamp, af = g["meta"]
    x, truth = orc.asd_signal(m, fs, fm, secs, trial=int(trial), amp_n=amp_n, arml_mod_amp=aamp, arml_mod_f=af)
    assert np.array_equal(x[:16], g["x_head"]) and np.array_equal(x[-16:], g["x_tail"])
    assert x.sum() == g["x_sum"][0] and np.abs(x).sum() == g["x_sum"][1]
    assert np.array_equal(truth[::4000], g["phi_sim"])
    assert np.array_equal(orc.nls_fit(x, fs, fm, 20, 10, schedule="sequential"), g["rows_seq"])
    assert np.array_equal(orc.nls_fit(x, fs, fm, 20, 10, schedule="seeded", n_chunks=3), g["rows_par3"])
    assert np.array_equal(orc.nls_fit(x, fs, fm, 20, 10, schedule="seeded", n_chunks=8), g["rows_par8"])
    # the schedule is observable on these records: seeding every buffer from buffer 0 changes flags
    each = orc.nls_fit(x, fs, fm, 20, 10, schedule="gpu")
    assert not np.array_equal(each[:, 6], g["rows_seq"][:, 6])


def test_full_ekf_channel_prefix_bit_exact(golden):
    """The oracle's loop against EKFFitter.fit on the first 0.25 s (50 000 steps) of a cfg-4 channel.  The filter's
    initial dc and R are whole-record moments, so the prefix is run with those of the full second."""
    g = golden("full_ekf_8ch")
    c = g["channels"][3]
    z = orc.snr_signal(6.0, 200e3, 1000.0, 1.0, 40.0, seed=int(c), phi0=2 * np.pi * c / 4096)
    assert np.array_equal(z[:16], g["x_head"][3])
    rows = orc.ekf_track(z[:48_000], 200e3, 1000.0, 20, r_val=np.var(z), init_dc=np.mean(z))
    assert np.array_equal(rows[:, :5], g["rows"][3][:12, :5])
