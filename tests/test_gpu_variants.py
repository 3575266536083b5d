"""Every build of the LM and EKF kernels that a launcher can select, held to the oracle.

The launchers pick a build from the problem size (dfk_b200.cu: pick_lanes, launch_first, launch_lm, the EKF
channels-per-warp rule), so the small records of the parity tests only reach a few of them.  Here each build is forced
with opts.lanes_per_fit or a development override and run on inputs the oracle has rows for, and the profiler shows
that the intended kernel is the one that ran (routing can bypass an override: a handful of fits go to one-warp blocks
whatever is set).  Also here: the EKF's checked replay past |w_m t| = 1e6, every DRIFT = true build of the folding
demodulation, and the grid statistics at their slice boundaries and non-finite edges.
"""
import math
import os

import numpy as np
import pytest

from oracle import dfmi_oracle as orc
from tests.test_gpu_parity import IQ_TOL, PARAM_TOL, _bulk_case, _case, assert_rows_match, gpu_demod

pytestmark = pytest.mark.gpu

EKF_TOL = 1e-11
F_SAMP, F_MOD = 200e3, 1000.0


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


def launched_kernels(fn):
    """Run fn() under torch.profiler (CUDA activity); return its result and the names of the kernels it launched
    (spaces removed, e.g. 'voiddfk::lm_first_kernel<2,5,128>(...)')."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, {e.name.replace(" ", "") for e in prof.events()}


def ran(names, kernel):
    """Whether the kernel dfk::<kernel> (template arguments included) is among the launched names."""
    k = "dfk::" + kernel.replace(" ", "")
    return any(k + "(" in n or n.endswith(k) for n in names)


def assert_ran(names, kernel):
    assert ran(names, kernel), (kernel, sorted(n.split("(")[0] for n in names))


# ---- 1. LM builds ---------------------------------------------------------------------------------------
# (lanes_per_fit, overrides, kernel that must run).  G = 1 cold fits take the per-lane state machine unless
# DFK_LM_FLAT = 0; MINB 4 / 5 are the 128- and 96-register builds of one PTX.
LM_COLD = ([(g, dict(DFK_LM_MINB=mb), f"lm_first_kernel<{g}, {mb}, 128>") for g in (2, 4, 8, 16, 32) for mb in (4, 5)]
           + [(1, dict(DFK_LM_FLAT=0, DFK_LM_MINB=mb), f"lm_first_kernel<1, {mb}, 128>") for mb in (4, 5)]
           + [(1, {}, "lm_flat_kernel<4>")])
LM_COLD_IDS = [k.replace(", ", "_").replace("<", "-").replace(">", "") for _, _, k in LM_COLD]
W0_BANK = 2.0 * np.pi * F_MOD / F_SAMP
FLAT_RETRY_MIN = 4096  # kFlatRetryMin: from this many parked fits the retry stage is a thread per fit


@pytest.fixture(scope="module")
def lm_bank():
    """The 1200 random cold starts of test_bulk_parity_over_random_cold_starts and their oracle rows; the tilings
    that put the retry stage on the warp-per-fit kernel ('warp': 4 copies, 4800 fits, so lm_retry_flat_kernel is
    launched too but stands aside) and on the thread-per-fit kernel ('flat': enough copies to park >= 4096)."""
    from multiprocessing import Pool
    rng = np.random.RandomState(2024)
    n = 1200
    ms = rng.uniform(2.0, 22.0, n)
    snrs = rng.choice([3.0, 10.0, 20.0, 40.0], n)
    init_m = np.where(rng.rand(n) < 0.5, 6.0, ms)
    phis, psis = rng.uniform(-3, 3, n), rng.uniform(-0.5, 0.5, n)
    jobs = [(ms[i], snrs[i], 1000 + i, init_m[i], phis[i], psis[i]) for i in range(n)]
    with Pool(min(16, os.cpu_count() or 1)) as pool:
        res = pool.map(_bulk_case, jobs, chunksize=25)
    x = np.stack([r[0] for r in res])
    ref = np.stack([r[1] for r in res])
    parked = int(np.sum(ref[:, 6] >= 1))  # a fit ends with flag 1 or 2 exactly when its first descent was parked
    tiles = {"warp": 4, "flat": -(-FLAT_RETRY_MIN // parked)}
    assert 4 * parked < FLAT_RETRY_MIN <= tiles["flat"] * parked, parked
    return {"x": x, "ref": ref, "init_m": init_m, "parked": parked, "tiles": tiles, "cache": {}}


def _lm_cold(torch, ctx, bank, retry, i):
    """Rows of variant LM_COLD[i] on the bank tiled for `retry`, cached; checks which kernels ran on the way."""
    from deepfmkit_b200 import _lib
    key = (retry, i)
    if key in bank["cache"]:
        return bank["cache"][key]
    lanes, over, kernel = LM_COLD[i]
    k = bank["tiles"][retry]
    x = np.tile(bank["x"], (k, 1))
    C = x.shape[0]
    xd = torch.from_numpy(x).cuda()
    g = np.zeros((C, 4))
    g[:, 0] = 1.6
    g[:, 1] = np.tile(bank["init_m"], k)
    gd = torch.from_numpy(g).cuda()
    rows = torch.full((C, 1, 8), float("nan"), dtype=torch.float64, device="cuda")
    opts = _lib.default_lm_opts()
    opts.lanes_per_fit = lanes

    def call():
        ctx.nls_fit_batch_dev(xd.data_ptr(), C, 1, 400, 400, 12, W0_BANK, [1.6, 6.0, 0.0, 0.0], gd.data_ptr(), 4,
                              False, opts, rows.data_ptr())
        ctx.synchronize()

    ctx.lm_counters(reset=True)
    with _lib.dev_overrides(**over):
        _, names = launched_kernels(call)
    parked = ctx.lm_counters(reset=True)["n_grid"]  # one grid search per parked fit, in either retry kernel
    assert_ran(names, kernel)
    assert_ran(names, "lm_retry_kernel")
    assert_ran(names, "lm_retry_flat_kernel")
    bank["cache"][key] = rows.cpu().numpy()[:, 0, :], parked
    return bank["cache"][key]


def assert_fits_match(rows, ref):
    """Flags identical to the oracle; amp and m within PARAM_TOL relative, phi and psi within PARAM_TOL absolute
    wherever the reference fits (flag 0 or 1)."""
    diff = np.flatnonzero(rows[:, 6] != ref[:, 6])
    assert diff.size == 0, (diff, rows[diff, :7], ref[diff])
    ok = ref[:, 6] < 2
    err = np.abs(rows[ok, :4] - ref[ok, :4])
    err[:, :2] /= np.abs(ref[ok, :2])
    assert err.max() <= PARAM_TOL, (err.max(), np.unravel_index(err.argmax(), err.shape))


@pytest.mark.parametrize("i", range(len(LM_COLD)), ids=LM_COLD_IDS)
@pytest.mark.parametrize("retry", ["warp", "flat"])
def test_lm_cold_build_vs_oracle(torch_mod, ctx, lm_bank, retry, i):
    """One forced build of the first descent (and the retry kernel the number of parked fits selects) on every fit of
    the tiled bank: each copy of the bank gives the same rows bit for bit (no dependence on a fit's lane, block or
    place in the retry list), those rows match the oracle's, and exactly the fits the oracle had to retry were
    handed to the retry stage."""
    rows, parked = _lm_cold(torch_mod, ctx, lm_bank, retry, i)
    n = len(lm_bank["ref"])
    copies = rows.reshape(-1, n, 8)
    assert all(np.array_equal(c, copies[0], equal_nan=True) for c in copies[1:])
    assert_fits_match(copies[0], lm_bank["ref"])
    assert parked == len(copies) * lm_bank["parked"], (parked, len(copies), lm_bank["parked"])
    assert (parked >= FLAT_RETRY_MIN) == (retry == "flat")


MINB_PAIRS = [(f"lm_first_kernel<{g}, 4, 128>", f"lm_first_kernel<{g}, 5, 128>") for g in (1, 2, 4, 8, 16, 32)]


@pytest.mark.parametrize("pair", MINB_PAIRS, ids=[f"{a}-vs-{b}" for a, b in MINB_PAIRS])
def test_lm_cold_register_budgets_are_bit_equal(torch_mod, ctx, lm_bank, pair):
    """Builds that differ only in __launch_bounds__' blocks per SM come from one PTX: the same rows, bit for bit."""
    kernels = [k for _, _, k in LM_COLD]
    for retry in ("warp", "flat"):
        a = _lm_cold(torch_mod, ctx, lm_bank, retry, kernels.index(pair[0]))[0]
        b = _lm_cold(torch_mod, ctx, lm_bank, retry, kernels.index(pair[1]))[0]
        assert np.array_equal(a, b, equal_nan=True), retry


def test_lm_cold_builds_pairwise_equality(torch_mod, ctx, lm_bank):
    """Which of the other builds agree to the bit (printed, not asserted: a lane count changes the order in which
    a fit's harmonic sums are reduced, so they agree to the oracle's gate, not necessarily to the bit).  On a B200,
    with either retry kernel, only G = 16 and G = 32 gave the same rows (N = 12 harmonics: both give every harmonic
    its own lane); the flat kernel against the lock-step G = 1 build and every other G against G differ."""
    kernels = [k for _, _, k in LM_COLD]
    pairs = [("lm_flat_kernel<4>", "lm_first_kernel<1, 4, 128>")] + \
        [(f"lm_first_kernel<{a}, 4, 128>", f"lm_first_kernel<{b}, 4, 128>") for a, b in
         ((1, 2), (2, 4), (4, 8), (8, 16), (16, 32), (1, 32))]
    for retry in ("warp", "flat"):
        for a, b in pairs:
            ra = _lm_cold(torch_mod, ctx, lm_bank, retry, kernels.index(a))[0]
            rb = _lm_cold(torch_mod, ctx, lm_bank, retry, kernels.index(b))[0]
            same = np.array_equal(ra, rb, equal_nan=True)
            print(f"LM pair {retry:4s} {a} vs {b}: {'bit-equal' if same else 'differs'}")


LM_WARM = [(g, dict(DFK_LM_MINB=mb), f"lm_first_kernel<{g}, {mb}, 128>") for g in (2, 8, 16) for mb in (4, 5)]
GOLDEN_NLS = ["cfg1_quickstart", "cfg2_1mhz", "cfg3_channel", "deep_mod_n62", "fallback_m16", "pathological_m3", "low_snr"]


@pytest.mark.parametrize("name", GOLDEN_NLS)
def test_lm_warm_builds_vs_reference(torch_mod, ctx, golden, name):
    """Warm-started readouts (every buffer from buffer 0's result) of the golden records through the builds that
    bigger batches select -- G = 2, 8, 16 at both register budgets -- against the reference's own rows."""
    from deepfmkit_b200 import _lib
    g, x, f_samp, f_mod, n, nh, R, w0 = _case(golden, name)
    meta = g["meta"]
    got = {}
    for lanes, over, kernel in LM_WARM:
        opts = _lib.default_lm_opts()
        opts.lanes_per_fit = lanes
        with _lib.dev_overrides(**over):
            rows, names = launched_kernels(
                lambda: ctx.nls_fit_host(x, R, nh, w0, [meta[11], meta[12], 0.0, meta[13]], seeded=True, opts=opts))
        assert_ran(names, kernel)
        assert_rows_match(rows, g["rows_seq"])
        if len(g["rows_par"]):
            assert_rows_match(rows, g["rows_par"])
        got[kernel] = rows
    for gl in (2, 8, 16):
        assert np.array_equal(got[f"lm_first_kernel<{gl}, 4, 128>"], got[f"lm_first_kernel<{gl}, 5, 128>"], equal_nan=True)


# ---- 2. EKF channels per warp -----------------------------------------------------------------------------
EKF_C, EKF_T, EKF_R = 67, 12_123, 4000
EKF_CHECK = (0, 1, 7, 8, 31, 32, 33, 63, 64, 66)  # both sides of every warp boundary for cpw 1..32, and the last
EKF_EXPLICIT = dict(init_a=1.1, init_m=6.0, init_phi=0.15, init_psi=0.02, p0_diag=np.array([0.5, 0.8, 1.2, 0.3, 0.6]),
                    q_diag=np.array([2e-8, 1e-8, 2e-6, 5e-7, 1e-8]), r_val=1e-3, init_dc=1.05)


def _ekf_ref(args):
    z, kw = args
    return orc.ekf_track(z, F_SAMP, F_MOD, 20, **kw)


def _ekf_opts(kw):
    from deepfmkit_b200 import _lib
    o = _lib.default_ekf_opts()
    if kw:
        o.init[0], o.init[1], o.init[2], o.init[3] = kw["init_a"], kw["init_m"], kw["init_phi"], kw["init_psi"]
        for i in range(5):
            o.p0_diag[i], o.q_diag[i] = kw["p0_diag"][i], kw["q_diag"][i]
        o.r_val, o.init_dc = kw["r_val"], kw["init_dc"]
    return o


@pytest.fixture(scope="module")
def ekf_bank():
    """67 channels (ragged for every cpw > 1) of 12 123 samples (a ragged last tile and buffer), distinct seeds, m
    and phi0, with the oracle's rows of the checked channels under default and explicit options."""
    from multiprocessing import Pool
    rng = np.random.RandomState(67)
    ms, phis = rng.uniform(3.0, 12.0, EKF_C), rng.uniform(-3.0, 3.0, EKF_C)
    z = np.stack([orc.snr_signal(ms[c], F_SAMP, F_MOD, 0.07, 40.0, seed=300 + c, phi0=phis[c])[:EKF_T]
                  for c in range(EKF_C)])
    # the explicit options start every channel from one guess: channels near it, so that every filter locks (a
    # filter that loses lock turns rounding differences into large ones, and the comparison says nothing)
    rng = np.random.RandomState(68)
    ms, phis = rng.uniform(5.95, 6.05, EKF_C), rng.uniform(0.1, 0.2, EKF_C)
    ze = np.stack([orc.snr_signal(ms[c], F_SAMP, F_MOD, 0.07, 40.0, seed=400 + c, phi0=phis[c])[:EKF_T]
                   for c in range(EKF_C)])
    jobs = [(z[c], {}) for c in EKF_CHECK] + [(ze[c], EKF_EXPLICIT) for c in EKF_CHECK]
    with Pool(min(16, os.cpu_count() or 1)) as pool:
        refs = pool.map(_ekf_ref, jobs)
    return {"z": z, "z_explicit": ze, "ref": dict(zip(EKF_CHECK, refs[:len(EKF_CHECK)])),
            "ref_explicit": dict(zip(EKF_CHECK, refs[len(EKF_CHECK):]))}


def _ekf_run(torch, ctx, z, layout, cpw, kw=None):
    from deepfmkit_b200 import _lib
    C, T = z.shape
    if layout == "channel_major":
        zd, ld_t, ld_c = torch.from_numpy(np.ascontiguousarray(z)).cuda(), 1, T
    else:
        zd, ld_t, ld_c = torch.from_numpy(np.ascontiguousarray(z.T)).cuda(), C, 1
    rows = torch.full((C, T // EKF_R, 8), float("nan"), dtype=torch.float64, device="cuda")
    opts = _ekf_opts(kw)
    over = dict(DFK_EKF_CPW=cpw) if cpw else {}

    def call():
        ctx.ekf_dev(zd.data_ptr(), T, C, ld_t, ld_c, EKF_R, F_SAMP, F_MOD, opts, rows.data_ptr())
        ctx.synchronize()

    with _lib.dev_overrides(**over):
        _, names = launched_kernels(call)
    assert_ran(names, "ekf_kernel")
    return rows.cpu().numpy()


def assert_ekf_rows(rows, ref):
    assert np.max(np.abs(rows[:, :5] - ref[:, :5])) < EKF_TOL
    assert np.all(rows[:, 5] == 0) and np.all(rows[:, 6] == 1)


@pytest.mark.parametrize("layout", ["channel_major", "time_major"])
def test_ekf_channels_per_warp(torch_mod, ctx, ekf_bank, layout):
    """DFK_EKF_CPW in {1, ..., 32}: a lane's arithmetic does not depend on it, so every value gives cpw 1's rows bit
    for bit, and those match the oracle on both sides of every warp boundary (initial dc and R from each channel's
    own statistics)."""
    z = ekf_bank["z"]
    base = _ekf_run(torch_mod, ctx, z, layout, 1)
    for c in EKF_CHECK:
        assert_ekf_rows(base[c], ekf_bank["ref"][c])
    for cpw in (2, 4, 8, 16, 32):
        rows = _ekf_run(torch_mod, ctx, z, layout, cpw)
        assert np.array_equal(rows, base), cpw


def test_ekf_channels_per_warp_explicit_options(torch_mod, ctx, ekf_bank):
    """Options given in full (initial state, P0, Q, R, dc): the same bit-equality over cpw, the oracle's rows."""
    z = ekf_bank["z_explicit"]
    base = _ekf_run(torch_mod, ctx, z, "channel_major", 1, EKF_EXPLICIT)
    for c in EKF_CHECK:
        assert_ekf_rows(base[c], ekf_bank["ref_explicit"][c])
    for cpw in (2, 4, 8, 16, 32):
        assert np.array_equal(_ekf_run(torch_mod, ctx, z, "channel_major", cpw, EKF_EXPLICIT), base), cpw


def test_ekf_heuristic_channels_per_warp(torch_mod, ctx):
    """1200 channels: the launcher packs 4 per warp (300 warps on 592 sub-partitions of a 148-SM B200); the same
    rows as one per warp, and the oracle's on a sample that includes the last channel."""
    from multiprocessing import Pool
    torch = torch_mod
    C, T = 1200, 8000
    xd = torch.empty((C, T), dtype=torch.float64, device="cuda")
    ctx.synth_snr_dev(xd.data_ptr(), T, C, F_SAMP, F_MOD, 7.0, dphi=0.37, snr_db=40.0, seed=1200)
    ctx.synchronize()
    z = xd.cpu().numpy()
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    cpw = 1
    while cpw < 32 and -(-C // cpw) > 4 * sm:
        cpw *= 2
    if sm == 148:
        assert cpw == 4
    auto = _ekf_run(torch, ctx, z, "channel_major", 0)
    one = _ekf_run(torch, ctx, z, "channel_major", 1)
    assert np.array_equal(auto, one)
    sample = (0, 3, 4, 599, 1196, 1199)
    with Pool(len(sample)) as pool:
        refs = pool.map(_ekf_ref, [(z[c], {}) for c in sample])
    for c, ref in zip(sample, refs):
        assert_ekf_rows(auto[c], ref)


# ---- 3. EKF checked replay ----------------------------------------------------------------------------------
REPLAY_R = 200  # n = 1 at 200 kHz / 1 kHz: a snapshot per period


def _tri(i, j):
    return i * 5 - (i * (i - 1)) // 2 + (j - i)


def _replay_inputs(k0, n, seed, nan_at=None):
    """A slab of n samples starting at absolute sample k0, synthesised at absolute time, and a carried filter state
    near the truth with a full (non-diagonal) covariance, as the kernel stores it."""
    rng = np.random.RandomState(seed)
    t = (k0 + np.arange(n)) / F_SAMP
    z = 1.1 + 1.0 * np.cos(0.7 + 6.2 * np.cos(2 * np.pi * F_MOD * t + 0.05)) + 0.01 * rng.randn(n)
    if nan_at is not None:
        z[nan_at] = np.nan
    x0 = np.array([1.02, 6.15, 0.68, 0.052, 1.098])
    L = 1e-4 * rng.randn(5, 5)
    P = L @ L.T + np.diag([1e-6, 2e-6, 1e-5, 1e-6, 1e-7])
    r = 1e-3  # above the noise variance (1e-4): a filter whose rows move by ~1e-15 when r moves by an ulp
    state = np.zeros(32)
    state[:5] = x0
    for i in range(5):
        for j in range(i, 5):
            state[5 + _tri(i, j)] = P[i, j]
    state[30] = r
    kw = dict(init_a=x0[0], init_m=x0[1], init_phi=x0[2], init_psi=x0[3], init_dc=x0[4], r_val=r, init_cov=P, k0=k0)
    return z, state, kw


def _replay_ref(args):
    z, kw = args
    return orc.ekf_track(z, F_SAMP, F_MOD, REPLAY_R // 200, **kw)


CROSS_SPLIT = 4800  # 150 tiles, 24 buffers: the second call starts 189 samples before the carrier angle reaches 1e6
REPLAY_CASES = {"crossing": (31_826_000, 24_000, 1, None), "one_hour": (720_000_000, 20_000, 2, None),
                "nan_mid_tile": (4_000_000, 8000, 3, 2005)}

@pytest.fixture(scope="module")
def replay_refs():
    from multiprocessing import Pool
    inputs = {k: _replay_inputs(*v) for k, v in REPLAY_CASES.items()}
    with Pool(len(inputs)) as pool:
        refs = pool.map(_replay_ref, [(z, kw) for z, _, kw in inputs.values()])
    return {k: (inp, ref) for (k, inp), ref in zip(inputs.items(), refs)}


def _stream(torch, ctx, z, state, k0):
    from deepfmkit_b200 import _lib
    T = len(z)
    zd = torch.from_numpy(z[None, :].copy()).cuda()
    sd = torch.from_numpy(state[None, :].copy()).cuda()
    rows = torch.full((1, T // REPLAY_R, 8), float("nan"), dtype=torch.float64, device="cuda")
    opts = _lib.default_ekf_opts()

    def call():
        ctx.ekf_stream_dev(zd.data_ptr(), T, 1, 1, T, REPLAY_R, F_SAMP, F_MOD, opts, k0, sd.data_ptr(), rows.data_ptr())
        ctx.synchronize()

    _, names = launched_kernels(call)
    assert_ran(names, "ekf_kernel")
    return rows.cpu().numpy()[0], sd.cpu().numpy()[0]


@pytest.mark.parametrize("case", list(REPLAY_CASES))
def test_ekf_checked_replay_vs_oracle(torch_mod, ctx, replay_refs, case):
    """Continuation slabs of dfk_ekf_stream_dev (state carried in by hand: x, the covariance's upper triangle in
    tri(i, j) order, r) deep into a record, against the oracle resumed from the same state at the same k0.

    The fast step reduces angles by Cody-Waite, exact only for |angle| < 1e6; a 32-sample tile in which any carrier
    angle w_m t_k + psi (or S, or the inner argument) left that range is rerun from the state saved at the tile's
    entry with the checked routines.  At 200 kHz / 1 kHz the carrier angle reaches 1e6 at k = 31 830 989 (159 s):
    'crossing' (k0 = 31 826 000, 24 000 samples) runs 4 989 samples of fast tiles, then the tile that holds that
    sample, then 19 000 samples of replayed tiles; 'one_hour' (k0 = 7.2e8, 3600 s) replays every tile.

    'crossing' is also run as two calls cut at sample 4800, a tile and buffer boundary: their rows must be the whole
    call's bit for bit.  The first part is held to the oracle from the hand-built state, the second to the oracle
    resumed from the state the first call carried out.  The whole slab is not held to one oracle run at 1e-11.  At an
    angle near 1e6 one ulp of w_m t_k + psi is 1.2e-10 rad.  The fast tiles leave psi ~1e-14 from the oracle's (their
    sincos and gain are accurate to rounding, not bit-equal to numpy), so over thousands of later steps the two
    carrier angles now and then round to neighbouring doubles.  Each such step moves the state by ~1e-11.  Measured on
    a B200: 1.0e-11 after 60 000 fast steps from k0 = 31 700 000 with no tile replayed.  Resuming the oracle from the
    kernel's own state at the cut removes that inherited difference, so the switch and the replay are held to 1e-11.

    'nan_mid_tile' puts a NaN at sample 2005 of the slab, inside the tile [1984, 2016) that also holds the snapshot
    after sample 1999 (row 9).  The NaN sample makes the state NaN; the next step's carrier angle (psi is NaN) fails
    the range check, so the tile is replayed and row 9 rewritten.  Rows 0-9 must still be the oracle's and every later
    row NaN, as in the oracle.  (A NaN on a tile's last sample fails the check only in the next tile, which is then
    the one replayed.)"""
    (z, state, kw), ref = replay_refs[case]
    k0 = kw["k0"]
    rows = _stream(torch_mod, ctx, z, state, k0)[0]
    assert np.all(rows[:, 5] == 0) and np.all(rows[:, 6] == 1)
    bad = np.isnan(ref[:, :5]).any(axis=1)
    assert np.array_equal(np.isnan(rows[:, :5]), np.isnan(ref[:, :5]))
    if case == "nan_mid_tile":
        assert not bad[:10].any() and bad[10:].all()
    else:
        assert not bad.any()
    if case != "crossing":
        assert np.max(np.abs(rows[~bad, :5] - ref[~bad, :5])) < EKF_TOL
        return
    # the same slab as two calls cut at the tile boundary CROSS_SPLIT (a whole number of buffers): bit for bit the
    # whole call's rows, so the first call's fast tiles and the second call's switch and replay are the whole call's
    a, state_a = _stream(torch_mod, ctx, z[:CROSS_SPLIT], state, k0)
    b, _ = _stream(torch_mod, ctx, z[CROSS_SPLIT:], state_a, k0 + CROSS_SPLIT)
    assert np.array_equal(np.concatenate([a, b]), rows)
    nb = CROSS_SPLIT // REPLAY_R
    assert np.max(np.abs(rows[:nb, :5] - ref[:nb, :5])) < EKF_TOL
    # the second part against the oracle resumed from the state the first call carried out (read back in the layout
    # the kernel writes: x, the upper triangle in tri(i, j) order, r)
    P = np.zeros((5, 5))
    for i in range(5):
        for j in range(i, 5):
            P[i, j] = P[j, i] = state_a[5 + _tri(i, j)]
    ref_b = orc.ekf_track(z[CROSS_SPLIT:], F_SAMP, F_MOD, REPLAY_R // 200, init_a=state_a[0], init_m=state_a[1],
                          init_phi=state_a[2], init_psi=state_a[3], init_dc=state_a[4], r_val=state_a[30], init_cov=P,
                          k0=k0 + CROSS_SPLIT)
    assert np.max(np.abs(b[:, :5] - ref_b[:, :5])) < EKF_TOL
    assert np.array_equal(_stream(torch_mod, ctx, z, state, k0)[0], rows)

# ---- 4. forced drift term --------------------------------------------------------------------------------
EXTREME_SHAPES = [(2048, 3, 10), (1536, 2, 7), (1000, 1, 64), (6, 50, 2), (2, 40, 1), (256, 5, 31), (258, 4, 16),
                  (200, 3, 40), (2050, 2, 5), (75, 20, 10), (100, 1, 10), (256, 1, 31), (4, 1, 1), (8, 1, 3),
                  (200, 1, 40), (202, 1, 10), (12, 1, 5), (200, 1, 16), (75, 1, 10), (333, 6, 12), (1001, 2, 9),
                  (4096, 3, 10), (10000, 2, 10), (16384, 2, 20), (2501, 2, 7), (10000, 20, 64), (6144, 1, 3),
                  (2052, 5, 64)]
TM_SHAPES = [(200, 20, 10, 256, 7), (200, 20, 10, 1, 9), (1000, 20, 10, 2, 5), (200, 3, 62, 5, 11), (128, 1, 15, 33, 4),
             (2000, 40, 40, 3, 3), (76, 2, 7, 27, 6)]


def _demod_names(names):
    return {n.split("(")[0].replace("void", "") for n in names if "demod_" in n or "project_interleaved" in n}


def test_forced_drift_channel_major_folds(torch_mod, ctx):
    """The shapes of test_demod_period_and_harmonic_extremes with DFK_FOLD_DRIFT = 1: every folding shape runs a
    DRIFT = true build (register fold at slot counts 1-4, column-chunked fold, tile kernel), and the first-order
    frequency-offset term holds the lock-in to IQ_TOL at any ramp."""
    from deepfmkit_b200 import _lib
    seen = set()
    for P, n, nh in EXTREME_SHAPES:
        f_samp = F_MOD * P
        R = P * n
        w0 = orc.rad_per_sample(f_samp, F_MOD)
        rng = np.random.RandomState(P + n)
        nbuf = 37
        t = np.arange(nbuf * R)
        x = 1.0 + np.cos(0.7 + 3.0 * np.cos(2 * np.pi * t / P + 0.2)) + 0.01 * rng.randn(nbuf * R)
        with _lib.dev_overrides(DFK_FOLD_DRIFT=1):
            (qi, dc), names = launched_kernels(lambda: gpu_demod(torch_mod, ctx, x, R, nh, w0))
        builds = _demod_names(names)
        if P % 2 == 0 or n % 2 == 0:
            assert builds and all("<true" in b for b in builds), (P, n, builds)
        seen |= builds
        for b in (0, 1, 17, nbuf - 1):
            buf = x[b * R:(b + 1) * R]
            ref = orc.lockin_means(buf, w0, nh)
            assert np.max(np.abs(qi[b] - ref)) <= IQ_TOL * max(np.abs(ref).max(), 1e-3), (P, n, nh, b)
            assert abs(dc[b] - buf.mean()) <= 1e-14 * abs(buf.mean())
    for k in ("demod_fold_kernel<true,1>", "demod_fold_kernel<true,2>", "demod_fold_kernel<true,3>",
              "demod_fold_kernel<true,4>", "demod_fold_long_kernel<true,false>"):
        assert "dfk::" + k in seen, (k, sorted(seen))
    assert any(s.startswith("dfk::demod_tile_kernel<true,") for s in seen), sorted(seen)


def test_forced_drift_time_major_fold(torch_mod, ctx):
    """The shapes of test_time_major_demod_matches_reference_lockin with DFK_FOLD_DRIFT = 1: the interleaved fold and
    its projection in their DRIFT = true builds, against the oracle's lock-in of every checked channel."""
    from deepfmkit_b200 import _lib
    torch = torch_mod
    for P, n, nh, C, nbuf in TM_SHAPES:
        f_samp = F_MOD * P
        R = P * n
        w0 = orc.rad_per_sample(f_samp, F_MOD)
        rng = np.random.RandomState(P + C)
        t = np.arange(nbuf * R)
        x = np.stack([1.0 + np.cos(0.3 * c + (3.0 + 0.01 * c) * np.cos(2 * np.pi * t / P + 0.2)) + 0.01 * rng.randn(nbuf * R)
                      for c in range(C)], axis=1)
        xd = torch.from_numpy(np.ascontiguousarray(x)).cuda()
        qi = torch.full((C * nbuf, 2 * nh), float("nan"), dtype=torch.float64, device="cuda")
        dc = torch.full((C * nbuf,), float("nan"), dtype=torch.float64, device="cuda")

        def call():
            ctx.demod_tm(xd.data_ptr(), nbuf, C, R, nh, w0, qi.data_ptr(), dc.data_ptr())
            ctx.synchronize()

        with _lib.dev_overrides(DFK_FOLD_DRIFT=1):
            _, names = launched_kernels(call)
        builds = _demod_names(names)
        assert builds == {"dfk::demod_fold_long_kernel<true,true>", "dfk::project_interleaved_kernel<true>"}, builds
        q, d = qi.cpu().numpy().reshape(C, nbuf, 2 * nh), dc.cpu().numpy().reshape(C, nbuf)
        for c in sorted({0, C // 2, C - 1}):
            for b in sorted({0, nbuf - 1}):
                buf = x[b * R:(b + 1) * R, c]
                ref = orc.lockin_means(buf, w0, nh)
                assert np.max(np.abs(q[c, b] - ref)) <= IQ_TOL * max(np.abs(ref).max(), 1e-3), (P, n, C, c, b)
                assert abs(d[c, b] - buf.mean()) <= 1e-14 * abs(buf.mean())



def test_drift_term_carries_weight(torch_mod, ctx):
    """In the shapes above the frequency offset is only the rounding of w0, so the drift term is nearly zero and a
    wrong sign or index in it would go unseen.  Here it is not: 2000 periods of 200 samples per buffer, 64 harmonics
    and a deep modulation (m = 20, harmonics up to ~20 carry weight) give a phase ramp of ~1e-10 rad over a buffer
    at the top harmonic.  With the term the lock-in holds IQ_TOL; without it (DFK_FOLD_DRIFT = 0) it misses by
    several times that."""
    from deepfmkit_b200 import _lib
    P, n, nh, nbuf = 200, 2000, 64, 3
    R, w0 = P * n, orc.rad_per_sample(F_MOD * P, F_MOD)
    rng = np.random.RandomState(2000)
    t = np.arange(nbuf * R)
    x = 1.0 + np.cos(0.7 + 20.0 * np.cos(2 * np.pi * t / P + 0.2)) + 0.01 * rng.randn(nbuf * R)
    refs = [orc.lockin_means(x[b * R:(b + 1) * R], w0, nh) for b in range(nbuf)]
    err = {}
    for drift in (1, 0):
        with _lib.dev_overrides(DFK_FOLD_DRIFT=drift):
            (qi, _), names = launched_kernels(lambda: gpu_demod(torch_mod, ctx, x, R, nh, w0))
        builds = _demod_names(names)
        assert builds and all(f"<{'true' if drift else 'false'}" in b for b in builds), builds
        err[drift] = max(np.max(np.abs(qi[b] - refs[b])) / np.abs(refs[b]).max() for b in range(nbuf))
    assert err[1] <= IQ_TOL, err
    assert err[0] > 4 * IQ_TOL, err

# ---- 5. grid statistics ----------------------------------------------------------------------------------------
def _col_ref(col, center=None):
    """nanmean (exact sum), nanstd, nanmin, nanmax, the first trial farthest from the centre (default: the mean),
    count -- with the reference's rules for infinities."""
    fin = col[~np.isnan(col)]
    nan = float("nan")
    if fin.size == 0:
        return [nan, nan, nan, nan, nan, 0.0]
    if np.isposinf(fin).any() and np.isneginf(fin).any():
        mean = nan
    else:
        mean = math.fsum(fin) / fin.size
    with np.errstate(all="ignore"):
        std = float(np.sqrt(np.mean((fin - np.mean(fin)) ** 2)))
        dist = np.abs(col - (mean if center is None else center))
    worst = nan if np.isnan(dist).all() else col[np.nanargmax(dist)]
    return [mean, std, fin.min(), fin.max(), worst, float(fin.size)]


def _trial_stats(torch, ctx, v, ncols, center=None):
    """dfk_trial_stats_dev on v[P, T, stride]; the output is followed by a guard record that must stay untouched."""
    P = v.shape[0]
    vd = torch.from_numpy(np.ascontiguousarray(v)).cuda()
    out = torch.full((P * ncols + 1, 6), -7.25, dtype=torch.float64, device="cuda")
    cd = torch.from_numpy(np.ascontiguousarray(center)).cuda() if center is not None else None

    def call():
        ctx.trial_stats_dev(vd.data_ptr(), P, v.shape[1], ncols, v.shape[2], out.data_ptr(),
                            center_ptr=cd.data_ptr() if cd is not None else None)
        ctx.synchronize()

    _, names = launched_kernels(call)
    assert_ran(names, "trial_stats_finish")
    o = out.cpu().numpy()
    assert np.all(o[-1] == -7.25)
    return o[:-1].reshape(P, ncols, 6)


def assert_stats(got, ref, col):
    mean, std, mn, mx, worst, count = ref
    scale = np.nanmax(np.abs(col[np.isfinite(col)])) if np.isfinite(col).any() else 0.0
    if np.isfinite(mean):
        assert abs(got[0] - mean) <= 1e-13 * abs(mean) + 1e-15 * scale, (got[0], mean)
    else:
        assert np.array_equal(got[0], mean, equal_nan=True), (got[0], mean)
    if np.isfinite(std):
        assert abs(got[1] - std) <= 1e-12 * std + 1e-15 * scale, (got[1], std)
    else:
        assert np.isnan(got[1]), got[1]
    assert np.array_equal(got[2:], [mn, mx, worst, count], equal_nan=True), (got[2:], [mn, mx, worst, count])


@pytest.mark.parametrize("npoints", [1, 19])
@pytest.mark.parametrize("ntrials", [1, 255, 256, 257, 16_385, 100_003])
def test_trial_stats_slices_vs_numpy(torch_mod, ctx, ntrials, npoints):
    """One slice (up to 256 trials) to 64 with a ragged last one; 7 result columns in records of 8 whose 8th holds
    NaN / 1e300 and must never be read; ~2 % NaN trials, one column mostly NaN."""
    rng = np.random.RandomState(ntrials + npoints)
    v = np.empty((npoints, ntrials, 8))
    v[..., :7] = rng.randn(npoints, ntrials, 7) * [1.0, 1e-3, 5.0, 1.0, 2.0, 1.0, 1e8] + [0.0, 6.0, 0.0, 1e3, -3.0, 0.0, 0.0]
    v[..., :7][rng.rand(npoints, ntrials, 7) < 0.02] = np.nan
    v[..., 5][rng.rand(npoints, ntrials) < 0.7] = np.nan
    v[..., 7] = np.where(np.arange(ntrials) % 2 == 0, np.nan, 1e300)
    s = _trial_stats(torch_mod, ctx, v, 7)
    cen = rng.randn(npoints, 7)
    s2 = _trial_stats(torch_mod, ctx, v, 7, center=cen)
    assert np.array_equal(s2[..., :4], s[..., :4], equal_nan=True) and np.array_equal(s2[..., 5], s[..., 5])
    for p in range(npoints):
        for c in range(7):
            col = v[p, :, c]
            assert_stats(s[p, c], _col_ref(col), col)
            assert np.array_equal(s2[p, c, 4], _col_ref(col, cen[p, c])[4], equal_nan=True), (p, c)


def test_trial_stats_ties_and_non_finite_columns(torch_mod, ctx):
    """Exact ties spread over slices (the first trial wins, as with nanargmax); +inf among finite values (mean inf,
    std NaN, worst = the first finite value); +inf and -inf together (mean, std, worst NaN, min -inf, max +inf, the
    count exact); a column without a finite value; a NaN centre (worst NaN, the rest unchanged)."""
    P, T = 3, 1000  # 4 slices of 250 per point
    rng = np.random.RandomState(5)
    v = np.zeros((P, T, 6))
    for p in range(P):
        v[p, [310 + p, 620, 905, 999], 0] = [-3.0, 3.0, -3.0, 3.0]  # mean exactly 0: four trials at distance 3
        v[p, :, 1] = rng.randn(T)
        v[p, [0, 17], 1] = np.nan
        v[p, [400 + p, 800], 1] = np.inf
        v[p, :, 2] = rng.randn(T)
        v[p, 100 + p, 2], v[p, 600, 2], v[p, 7, 2] = np.inf, -np.inf, np.nan
        v[p, :, 3] = np.nan
        v[p, :, 4] = rng.randn(T) + 2.0
        v[p, :, 5] = np.nan if p == 1 else 1e300
    s = _trial_stats(torch_mod, ctx, v, 5)
    for p in range(P):
        for c in range(5):
            assert_stats(s[p, c], _col_ref(v[p, :, c]), v[p, :, c])
        assert s[p, 0, 4] == -3.0 and s[p, 1, 4] == v[p, 1, 1] and np.isnan(s[p, 2, 4])
        assert np.isinf(s[p, 1, 0]) and np.isnan(s[p, 1, 1]) and s[p, 1, 5] == T - 2
        assert np.isnan(s[p, 2, :2]).all() and s[p, 2, 2] == -np.inf and s[p, 2, 3] == np.inf and s[p, 2, 5] == T - 1
        assert np.isnan(s[p, 3, :5]).all() and s[p, 3, 5] == 0
    cen = np.zeros((P, 5))
    cen[:, 4] = np.nan
    s2 = _trial_stats(torch_mod, ctx, v, 5, center=cen)
    assert np.array_equal(s2[..., [0, 1, 2, 3, 5]], s[..., [0, 1, 2, 3, 5]], equal_nan=True)
    for p in range(P):
        for c in range(5):
            assert np.array_equal(s2[p, c, 4], _col_ref(v[p, :, c], cen[p, c])[4], equal_nan=True), (p, c)
        assert np.isnan(s2[p, 4, 4]) and s2[p, 0, 4] == -3.0
