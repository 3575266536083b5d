"""Randomised geometry sweep of the TMA-fed demodulation kernels against a plain numpy lock-in.

The ring protocols of the fold / long-fold / tile / single-period kernels (mbarrier phases, the issued-chunk counter, per-warp
ownership of stages) fail as hangs or as stale data, and which warp meets which stage depends on the number of
buffers, the ring depth and the group size -- so the sweep draws those at random (fixed seed) and repeats every
launch, comparing with an independent CPU result.  compute-sanitizer is not available on this pool; this is the
substitute.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def numpy_lockin(x, R, nh, w0):
    nbuf = len(x) // R
    t = np.arange(R)
    k = np.arange(1, nh + 1)[:, None]
    ang = (k * w0) * t[None, :]  # the reference's fl(fl(k*w0)*t)
    xb = x[: nbuf * R].reshape(nbuf, R)
    q = xb @ np.cos(ang).T / R
    i = xb @ np.sin(ang).T / R
    return np.concatenate([q, i], axis=1), xb.mean(axis=1)


def test_random_geometries(monkeypatch):
    import torch
    from deepfmkit_b200 import _lib
    ctx = _lib.Context(0)
    lib = _lib.load_library()
    ctx.use_torch_stream()  # the NaN pre-fills below are torch kernels: same stream, so they are ordered before ours
    rng = np.random.RandomState(31337)
    worst = 0.0
    cases = 0
    for trial in range(84):
        kind = trial % 6
        if kind == 0:    # single-period kernel: P % 4 == 0, n = 1
            P, n = 4 * rng.randint(1, 65), 1
        elif kind == 1:  # tile kernel, grouped buffers
            P, n = 2 * rng.randint(1, 129), rng.randint(1, 5)
        elif kind == 2:  # tile kernel, one buffer per group
            P, n = 2 * rng.randint(20, 129), rng.randint(8, 40)
        elif kind == 3:  # fold kernel
            P, n = 2 * rng.randint(129, 1025), rng.randint(1, 9)
        elif kind == 4:  # odd period folded over two periods
            P, n = 2 * rng.randint(3, 300) + 1, 2 * rng.randint(1, 8)
        else:            # fold lengths beyond 2048: the column-chunked kernel (ragged last chunk included)
            P, n = 2 * rng.randint(1025, 6000), rng.randint(1, 7)
        nh = int(rng.randint(1, 21))
        nbuf = int(rng.choice([1, 2, 7, 8, 9, 63, 148, 149, 300, 1185, 2371, 5000]))
        if P * n * nbuf > 40_000_000:
            nbuf = max(1, 40_000_000 // (P * n))
        R = P * n
        w0 = 2.0 * np.pi * 1000.0 / (1000.0 * P)
        lib.dfk_dev_clear()
        if rng.rand() < 0.3:
            lib.dfk_dev_set(b"DFK_TILE_NSTAGES", int(rng.randint(2, 6)))
        if kind == 0 and rng.rand() < 0.6:  # ring depth of the single-period kernel
            lib.dfk_dev_set(b"DFK_PERIOD_NSTAGES", int(rng.randint(2, 13)))
        t = np.arange(nbuf * R)
        x = 1.0 + np.cos(0.3 + 4.0 * np.cos(2 * np.pi * t / P + 0.1)) + 0.05 * rng.randn(nbuf * R)
        ref_qi, ref_dc = numpy_lockin(x, R, nh, w0)
        xd = torch.from_numpy(x).cuda()
        scale = np.maximum(np.abs(ref_qi).max(axis=1, keepdims=True), 1e-3)
        for rep in range(2):
            qi = torch.full((nbuf, 2 * nh), float("nan"), dtype=torch.float64, device="cuda")
            dc = torch.full((nbuf,), float("nan"), dtype=torch.float64, device="cuda")
            ctx.demod(xd.data_ptr(), nbuf, R, nh, w0, qi.data_ptr(), dc.data_ptr())
            ctx.synchronize()
            err = float(np.max(np.abs(qi.cpu().numpy() - ref_qi) / scale))
            assert err <= 1e-12, (trial, kind, P, n, nh, nbuf, rep, err)
            assert np.max(np.abs(dc.cpu().numpy() - ref_dc)) <= 1e-13, (trial, kind, P, n, nh, nbuf, rep)
            worst = max(worst, err)
        cases += 1
    lib.dfk_dev_clear()
    ctx.close()
    assert cases == 84 and worst <= 1e-12


@pytest.mark.parametrize("pinned", [False, True])
def test_host_entry_boundaries(pinned):
    """Record lengths straddling the host pipeline's boundaries (64 MiB staging pieces, 128 MiB device slabs), from
    pageable and from pinned memory: the rows must equal those of the device-resident call, bit for bit."""
    import torch
    from deepfmkit_b200 import _lib
    ctx = _lib.Context(0)
    R, nh = 1000, 6
    w0 = 2.0 * np.pi / 100.0
    stage, slab = (64 << 20) // (R * 8), (128 << 20) // (R * 8)
    for nbuf in (1, stage - 1, stage, stage + 1, slab - 1, slab, slab + 1, 2 * slab + 3):
        xd = torch.empty(nbuf * R + 7, dtype=torch.float64, device="cuda")  # + a ragged tail the entry must ignore
        ctx.synth_snr_dev(xd.data_ptr(), nbuf * R + 7, 1, 100e3, 1000.0, 6.0, snr_db=40.0, seed=nbuf)
        ref = torch.empty((nbuf, 8), dtype=torch.float64, device="cuda")
        ctx.nls_fit_dev(xd.data_ptr(), nbuf, R, nh, w0, [1.6, 6.0, 0.0, 0.0], True, None, ref.data_ptr())
        ctx.synchronize()
        if pinned:
            xh = torch.empty(nbuf * R + 7, dtype=torch.float64, pin_memory=True)
            xh.copy_(xd)
            x = xh.numpy()
        else:
            x = xd.cpu().numpy()
        rows = ctx.nls_fit_host(x, R, nh, w0, [1.6, 6.0, 0.0, 0.0], seeded=True)
        assert rows.shape == (nbuf, 8)
        r = ref.cpu().numpy()
        # slabs are fitted separately, so the lanes-per-fit choice (hence the summation order) can differ from the
        # one-launch device call: equality to rounding, not to the bit
        assert np.array_equal(rows[:, 6], r[:, 6]), (nbuf, pinned)
        assert np.max(np.abs(rows[:, :6] - r[:, :6])) < 1e-9, (nbuf, pinned, np.max(np.abs(rows[:, :6] - r[:, :6])))
        assert np.array_equal(rows[:, 4], r[:, 4]), (nbuf, pinned)  # dc comes from the demodulation alone: bit equal
    ctx.close()
