"""CPU-side checks: the C-ABI library builds, loads and exports every symbol include/dfk_b200.h declares;
host-side logic of the fitter API; slab sharding over a 2-rank gloo group.  No compute call is made here
(the library has no CPU path): anything numerical on the product side is covered by `-m gpu` tests."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from deepfmkit_b200 import _build, _lib
    _build.build_library()
    return _lib.load_library()


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "dfk_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(dfk_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_exported_and_bound(lib):
    from deepfmkit_b200 import _lib
    names = declared_symbols()
    assert len(names) >= 20
    for name in names:
        assert hasattr(lib, name), f"{name} declared in the header but not exported"
        assert name in _lib.SYMBOLS, f"{name} has no ctypes prototype"
    assert sorted(_lib.SYMBOLS) == names


def test_struct_layouts_match_header(lib):
    from deepfmkit_b200 import _lib
    assert ctypes.sizeof(_lib.LmOpts) == 8 + 8 * 8
    assert ctypes.sizeof(_lib.EkfOpts) == 16 * 8
    assert ctypes.sizeof(_lib.LmCounters) == 5 * 8
    o = _lib.default_lm_opts()
    assert (o.max_lma_steps, o.conv_improve, o.conv_param, o.fitok_threshold) == (100, 1e-9, 1e-9, 1e-3)
    assert (o.m_grid_min, o.m_grid_max, o.m_grid_step) == (5.0, 30.0, 0.5)
    assert (o.bessel_amp_threshold, o.sincos_amp_threshold) == (0.05, 0.1)
    e = _lib.default_ekf_opts()
    assert list(e.init) == [1.6, 6.0, 0.0, 0.0] and list(e.p0_diag) == [1.0] * 5
    assert list(e.q_diag) == [1e-8, 1e-8, 1e-6, 1e-6, 1e-8] and np.isnan(e.r_val) and np.isnan(e.init_dc)


def test_no_gpu_means_loud_failure(lib):
    """Without a device the product path raises: there is no CPU fallback to fall into."""
    from deepfmkit_b200 import _lib
    if _lib.device_count() > 0:
        pytest.skip("a GPU is visible")
    with pytest.raises(RuntimeError, match="no CUDA device"):
        _lib.Context(0)
    from deepfmkit_b200 import DeepRawObject, StandardNLSFitter
    raw = DeepRawObject(data=np.ones(8000), f_samp=200e3, f_mod=1000)
    with pytest.raises(RuntimeError):
        StandardNLSFitter({"n": 20}).fit(raw)


def test_product_never_imports_oracle():
    """Only tests/, smoke() and bench.py's CPU legs may touch oracle/: not the package, not the dev tools."""
    for sub in ("deepfmkit_b200", "benchmarks", "include"):
        for dirpath, _, files in os.walk(os.path.join(ROOT, sub)):
            for f in files:
                if f.endswith((".py", ".cu", ".cuh", ".h")):
                    text = open(os.path.join(dirpath, f)).read()
                    assert not re.search(r"^\s*(from|import)\s+oracle", text, flags=re.M), f
                    assert "dfmi_oracle" not in text, f
                    if sub == "deepfmkit_b200":
                        assert "scipy" not in text or f == "dfk_bessel.cuh", f


def test_missing_library_is_a_loud_error(monkeypatch):
    from deepfmkit_b200 import _lib
    monkeypatch.setenv("DFK_LIB_PATH", os.path.join(ROOT, "deepfmkit_b200", "no_such_library.so"))
    monkeypatch.setattr(_lib, "_lib", None)
    with pytest.raises(RuntimeError, match="is missing"):
        _lib.load_library()


def test_demod_plan_selection(lib):
    from deepfmkit_b200 import _lib
    w = lambda fs, fm: 2.0 * np.pi * fm / fs
    assert _lib.demod_path(4000, w(200e3, 1000.0)) == 1
    assert _lib.demod_path(20000, w(1e6, 1000.0)) == 1
    assert _lib.demod_path(200, w(200e3, 1000.0)) == 1
    assert _lib.demod_path(1500, w(30e3, 400.0)) == 1      # 75 samples per period: folds at 150 (two periods)
    assert _lib.demod_path(75, w(30e3, 400.0)) == 0        # a single odd period per buffer cannot fold
    assert _lib.demod_path(3240, w(200e3, 1234.5)) == 0    # non-integer period
    assert _lib.demod_path(4100, w(200e3, 1000.0)) == 0    # buffer is not a whole number of periods


def test_fitter_host_logic():
    import pandas as pd
    from deepfmkit_b200 import BaseFitter, DeepFitFramework, DeepRawObject, StandardNLSFitter, rows_to_frame
    from deepfmkit_b200.fitters import _calculate_fit_params, _record_values
    with pytest.raises(ValueError, match="must include 'n'"):
        StandardNLSFitter({"ndata": 10})
    with pytest.raises(TypeError):
        BaseFitter({"n": 1})  # abstract
    raw = DeepRawObject(data=pd.DataFrame(np.arange(10000.0), columns=["ch0"]), f_samp=200e3, f_mod=1000)
    assert _calculate_fit_params(raw, 20) == (4000, 50.0, 2)
    assert _calculate_fit_params(raw, 100)[2] == 0
    v = _record_values(raw)
    assert v.dtype == np.float64 and v.flags.c_contiguous and v.shape == (10000,)
    rows = np.arange(24.0).reshape(3, 8)
    df = rows_to_frame(rows)
    assert list(df.columns) == ["amp", "m", "phi", "psi", "dc", "ssq", "fitok"]
    assert str(df["fitok"].dtype) == "int64" and all(str(df[c].dtype) == "float64" for c in df.columns[:6])
    dff = DeepFitFramework()
    dff.load_raw_object(raw, "r")
    assert dff.fit_init("r", 20) == (4000, 50.0, 2)
    assert dff.fit("missing") is None and dff.fit("r", method="wdfmi_nls") is None


def test_tunables_snapshot_follows_module_patches(lib):
    import types
    from deepfmkit_b200 import fit as tun
    old = tun.FITOK_THRESHOLD
    try:
        tun.FITOK_THRESHOLD = 5e-4
        assert tun.current_lm_opts().fitok_threshold == 5e-4
    finally:
        tun.FITOK_THRESHOLD = old
    ref_like = types.SimpleNamespace(MAX_LMA_STEPS=7, M_GRID_STEP=0.25)  # a patched reference fit module
    o = tun.current_lm_opts(ref_like)
    assert o.max_lma_steps == 7 and o.m_grid_step == 0.25 and o.fitok_threshold == 1e-3


def test_slab_bounds_cover_and_balance():
    from deepfmkit_b200.sharding import all_slab_bounds, slab_bounds
    for n, w in ((180000, 8), (7, 3), (2, 4), (0, 2), (12800001, 8)):
        b = all_slab_bounds(n, w)
        assert b[0][0] == 0 and b[-1][1] == n
        assert all(b[i][1] == b[i + 1][0] for i in range(w - 1))
        sizes = [hi - lo for lo, hi in b]
        assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        slab_bounds(10, 2, 2)


def test_dev_overrides_are_explicit_and_validated(lib):
    """Tuning overrides exist only through dfk_dev_set (the library never reads the environment); names are bounded,
    the staged-copy geometry is range-checked, and dfk_dev_clear restores the defaults.  Host calls only."""
    assert lib.dfk_dev_set(b"DFK_NO_TILE", 1) == 0
    assert lib.dfk_dev_set(b"X" * 40, 1) != 0 and b"override name" in lib.dfk_last_error()
    assert lib.dfk_dev_set(b"", 1) != 0
    for name, good, bad in ((b"DFK_STAGE_KB", 4096, 16), (b"DFK_STAGE_KB", 65536, 65537 * 2), (b"DFK_STAGERS", 6, 1),
                            (b"DFK_STAGERS", 8, 9)):
        assert lib.dfk_dev_set(name, good) == 0, name
        assert lib.dfk_dev_set(name, bad) != 0, (name, bad)
    assert lib.dfk_dev_set(b"DFK_COPY_THREADS", 0) == 0 and lib.dfk_dev_set(b"DFK_COPY_NT", 1) == 0
    for i in range(40):  # the table of kernel overrides is finite and says so
        rc = lib.dfk_dev_set(f"DFK_TEST_{i}".encode(), i)
        if rc != 0:
            assert b"table full" in lib.dfk_last_error()
            break
    else:
        raise AssertionError("override table never filled")
    lib.dfk_dev_clear()
    assert lib.dfk_dev_set(b"DFK_NO_TILE", 0) == 0
    lib.dfk_dev_clear()


def test_header_is_plain_c(tmp_path):
    """The drop-in boundary is a C ABI: include/dfk_b200.h must compile as C99 with no C++ or CUDA types in it, and
    carry the ABI version the binding expects."""
    from deepfmkit_b200 import _lib
    src = tmp_path / "abi.c"
    src.write_text('#include "dfk_b200.h"\n'
                   f'int main(void) {{ return DFK_ABI_VERSION == {_lib.ABI_VERSION} && DFK_ASD_TRIAL_DOUBLES == '
                   f'{_lib.ASD_TRIAL_DOUBLES} ? 0 : 1; }}\n')
    exe = tmp_path / "abi"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"),
                           str(src), "-o", str(exe)])
    assert subprocess.call([str(exe)]) == 0


_GLOO_WORKER = r"""
import os, sys
sys.path.insert(0, {root!r})
import numpy as np
import torch.distributed as dist
from deepfmkit_b200.sharding import slab_bounds, gather_rows, broadcast_seed
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
nbuf = 11
lo, hi = slab_bounds(nbuf, world, rank)
seed = broadcast_seed([1.0, 6.0, 0.25, -0.5] if rank == 0 else [0, 0, 0, 0])
assert list(seed) == [1.0, 6.0, 0.25, -0.5]
rows = np.zeros((hi - lo, 8))
rows[:, 0] = np.arange(lo, hi)      # stand-in for the per-slab fit: row index ...
rows[:, 1] = seed[1] + rank         # ... and something that depends on the seed and the rank
table = gather_rows(rows, nbuf)
if rank == 0:
    assert table.shape == (nbuf, 8)
    assert np.array_equal(table[:, 0], np.arange(nbuf))
    assert np.array_equal(table[:, 1], np.where(np.arange(nbuf) < 6, 6.0, 7.0))
    print("GLOO_OK")
else:
    assert table is None
dist.destroy_process_group()
"""


def test_sharded_gather_world_size_2_gloo(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_GLOO_WORKER.format(root=ROOT))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", "29611", str(script)]
    env = dict(os.environ, OMP_NUM_THREADS="1")
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=240, env=env)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "GLOO_OK" in out.stdout


_GLOO_EXPERIMENT_WORKER = r"""
import os, sys
sys.path.insert(0, {root!r})
import numpy as np
import torch.distributed as dist
from deepfmkit_b200 import Experiment
from deepfmkit_b200.experiments import RESULT_KEYS
from deepfmkit_b200.sharding import slab_bounds
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
exp = Experiment("gloo")
exp.add_axis("a", np.arange(3.0)); exp.add_axis("b", np.arange(5.0))
exp.add_analysis("nls", "nls"); exp.add_analysis("ekf", "ekf", result_cols=["m", "nope"])
grid_shape, ntr, npoints = (3, 5), 4, 15
lo, hi = slab_bounds(npoints, world, rank)
# stand-in for the per-rank simulate + fit + statistics: every entry encodes (point, trial, column, statistic)
pts = np.arange(lo, hi)
local = {{}}
for name, off in (("nls", 0.0), ("ekf", 0.5)):
    st = off + pts[:, None, None] * 100 + np.arange(len(RESULT_KEYS))[None, :, None] * 10 + np.arange(6)[None, None, :]
    v = off + pts[:, None, None] * 100 + np.arange(ntr)[None, :, None] * 10 + np.arange(len(RESULT_KEYS))[None, None, :]
    local[name] = (st.astype(float), v.astype(float))
parts = [None] * world
dist.all_gather_object(parts, local)
res = exp._assemble_results(parts, grid_shape, ntr)
c = RESULT_KEYS.index("m")
point = np.arange(npoints).reshape(grid_shape)
assert np.array_equal(res["nls"]["m"]["mean"], point * 100 + c * 10 + 0)
assert np.array_equal(res["nls"]["m"]["worst"], point * 100 + c * 10 + 4)
assert np.array_equal(res["ekf"]["m"]["all_trials"], 0.5 + point[..., None] * 100 + np.arange(ntr) * 10 + c)
assert np.all(np.isnan(res["ekf"]["nope"]["mean"])) and res["ekf"]["nope"]["all_trials"].shape == (3, 5, 4)
assert sorted(res["nls"]) == sorted(RESULT_KEYS) and sorted(res["ekf"]) == ["m", "nope"]
if rank == 0:
    print("GLOO_EXPERIMENT_OK")
dist.destroy_process_group()
"""


def test_experiment_assembly_world_size_2_gloo(tmp_path):
    """Experiment.run(group=...): grid points in contiguous ranges per rank, per-rank tables gathered as objects and
    assembled in rank order -- the host side of it, with stand-in tables, over a 2-rank gloo group."""
    script = tmp_path / "worker_exp.py"
    script.write_text(_GLOO_EXPERIMENT_WORKER.format(root=ROOT))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", "29613", str(script)]
    env = dict(os.environ, OMP_NUM_THREADS="1")
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=240, env=env)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "GLOO_EXPERIMENT_OK" in out.stdout


def test_bench_reference_arm_contract():
    """bench.py's CPU arm: the port's pool schedule agrees with the sequential oracle, and the arm that times the
    reference itself (baseline/_ref, when installed) returns the same rows as the port on the same sample."""
    sys.path.insert(0, ROOT)
    import bench
    from oracle import dfmi_oracle as orc
    x = orc.snr_signal(bench.M_TRUE, bench.F_SAMP, bench.F_MOD, 6 * bench.R / bench.F_SAMP, bench.SNR_DB, seed=1)
    assert len(x) == 6 * bench.R
    rows = orc.nls_fit_pool(x, bench.F_SAMP, bench.F_MOD, bench.N_CYCLES, bench.NDATA, n_procs=2)
    ref = orc.nls_fit(x, bench.F_SAMP, bench.F_MOD, bench.N_CYCLES, bench.NDATA, schedule="seeded", n_chunks=2)
    assert np.array_equal(rows, ref)
    assert bench.NBUF == 180000 and bench.R == 20000
    arm = bench.cpu_arm()
    assert arm.kind in ("reference", "port")
    if arm.kind == "reference":
        df = arm.rfitters.StandardNLSFitter({"n": bench.N_CYCLES, "ndata": bench.NDATA}).fit(
            arm._raw(x, bench.F_SAMP, bench.F_MOD), parallel=True, n_cores=2)
        got = df[["amp", "m", "phi", "psi", "dc", "ssq", "fitok"]].to_numpy(dtype=float)
        assert np.array_equal(got, ref)
    assert arm.nls_pool(x, bench.F_SAMP, bench.F_MOD, bench.N_CYCLES, bench.NDATA, 2) > 0


def test_reference_facade_dispatches_to_b200_fitters(lib, tmp_path):
    """INTEGRATION.md section 1 on the real thing: the unmodified reference (a DeepFMKit checkout named by
    DFK_REFERENCE; it is not part of this repository) with its two fitter classes swapped for ours.  The facade reaches
    our C ABI: without a GPU, that shows as the library's loud 'no CUDA device' error; the frame-level parity of the
    same call is what `-m gpu` tests check against fixtures minted from this very reference."""
    ref = os.environ.get("DFK_REFERENCE")
    if not ref or not os.path.isdir(ref):
        pytest.skip("set DFK_REFERENCE to a DeepFMKit checkout to run this test")
    from unittest.mock import MagicMock
    saved = {k: sys.modules.get(k) for k in ("matplotlib", "matplotlib.pyplot", "matplotlib.colors",
                                             "matplotlib.dates", "matplotlib.cm", "pyplnoise")}
    for name in saved:
        sys.modules[name] = MagicMock()
    os.symlink(ref, tmp_path / "DeepFMKit")
    sys.path.insert(0, str(tmp_path))
    old_dont_write = sys.dont_write_bytecode
    sys.dont_write_bytecode = True
    try:
        import DeepFMKit.core as core
        import deepfmkit_b200 as b2
        from deepfmkit_b200 import _lib
        core.StandardNLSFitter, core.EKFFitter = b2.StandardNLSFitter, b2.EKFFitter
        dff = core.DeepFitFramework()
        laser = core.LaserConfig(label="l")
        laser.f_mod = 1000
        ifo = core.InterferometerConfig(label="i")
        core.set_laser_df_for_effect(laser, ifo, 6.0)
        sim = core.DFMIObject(label="ch", laser_config=laser, ifo_config=ifo, f_samp=200e3)
        dff.load_sim(sim)
        dff.simulate(main_label="ch", n_seconds=0.1, mode="snr", snr_db=40)
        if _lib.device_count() == 0:
            for method in ("nls", "ekf"):
                with pytest.raises(RuntimeError, match="no CUDA device"):
                    dff.fit("ch", method=method, verbose=False)
        else:
            fobj = dff.fit("ch", parallel=True)
            assert list(dff.fits_df["ch_nls"].columns) == ["amp", "m", "phi", "psi", "dc", "ssq", "fitok", "tau"]
            assert fobj.nbuf == 5 and abs(fobj.m.mean() - 6.0) < 1e-2
    finally:
        sys.dont_write_bytecode = old_dont_write
        sys.path.remove(str(tmp_path))
        for k in list(sys.modules):
            if k == "DeepFMKit" or k.startswith("DeepFMKit."):
                del sys.modules[k]
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def test_bench_reference_arm_emits_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside ours): one JSON line on stdout with the
    contract's keys, nothing else on stdout."""
    import json
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert key in d, key
    assert d["impl"] == "reference" and d["dtype"] == "f64" and d["vs_baseline"] is None and d["value"] > 0
    assert d["config"]["workload"].startswith("cfg2") and "model" not in d["config"]
    assert set(d["cpu_baseline"]) >= {"value", "unit", "cores", "kind", "sample"} and d["cpu_baseline"]["kind"] in ("reference", "port")
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
