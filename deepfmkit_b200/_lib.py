"""ctypes binding of libdfk_b200.so (the C ABI in include/dfk_b200.h).

There is no CPU implementation behind this module: if the library is missing or no B200 is
visible, every call raises.  PyTorch is used by callers only for device memory and streams;
the library itself takes raw device/host pointers.
"""
from __future__ import annotations

import ctypes
import os
import threading

import numpy as np

from ._build import LIB_PATH

ROW_STRIDE = 8
COV_STRIDE = 8          # [C_aa, C_am, C_aphi, C_mm, C_mphi, C_phiphi, C_psipsi, s^2] per result row
MAX_HARMONICS = 64
ABI_VERSION = 6
PROFILE_KINDS = 4
ASD_TRIAL_DOUBLES = 37
TRIAL_STATS_DOUBLES = 6
SCHED_INDEPENDENT = 0   # every buffer a cold start from init
SCHED_EACH = -1         # every buffer its own chunk, seeded from buffer 0 (pool schedule at n_cores >= nbuf - 1)
ROW_COLUMNS = ("amp", "m", "phi", "psi", "dc", "ssq", "fitok")
STAB_PHASE, STAB_FREQ = 0, 1                   # DFK_STAB_PHASE, DFK_STAB_FREQ
STAB_KINDS = ("oadev", "mdev", "tdev", "ohdev")  # the slot order of dfk_stability_dev's outputs
STAB_BITS = {"oadev": 1, "mdev": 2, "tdev": 4, "ohdev": 8}

c_double_p = ctypes.POINTER(ctypes.c_double)


class LmOpts(ctypes.Structure):
    _fields_ = [("max_lma_steps", ctypes.c_int32), ("lanes_per_fit", ctypes.c_int32),
                ("conv_improve", ctypes.c_double), ("conv_param", ctypes.c_double),
                ("fitok_threshold", ctypes.c_double), ("m_grid_min", ctypes.c_double),
                ("m_grid_max", ctypes.c_double), ("m_grid_step", ctypes.c_double),
                ("bessel_amp_threshold", ctypes.c_double), ("sincos_amp_threshold", ctypes.c_double)]


class EkfOpts(ctypes.Structure):
    _fields_ = [("init", ctypes.c_double * 4), ("p0_diag", ctypes.c_double * 5),
                ("q_diag", ctypes.c_double * 5), ("r_val", ctypes.c_double), ("init_dc", ctypes.c_double)]


class RawHeader(ctypes.Structure):
    _fields_ = [("channels", ctypes.c_int32), ("pad_", ctypes.c_int32), ("t0", ctypes.c_int64),
                ("f_samp", ctypes.c_double), ("f_mod", ctypes.c_double), ("data_offset", ctypes.c_int64)]


RAW_DTYPES = {"int16": 0, "int32": 1, "float32": 2, "float64": 3}


class LpsdOpts(ctypes.Structure):
    _fields_ = [("olap", ctypes.c_double), ("bmin", ctypes.c_double), ("lmin", ctypes.c_int64),
                ("jdes", ctypes.c_int32), ("kdes", ctypes.c_int32), ("order", ctypes.c_int32),
                ("window", ctypes.c_int32), ("psll", ctypes.c_double)]


class LmCounters(ctypes.Structure):
    _fields_ = [("n_state", ctypes.c_uint64), ("n_ssq", ctypes.c_uint64), ("n_solve", ctypes.c_uint64),
                ("n_grid", ctypes.c_uint64), ("n_bessel_steps", ctypes.c_uint64)]


# every symbol include/dfk_b200.h declares: name -> (restype, argtypes)
_vp = ctypes.c_void_p
_i64 = ctypes.c_int64
_i32 = ctypes.c_int32
_d = ctypes.c_double
SYMBOLS = {
    "dfk_abi_version": (ctypes.c_int, []),
    "dfk_last_error": (ctypes.c_char_p, []),
    "dfk_device_count": (ctypes.c_int, []),
    "dfk_create": (ctypes.c_int, [ctypes.c_int, ctypes.POINTER(_vp)]),
    "dfk_destroy": (ctypes.c_int, [_vp]),
    "dfk_set_stream": (ctypes.c_int, [_vp, _vp]),
    "dfk_use_legacy_default_stream": (ctypes.c_int, [_vp, ctypes.c_int]),
    "dfk_synchronize": (ctypes.c_int, [_vp]),
    "dfk_default_lm_opts": (None, [ctypes.POINTER(LmOpts)]),
    "dfk_default_ekf_opts": (None, [ctypes.POINTER(EkfOpts)]),
    "dfk_demod": (ctypes.c_int, [_vp, _vp, _i64, _i64, _i32, _d, _vp, _vp]),
    "dfk_lm_fit": (ctypes.c_int, [_vp, _vp, _i64, _i32, _vp, _i64, _vp, ctypes.POINTER(LmOpts), _vp]),
    "dfk_lm_cov": (ctypes.c_int, [_vp, _vp, _i64, _i32, _vp, _vp]),
    "dfk_nls_fit_dev": (ctypes.c_int, [_vp, _vp, _i64, _i64, _i32, _d, c_double_p, _i32, ctypes.POINTER(LmOpts), _vp]),
    "dfk_nls_fit_cov_dev": (ctypes.c_int, [_vp, _vp, _i64, _i64, _i32, _d, c_double_p, _i32, ctypes.POINTER(LmOpts), _vp,
                                           _vp]),
    "dfk_nls_fit_seeded_dev": (ctypes.c_int, [_vp, _vp, _i64, _i64, _i32, _d, c_double_p, _i32, ctypes.POINTER(LmOpts), _vp]),
    "dfk_nls_fit_batch_dev": (ctypes.c_int, [_vp, _vp, _i64, _i64, _i64, _i64, _i32, _d, c_double_p, _vp, _i64, _i32,
                                             ctypes.POINTER(LmOpts), _vp]),
    "dfk_nls_fit_batch_cov_dev": (ctypes.c_int, [_vp, _vp, _i64, _i64, _i64, _i64, _i32, _d, c_double_p, _vp, _i64, _i32,
                                                 ctypes.POINTER(LmOpts), _vp, _vp]),
    "dfk_demod_tm_dev": (ctypes.c_int, [_vp, _vp, _i64, _i64, _i64, _i32, _d, _vp, _vp]),
    "dfk_nls_fit_batch_tm_dev": (ctypes.c_int, [_vp, _vp, _i64, _i64, _i64, _i32, _d, c_double_p, _vp, _i64, _i32,
                                                ctypes.POINTER(LmOpts), _vp]),
    "dfk_nls_fit_batch_tm_cov_dev": (ctypes.c_int, [_vp, _vp, _i64, _i64, _i64, _i32, _d, c_double_p, _vp, _i64, _i32,
                                                    ctypes.POINTER(LmOpts), _vp, _vp]),
    "dfk_ekf_dev": (ctypes.c_int, [_vp, _vp, _i64, _i64, _i64, _i64, _i64, _d, _d, ctypes.POINTER(EkfOpts), _vp]),
    "dfk_ekf_stream_dev": (ctypes.c_int, [_vp, _vp, _i64, _i64, _i64, _i64, _i64, _d, _d, ctypes.POINTER(EkfOpts), _i64,
                                          _vp, _vp]),
    "dfk_ekf_smooth_dev": (ctypes.c_int, [_vp, _vp, _i64, _i64, _i64, _i64, _i64, _d, _d, ctypes.POINTER(EkfOpts), _i64,
                                          _vp, _i64, _vp, _vp, _vp, _vp]),
    "dfk_ekf_em_dev": (ctypes.c_int, [_vp, _vp, _i64, _i64, _i64, _i64, _i64, _d, _d, ctypes.POINTER(EkfOpts), _vp,
                                      ctypes.c_uint32, _i32, _d, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "dfk_synth_snr_slab_dev": (ctypes.c_int, [_vp, _vp, _i64, _i64, _i64, _i64, _d, _d, _d, _d, _d, _d, _d, _d, _d,
                                              ctypes.c_uint64]),
    "dfk_synth_snr_dev": (ctypes.c_int, [_vp, _vp, _i64, _i64, _d, _d, _d, _d, _d, _d, _d, _d, _d, ctypes.c_uint64]),
    "dfk_sweep_demod_dev": (ctypes.c_int, [_vp, _i64, _i64, _i64, _i32, _d, _d, _d, _d, _d, _d, _d, _d, ctypes.c_uint64, _vp, _vp]),
    "dfk_nls_sweep_dev": (ctypes.c_int, [_vp, c_double_p, _i32, _i64, _i64, _i64, _i64, _i32, _d, _d, _d, _d, _d, _d, _d,
                                         ctypes.c_uint64, _d, _d, ctypes.POINTER(LmOpts), _vp]),
    "dfk_nls_sweep_cov_dev": (ctypes.c_int, [_vp, c_double_p, _i32, _i64, _i64, _i64, _i64, _i32, _d, _d, _d, _d, _d, _d,
                                             _d, ctypes.c_uint64, _d, _d, ctypes.POINTER(LmOpts), _vp, _vp]),
    "dfk_nls_fit_host": (ctypes.c_int, [_vp, _vp, _i64, _i64, _i32, _d, c_double_p, _i32, ctypes.POINTER(LmOpts), _vp]),
    "dfk_nls_fit_cov_host": (ctypes.c_int, [_vp, _vp, _i64, _i64, _i32, _d, c_double_p, _i32, ctypes.POINTER(LmOpts), _vp,
                                            _vp]),
    "dfk_nls_fit_seeded_host": (ctypes.c_int, [_vp, _vp, _i64, _i64, _i32, _d, c_double_p, _i32, ctypes.POINTER(LmOpts), _vp]),
    "dfk_ekf_host": (ctypes.c_int, [_vp, _vp, _i64, _i64, _i64, _d, _d, ctypes.POINTER(EkfOpts), _vp]),
    "dfk_set_host_slab_bytes": (ctypes.c_int, [_vp, _i64]),
    "dfk_raw_parse_header": (ctypes.c_int, [ctypes.c_char_p, ctypes.POINTER(RawHeader)]),
    "dfk_text_load_file": (ctypes.c_int, [_vp, ctypes.c_char_p, _i64, ctypes.POINTER(_i64), ctypes.POINTER(_i64)]),
    "dfk_text_load_host": (ctypes.c_int, [_vp, _vp, _i64, ctypes.POINTER(_i64)]),
    "dfk_text_parse_dev": (ctypes.c_int, [_vp, _i32, _vp, _vp, _i64, ctypes.POINTER(_i64)]),
    "dfk_text_release": (ctypes.c_int, [_vp]),
    "dfk_widen_dev": (ctypes.c_int, [_vp, _vp, _i32, _i64, _i64, _i32, _d, _d, _vp, _i64]),
    "dfk_ingest_binary_host": (ctypes.c_int, [_vp, _vp, _i32, _i64, _i64, _i32, _d, _d, _vp, _i64]),
    "dfk_ingest_binary_file": (ctypes.c_int, [_vp, ctypes.c_char_p, _i64, _i32, _i64, _i64, _i32, _d, _d, _vp, _i64]),
    "dfk_synth_asd_dev": (ctypes.c_int, [_vp, _vp, _i64, _i64, _d, _vp, _i64, _vp, _i64, _vp]),
    "dfk_synth_asd_noise_dev": (ctypes.c_int, [_vp, _vp, _i64, _i64, _d, _vp, _i64, _vp, _i64, _vp, _i64, _vp]),
    "dfk_trial_stats_dev": (ctypes.c_int, [_vp, _vp, _i64, _i64, _i32, _i64, _vp, _vp]),
    "dfk_downsample_dev": (ctypes.c_int, [_vp, _vp, _i64, _i64, _vp]),
    "dfk_downsample_host": (ctypes.c_int, [_vp, _vp, _i64, _i64, _vp]),
    "dfk_default_lpsd_opts": (None, [ctypes.POINTER(LpsdOpts)]),
    "dfk_lpsd_plan": (ctypes.c_int, [_i64, _d, ctypes.POINTER(LpsdOpts), _i32, ctypes.POINTER(_i32), _vp, _vp, _vp, _vp,
                                     _vp]),
    "dfk_lpsd_dev": (ctypes.c_int, [_vp, _vp, _i64, _i64, _i64, _i64, _d, ctypes.POINTER(LpsdOpts), _i32,
                                    ctypes.POINTER(_i32), _vp, _vp, _vp, _vp, _vp]),
    "dfk_lcsd_dev": (ctypes.c_int, [_vp, _vp, _i64, _i64, _vp, _i64, _i64, _i64, _i64, _d, ctypes.POINTER(LpsdOpts),
                                    _i32, ctypes.POINTER(_i32), _vp, _vp, _vp, _vp, _vp, _vp]),
    "dfk_lcsd_cond_dev": (ctypes.c_int, [_vp, _vp, _i64, _i64, _vp, _i64, _i64, _i64, _i64, _d,
                                         ctypes.POINTER(LpsdOpts), _i32, ctypes.POINTER(_i32), _vp, _vp, _vp, _vp, _vp,
                                         _vp, _vp, _vp, _vp]),
    "dfk_wiener_dev": (ctypes.c_int, [_vp, _vp, _i64, _i64, _vp, _i64, _i64, _i64, _i64, _i64, _i64, _d, _vp, _i64, _vp,
                                      _vp, _vp, ctypes.POINTER(_i32)]),
    "dfk_stability_dev": (ctypes.c_int, [_vp, _vp, _i64, _i64, _i64, _i64, _d, _i32, _i32, _vp, _i32, _vp, _vp]),
    "dfk_lm_counters_read": (ctypes.c_int, [_vp, ctypes.POINTER(LmCounters), _i32]),
    "dfk_profile_enable": (ctypes.c_int, [_vp, _i32]),
    "dfk_profile_read": (ctypes.c_int, [_vp, c_double_p, ctypes.POINTER(_i64), _i32]),
    "dfk_probe_fp64": (ctypes.c_int, [_vp, c_double_p]),
    "dfk_dev_set": (ctypes.c_int, [ctypes.c_char_p, _i32]),
    "dfk_dev_clear": (None, []),
    "dfk_launch_count": (_i64, [_vp]),
    "dfk_demod_path": (ctypes.c_int, [_i64, _d]),
    "dfk_bessel_dev": (ctypes.c_int, [_vp, _vp, _i64, _i32, _vp]),
}

_lib = None
_lib_lock = threading.Lock()


def load_library():
    """dlopen the in-tree library and type every entry point. Raises if it has not been built."""
    global _lib
    with _lib_lock:
        if _lib is not None:
            return _lib
        path = os.environ.get("DFK_LIB_PATH", LIB_PATH)  # development: A/B two builds of the library
        if not os.path.exists(path):
            raise RuntimeError(
                f"{path} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(deepfmkit_b200 has no CPU fallback)")
        lib = ctypes.CDLL(path)
        for name, (restype, argtypes) in SYMBOLS.items():
            fn = getattr(lib, name)
            fn.restype = restype
            fn.argtypes = argtypes
        if lib.dfk_abi_version() != ABI_VERSION:
            raise RuntimeError("libdfk_b200.so ABI version mismatch")
        _lib = lib
        return lib


def schedule_code(seeded) -> int:
    """The C ABI's `seeded` argument: False/0 -> independent starts, True -> every buffer seeded from buffer 0
    (DFK_SCHED_EACH), an int k >= 1 -> the reference's k-chunk chain schedule (k = 1: the sequential chain)."""
    if seeded is True:
        return SCHED_EACH
    if seeded is False or seeded is None:
        return SCHED_INDEPENDENT
    k = int(seeded)
    if k < -1:
        raise ValueError("schedule must be False, True, -1 or a chunk count >= 1")
    return k


def _check(lib, rc):
    if rc != 0:
        raise RuntimeError(f"dfk_b200 error {rc}: {lib.dfk_last_error().decode(errors='replace')}")


def default_lm_opts() -> LmOpts:
    o = LmOpts()
    load_library().dfk_default_lm_opts(ctypes.byref(o))
    return o


def default_ekf_opts() -> EkfOpts:
    o = EkfOpts()
    load_library().dfk_default_ekf_opts(ctypes.byref(o))
    return o


def default_lpsd_opts() -> LpsdOpts:
    o = LpsdOpts()
    load_library().dfk_default_lpsd_opts(ctypes.byref(o))
    return o


def raw_parse_header(path) -> dict:
    """Header of a DFMSWPM raw_data file (host only): channels, t0, f_samp, f_mod, data_offset."""
    lib = load_library()
    h = RawHeader()
    _check(lib, lib.dfk_raw_parse_header(os.fsencode(path), ctypes.byref(h)))
    return {"channels": int(h.channels), "t0": int(h.t0), "f_samp": float(h.f_samp), "f_mod": float(h.f_mod),
            "data_offset": int(h.data_offset)}


def lpsd_plan(N, fs, opts=None) -> dict:
    """Frequency plan of the log-frequency estimate (host only, no GPU needed): f, r, m, L, K arrays."""
    lib = load_library()
    opts = opts if opts is not None else default_lpsd_opts()
    nf = _i32()
    _check(lib, lib.dfk_lpsd_plan(int(N), float(fs), ctypes.byref(opts), 0, ctypes.byref(nf), None, None, None, None, None))
    n = int(nf.value)
    f, r, m = np.empty(n), np.empty(n), np.empty(n)
    L, K = np.empty(n, dtype=np.int64), np.empty(n, dtype=np.int64)
    _check(lib, lib.dfk_lpsd_plan(int(N), float(fs), ctypes.byref(opts), n, ctypes.byref(nf), f.ctypes.data, r.ctypes.data,
                                  m.ctypes.data, L.ctypes.data, K.ctypes.data))
    return {"f": f, "r": r, "m": m, "L": L, "K": K}


def _host_array(a):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a, a.ctypes.data


class Context:
    """One dfk_ctx: a device, its streams and scratch. Not shared between threads."""

    def __init__(self, device: int = 0, own_stream: bool = False):
        """own_stream=False (default): device-pointer calls are issued on the legacy default stream, the one torch
        uses unless told otherwise, so they are ordered with the torch kernels that produce their inputs.
        own_stream=True: on the context's private non-blocking stream -- the caller orders things itself."""
        self.lib = load_library()
        self._h = _vp()
        _check(self.lib, self.lib.dfk_create(int(device), ctypes.byref(self._h)))
        self.device = int(device)
        self._own_default = bool(own_stream)
        self.use_default_stream()

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self.lib.dfk_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # ---- streams ----------------------------------------------------------------------------------
    def use_torch_stream(self, stream=None):
        """Issue device-pointer calls on a torch stream (default: torch's current stream)."""
        import torch
        stream = stream if stream is not None else torch.cuda.current_stream(self.device)
        handle = int(stream.cuda_stream)
        if handle == 0:
            _check(self.lib, self.lib.dfk_use_legacy_default_stream(self._h, 1))
        else:
            _check(self.lib, self.lib.dfk_set_stream(self._h, _vp(handle)))

    def use_own_stream(self):
        _check(self.lib, self.lib.dfk_set_stream(self._h, None))

    def use_default_stream(self):
        """Back to the stream this context was created with (see __init__)."""
        if self._own_default:
            self.use_own_stream()
        else:
            _check(self.lib, self.lib.dfk_use_legacy_default_stream(self._h, 1))

    def synchronize(self):
        _check(self.lib, self.lib.dfk_synchronize(self._h))

    # ---- device-pointer calls (pointers are ints, e.g. tensor.data_ptr()) -----------------------------
    def demod(self, x_ptr, nbuf, R, N, w0, qi_ptr, dc_ptr):
        _check(self.lib, self.lib.dfk_demod(self._h, x_ptr, nbuf, R, N, w0, qi_ptr, dc_ptr))

    def lm_fit(self, qi_ptr, nbuf, N, guess_ptr, guess_stride, dc_ptr, opts, rows_ptr):
        _check(self.lib, self.lib.dfk_lm_fit(self._h, qi_ptr, nbuf, N, guess_ptr, guess_stride, dc_ptr,
                                             ctypes.byref(opts) if opts is not None else None, rows_ptr))

    def lm_cov(self, qi_ptr, nbuf, N, rows_ptr, cov_ptr):
        """Covariance rows [nbuf, COV_STRIDE] of fitted rows on their harmonic vectors (dfk_lm_cov)."""
        _check(self.lib, self.lib.dfk_lm_cov(self._h, qi_ptr, int(nbuf), int(N), rows_ptr, cov_ptr))

    # The record calls take an optional cov_ptr (device, [units, COV_STRIDE]): given, they route to the _cov entry,
    # which also writes every buffer's parameter covariance there.
    def nls_fit_dev(self, x_ptr, nbuf, R, N, w0, init, seeded, opts, rows_ptr, cov_ptr=None):
        init_arr = (ctypes.c_double * 4)(*[float(v) for v in init])
        args = (self._h, x_ptr, nbuf, R, N, w0, init_arr, schedule_code(seeded),
                ctypes.byref(opts) if opts is not None else None, rows_ptr)
        if cov_ptr is None:
            _check(self.lib, self.lib.dfk_nls_fit_dev(*args))
        else:
            _check(self.lib, self.lib.dfk_nls_fit_cov_dev(*args, cov_ptr))

    def nls_fit_seeded_dev(self, x_ptr, nbuf, R, N, w0, seed, opts, rows_ptr, chunks=1):
        seed_arr = (ctypes.c_double * 4)(*[float(v) for v in seed])
        _check(self.lib, self.lib.dfk_nls_fit_seeded_dev(self._h, x_ptr, nbuf, R, N, w0, seed_arr, int(chunks),
                                                         ctypes.byref(opts) if opts is not None else None, rows_ptr))

    def nls_fit_batch_dev(self, x_ptr, C, bufs_per_channel, ld_c, R, N, w0, init, init_dev_ptr, init_stride, seeded,
                          opts, rows_ptr, cov_ptr=None):
        init_arr = (ctypes.c_double * 4)(*[float(v) for v in init]) if init is not None else None
        args = (self._h, x_ptr, C, bufs_per_channel, ld_c, R, N, w0, init_arr, init_dev_ptr, init_stride,
                schedule_code(seeded), ctypes.byref(opts) if opts is not None else None, rows_ptr)
        if cov_ptr is None:
            _check(self.lib, self.lib.dfk_nls_fit_batch_dev(*args))
        else:
            _check(self.lib, self.lib.dfk_nls_fit_batch_cov_dev(*args, cov_ptr))

    def demod_tm(self, x_ptr, bufs_per_channel, C, R, N, w0, qi_ptr, dc_ptr):
        _check(self.lib, self.lib.dfk_demod_tm_dev(self._h, x_ptr, int(bufs_per_channel), int(C), int(R), int(N), float(w0),
                                                   qi_ptr, dc_ptr))

    def nls_fit_batch_tm_dev(self, x_ptr, C, bufs_per_channel, R, N, w0, init, init_dev_ptr, init_stride, seeded, opts, rows_ptr,
                             cov_ptr=None):
        init_arr = (ctypes.c_double * 4)(*[float(v) for v in init]) if init is not None else None
        args = (self._h, x_ptr, int(C), int(bufs_per_channel), int(R), int(N), float(w0), init_arr, init_dev_ptr,
                int(init_stride), schedule_code(seeded), ctypes.byref(opts) if opts is not None else None, rows_ptr)
        if cov_ptr is None:
            _check(self.lib, self.lib.dfk_nls_fit_batch_tm_dev(*args))
        else:
            _check(self.lib, self.lib.dfk_nls_fit_batch_tm_cov_dev(*args, cov_ptr))

    def ekf_dev(self, z_ptr, T, C, ld_t, ld_c, R, f_samp, f_mod, opts, rows_ptr):
        _check(self.lib, self.lib.dfk_ekf_dev(self._h, z_ptr, T, C, ld_t, ld_c, R, f_samp, f_mod,
                                              ctypes.byref(opts) if opts is not None else None, rows_ptr))

    def ekf_stream_dev(self, z_ptr, T, C, ld_t, ld_c, R, f_samp, f_mod, opts, k0, state_ptr, rows_ptr):
        _check(self.lib, self.lib.dfk_ekf_stream_dev(self._h, z_ptr, T, C, ld_t, ld_c, R, f_samp, f_mod,
                                                     ctypes.byref(opts) if opts is not None else None, k0, state_ptr,
                                                     rows_ptr))

    def ekf_smooth_dev(self, z_ptr, T, C, ld_t, ld_c, R, f_samp, f_mod, opts, k0, state_ptr, block, rows_ptr,
                       var_ptr=None, filt_rows_ptr=None, filt_var_ptr=None):
        """RTS smoother over a resident window (dfk_ekf_smooth_dev); outputs not wanted are None."""
        _check(self.lib, self.lib.dfk_ekf_smooth_dev(self._h, z_ptr, int(T), int(C), int(ld_t), int(ld_c), int(R),
                                                     float(f_samp), float(f_mod),
                                                     ctypes.byref(opts) if opts is not None else None, int(k0),
                                                     state_ptr, int(block), rows_ptr, var_ptr, filt_rows_ptr,
                                                     filt_var_ptr))

    def ekf_em_dev(self, z_ptr, T, C, ld_t, ld_c, R, f_samp, f_mod, opts, qr_init_ptr, estimate_mask, max_iter, tol,
                   block, qr_out_ptr, loglik_ptr, iters_ptr, rows_ptr=None, var_ptr=None, filt_rows_ptr=None,
                   filt_var_ptr=None):
        """EM estimates of the EKF's q and r per channel, then the smoother at them (dfk_ekf_em_dev)."""
        _check(self.lib, self.lib.dfk_ekf_em_dev(self._h, z_ptr, int(T), int(C), int(ld_t), int(ld_c), int(R),
                                                 float(f_samp), float(f_mod),
                                                 ctypes.byref(opts) if opts is not None else None, qr_init_ptr,
                                                 int(estimate_mask), int(max_iter), float(tol), int(block), qr_out_ptr,
                                                 loglik_ptr, iters_ptr, rows_ptr, var_ptr, filt_rows_ptr, filt_var_ptr))

    def synth_snr_slab_dev(self, x_ptr, T, C, ld_c, t0, f_samp, f_mod, m, amp=1.0, visibility=1.0, phi0=0.0, dphi=0.0,
                           psi0=0.0, snr_db=40.0, seed=0):
        _check(self.lib, self.lib.dfk_synth_snr_slab_dev(self._h, x_ptr, T, C, ld_c, t0, f_samp, f_mod, m, amp,
                                                         visibility, phi0, dphi, psi0, snr_db, int(seed)))

    def synth_snr_dev(self, x_ptr, T, C, f_samp, f_mod, m, amp=1.0, visibility=1.0, phi0=0.0, dphi=0.0, psi0=0.0,
                      snr_db=40.0, seed=0):
        _check(self.lib, self.lib.dfk_synth_snr_dev(self._h, x_ptr, T, C, f_samp, f_mod, m, amp, visibility, phi0,
                                                    dphi, psi0, snr_db, int(seed)))

    def sweep_demod_dev(self, nbuf, c0, R, N, f_samp, f_mod, m, qi_ptr, dc_ptr, amp=1.0, visibility=1.0, phi0=0.0, psi0=0.0,
                        snr_db=40.0, seed=0):
        _check(self.lib, self.lib.dfk_sweep_demod_dev(self._h, int(nbuf), int(c0), int(R), int(N), float(f_samp),
                                                      float(f_mod), float(m), amp, visibility, phi0, psi0, snr_db,
                                                      int(seed), qi_ptr, dc_ptr))

    def nls_sweep_dev(self, m_values, ntrials, trial0, seed_stride, R, N, f_samp, f_mod, rows_ptr, amp=1.0, visibility=1.0,
                      phi0=0.0, psi0=0.0, snr_db=40.0, seed=0, init_a=1.6, init_m=None, opts=None, cov_ptr=None):
        ms = np.ascontiguousarray(m_values, dtype=np.float64)
        args = (self._h, ms.ctypes.data_as(c_double_p), len(ms), int(ntrials), int(trial0), int(seed_stride), int(R), int(N),
                float(f_samp), float(f_mod), amp, visibility, phi0, psi0, snr_db, int(seed), float(init_a),
                float("nan") if init_m is None else float(init_m), ctypes.byref(opts) if opts is not None else None, rows_ptr)
        if cov_ptr is None:
            _check(self.lib, self.lib.dfk_nls_sweep_dev(*args))
        else:
            _check(self.lib, self.lib.dfk_nls_sweep_cov_dev(*args, cov_ptr))

    def bessel_dev(self, x_ptr, n, nmax, out_ptr):
        _check(self.lib, self.lib.dfk_bessel_dev(self._h, x_ptr, n, nmax, out_ptr))

    # ---- host-pointer calls ----------------------------------------------------------------------------
    def nls_fit_host(self, x, R, N, w0, init, seeded=True, opts=None, rows_out=None, cov_out=None):
        """x: 1-D float64 host array (numpy or a pinned torch tensor's numpy view). Returns rows[nbuf, 8].
        seeded: see schedule_code (True: every buffer from buffer 0's result; k: the reference's k-chunk chain).
        cov_out: a C-contiguous float64 array [nbuf, COV_STRIDE] that receives every buffer's parameter covariance."""
        x, xp = _host_array(x)
        nbuf = x.size // int(R)
        rows = rows_out if rows_out is not None else np.empty((nbuf, ROW_STRIDE), dtype=np.float64)
        init_arr = (ctypes.c_double * 4)(*[float(v) for v in init])
        args = (self._h, xp, x.size, int(R), int(N), float(w0), init_arr, schedule_code(seeded),
                ctypes.byref(opts) if opts is not None else None, rows.ctypes.data)
        if cov_out is None:
            _check(self.lib, self.lib.dfk_nls_fit_host(*args))
        else:
            if not (isinstance(cov_out, np.ndarray) and cov_out.dtype == np.float64 and cov_out.flags.c_contiguous
                    and cov_out.size >= nbuf * COV_STRIDE):
                raise ValueError(f"cov_out must be a C-contiguous float64 array of [{nbuf}, {COV_STRIDE}]")
            _check(self.lib, self.lib.dfk_nls_fit_cov_host(*args, cov_out.ctypes.data))
        return rows

    def nls_fit_seeded_host(self, x, R, N, w0, seed, chunks=1, opts=None, rows_out=None):
        """A host slab of a record whose buffer 0 was fitted elsewhere: `chunks` chains started from seed[4]."""
        x, xp = _host_array(x)
        nbuf = x.size // int(R)
        rows = rows_out if rows_out is not None else np.empty((nbuf, ROW_STRIDE), dtype=np.float64)
        seed_arr = (ctypes.c_double * 4)(*[float(v) for v in seed])
        _check(self.lib, self.lib.dfk_nls_fit_seeded_host(self._h, xp, x.size, int(R), int(N), float(w0), seed_arr,
                                                          int(chunks), ctypes.byref(opts) if opts is not None else None,
                                                          rows.ctypes.data))
        return rows

    def ekf_host(self, z, R, f_samp, f_mod, opts=None):
        """z: [C, T] float64 host array (channel-major). Returns rows[C, nbuf, 8]."""
        z, zp = _host_array(np.atleast_2d(z))
        C, T = z.shape
        nbuf = T // int(R)
        rows = np.empty((C, nbuf, ROW_STRIDE), dtype=np.float64)
        _check(self.lib, self.lib.dfk_ekf_host(self._h, zp, T, C, int(R), float(f_samp), float(f_mod),
                                               ctypes.byref(opts) if opts is not None else None, rows.ctypes.data))
        return rows

    # ---- raw-data ingest ---------------------------------------------------------------------------------
    def text_load_file(self, path, byte_offset=0):
        """Upload the data region of a text file and index its rows. Returns (nbytes, nrows)."""
        nb, nr = _i64(), _i64()
        _check(self.lib, self.lib.dfk_text_load_file(self._h, os.fsencode(path), int(byte_offset), ctypes.byref(nb),
                                                     ctypes.byref(nr)))
        return int(nb.value), int(nr.value)

    def text_load_host(self, text: bytes):
        nr = _i64()
        buf = ctypes.create_string_buffer(text, len(text)) if len(text) else None
        _check(self.lib, self.lib.dfk_text_load_host(self._h, ctypes.cast(buf, _vp) if buf is not None else None,
                                                     len(text), ctypes.byref(nr)))
        return int(nr.value)

    def text_parse_dev(self, ncols, out_ptr, ld_c, usecols=None):
        """Parse the resident text into out_ptr[c * ld_c + r]. Returns the number of bad (NaN) fields."""
        nbad = _i64()
        cols = (ctypes.c_int32 * int(ncols))(*[int(c) for c in usecols]) if usecols is not None else None
        _check(self.lib, self.lib.dfk_text_parse_dev(self._h, int(ncols), cols, out_ptr, int(ld_c), ctypes.byref(nbad)))
        return int(nbad.value)

    def text_release(self):
        _check(self.lib, self.lib.dfk_text_release(self._h))

    def widen_dev(self, src_ptr, dtype, T, C, time_major, out_ptr, ld_c, scale=1.0, offset=0.0):
        _check(self.lib, self.lib.dfk_widen_dev(self._h, src_ptr, RAW_DTYPES[str(dtype)], int(T), int(C),
                                                int(bool(time_major)), float(scale), float(offset), out_ptr, int(ld_c)))

    def ingest_binary_host(self, src, T, C, time_major, out_ptr, ld_c, scale=1.0, offset=0.0):
        """src: contiguous numpy array of int16 / int32 / float32 / float64 holding T * C samples."""
        src = np.ascontiguousarray(src)
        _check(self.lib, self.lib.dfk_ingest_binary_host(self._h, src.ctypes.data, RAW_DTYPES[src.dtype.name], int(T),
                                                         int(C), int(bool(time_major)), float(scale), float(offset),
                                                         out_ptr, int(ld_c)))

    def ingest_binary_file(self, path, byte_offset, dtype, T, C, time_major, out_ptr, ld_c, scale=1.0, offset=0.0):
        _check(self.lib, self.lib.dfk_ingest_binary_file(self._h, os.fsencode(path), int(byte_offset),
                                                         RAW_DTYPES[str(dtype)], int(T), int(C), int(bool(time_major)),
                                                         float(scale), float(offset), out_ptr, int(ld_c)))

    # ---- batched experiments ---------------------------------------------------------------------------
    def synth_asd_dev(self, trials_ptr, ntrials, N, f_samp, y_ptr, ld, tables_ptr=None, ntables=0, truth_ptr=None):
        _check(self.lib, self.lib.dfk_synth_asd_dev(self._h, trials_ptr, int(ntrials), int(N), float(f_samp), tables_ptr,
                                                    int(ntables), y_ptr, int(ld), truth_ptr))

    NOISE_KEYS = ("laser_frequency", "amplitude", "df", "armlength")  # DFK_NOISE_* order

    def synth_asd_noise_dev(self, trials_ptr, ntrials, N, f_samp, y_ptr, ld, noise_ptrs, noise_rows, tables_ptr=None,
                            ntables=0, truth_ptr=None):
        """noise_ptrs: four device pointers (or None) in NOISE_KEYS order, each ``noise_rows x N`` doubles."""
        arr = (ctypes.c_void_p * 4)(*[p if p else None for p in noise_ptrs])
        _check(self.lib, self.lib.dfk_synth_asd_noise_dev(self._h, trials_ptr, int(ntrials), int(N), float(f_samp),
                                                          tables_ptr, int(ntables), arr, int(noise_rows), y_ptr, int(ld),
                                                          truth_ptr))

    def trial_stats_dev(self, values_ptr, npoints, ntrials, ncols, col_stride, out_ptr, center_ptr=None):
        _check(self.lib, self.lib.dfk_trial_stats_dev(self._h, values_ptr, int(npoints), int(ntrials), int(ncols),
                                                      int(col_stride), center_ptr, out_ptr))

    # ---- post-fit step ---------------------------------------------------------------------------------
    def downsample_dev(self, x_ptr, n, R, out_ptr):
        _check(self.lib, self.lib.dfk_downsample_dev(self._h, x_ptr, int(n), int(R), out_ptr))

    def downsample_host(self, x, R):
        x, xp = _host_array(x)
        out = np.empty(x.size // int(R), dtype=np.float64)
        _check(self.lib, self.lib.dfk_downsample_host(self._h, xp, x.size, int(R), out.ctypes.data))
        return out

    def lpsd_dev(self, x_ptr, N, stride, C, ld_c, fs, opts=None) -> dict:
        """Spectra of C device-resident series; returns host arrays f[nf], ps[C, nf], psd[C, nf], enbw[nf], navs[nf]."""
        opts = opts if opts is not None else default_lpsd_opts()
        nf = _i32()
        _check(self.lib, self.lib.dfk_lpsd_plan(int(N), float(fs), ctypes.byref(opts), 0, ctypes.byref(nf), None, None,
                                                None, None, None))
        n = int(nf.value)
        f, enbw, navs = np.empty(n), np.empty(n), np.empty(n, dtype=np.int64)
        ps, psd = np.empty((int(C), n)), np.empty((int(C), n))
        _check(self.lib, self.lib.dfk_lpsd_dev(self._h, x_ptr, int(N), int(stride), int(C), int(ld_c), float(fs),
                                               ctypes.byref(opts), n, ctypes.byref(nf), f.ctypes.data, ps.ctypes.data,
                                               psd.ctypes.data, enbw.ctypes.data, navs.ctypes.data))
        return {"f": f, "ps": ps, "psd": psd, "enbw": enbw, "navs": navs}

    def lcsd_dev(self, x_ptr, Cx, ldx, y_ptr, Cy, ldy, N, stride, fs, opts=None) -> dict:
        """Cross-spectral densities of Cx device-resident series x against Cy series y on the LPSD plan; returns host
        arrays f[nf], Sxx[Cx, nf], Syy[Cy, nf], Sxy[Cx, Cy, nf] (complex128), enbw[nf], navs[nf]."""
        opts = opts if opts is not None else default_lpsd_opts()
        nf = _i32()
        _check(self.lib, self.lib.dfk_lpsd_plan(int(N), float(fs), ctypes.byref(opts), 0, ctypes.byref(nf), None, None,
                                                None, None, None))
        n = int(nf.value)
        f, enbw, navs = np.empty(n), np.empty(n), np.empty(n, dtype=np.int64)
        sxx, syy = np.empty((int(Cx), n)), np.empty((int(Cy), n))
        sxy = np.empty((int(Cx), int(Cy), n), dtype=np.complex128)
        _check(self.lib, self.lib.dfk_lcsd_dev(self._h, x_ptr, int(Cx), int(ldx), y_ptr, int(Cy), int(ldy), int(N),
                                               int(stride), float(fs), ctypes.byref(opts), n, ctypes.byref(nf),
                                               f.ctypes.data, sxx.ctypes.data, syy.ctypes.data, sxy.ctypes.data,
                                               enbw.ctypes.data, navs.ctypes.data))
        return {"f": f, "Sxx": sxx, "Syy": syy, "Sxy": sxy, "enbw": enbw, "navs": navs}

    def lcsd_cond_dev(self, x_ptr, Cx, ldx, y_ptr, Cy, ldy, N, stride, fs, opts=None) -> dict:
        """Conditioned spectra of Cy device-resident targets y given Cx witnesses x on the LPSD plan; returns host
        arrays f[nf], Sxx[Cx, Cx, nf], Syy[Cy, nf], Sxy[Cx, Cy, nf], H[Cx, Cy, nf] (complex128), Sres[Cy, nf],
        mcoh[Cy, nf], enbw[nf], navs[nf]."""
        opts = opts if opts is not None else default_lpsd_opts()
        nf = _i32()
        _check(self.lib, self.lib.dfk_lpsd_plan(int(N), float(fs), ctypes.byref(opts), 0, ctypes.byref(nf), None, None,
                                                None, None, None))
        n, cx, cy = int(nf.value), int(Cx), int(Cy)
        f, enbw, navs = np.empty(n), np.empty(n), np.empty(n, dtype=np.int64)
        sxx = np.empty((cx, cx, n), dtype=np.complex128)
        syy, sres, mcoh = np.empty((cy, n)), np.empty((cy, n)), np.empty((cy, n))
        sxy, h = np.empty((cx, cy, n), dtype=np.complex128), np.empty((cx, cy, n), dtype=np.complex128)
        _check(self.lib, self.lib.dfk_lcsd_cond_dev(self._h, x_ptr, cx, int(ldx), y_ptr, cy, int(ldy), int(N),
                                                    int(stride), float(fs), ctypes.byref(opts), n, ctypes.byref(nf),
                                                    f.ctypes.data, sxx.ctypes.data, syy.ctypes.data, sxy.ctypes.data,
                                                    h.ctypes.data, sres.ctypes.data, mcoh.ctypes.data,
                                                    enbw.ctypes.data, navs.ctypes.data))
        return {"f": f, "enbw": enbw, "navs": navs, "Sxx": sxx, "Syy": syy, "Sxy": sxy, "H": h, "Sres": sres,
                "mcoh": mcoh}

    def wiener_dev(self, x_ptr, Cx, ldx, y_ptr, Cy, ldy, N, stride, L, lead, ridge=0.0, res_ptr=None, ld_res=0,
                   filters=True, variances=True) -> dict:
        """Least-squares multi-input FIR filters of Cy device-resident targets y on Cx witnesses x (L taps, lead k0)
        and, when ``res_ptr`` is given, the residual written there ([Cy][ld_res], M = N - L + 1 samples per target).
        Returns host arrays h[Cy, Cx, L] (if ``filters``), var_y[Cy] and var_res[Cy] (if ``variances``) and the
        ``singular`` flag; an output not asked for is passed to the library as NULL."""
        cx, cy, taps = int(Cx), int(Cy), int(L)
        h = np.empty((cy, cx, taps)) if filters else None
        var_y = np.empty(cy) if variances else None
        var_res = np.empty(cy) if variances else None
        singular = _i32()
        ptr = lambda a: a.ctypes.data if a is not None else None  # noqa: E731
        _check(self.lib, self.lib.dfk_wiener_dev(self._h, x_ptr, cx, int(ldx), y_ptr, cy, int(ldy), int(N), int(stride),
                                                 taps, int(lead), float(ridge), res_ptr, int(ld_res), ptr(h),
                                                 ptr(var_y), ptr(var_res), ctypes.byref(singular)))
        return {"h": h, "var_y": var_y, "var_res": var_res, "singular": bool(singular.value)}

    def stability_dev(self, v_ptr, N, stride, C, ld_c, fs, data_type, kinds, m):
        """Stability deviations of C device-resident series (dfk_stability_dev) at the averaging factors ``m``.
        ``data_type``: STAB_PHASE or STAB_FREQ; ``kinds``: a bitmask of STAB_BITS.  Returns host arrays dev[4, C, n_m]
        and n[4, n_m] in STAB_KINDS order; slots of kinds not requested stay NaN and 0."""
        ms = np.ascontiguousarray(m, dtype=np.int64)
        dev = np.full((4, int(C), ms.size), np.nan)
        n = np.zeros((4, ms.size), dtype=np.int64)
        _check(self.lib, self.lib.dfk_stability_dev(self._h, v_ptr, int(N), int(stride), int(C), int(ld_c), float(fs),
                                                    int(data_type), int(kinds), ms.ctypes.data, ms.size,
                                                    dev.ctypes.data, n.ctypes.data))
        return dev, n

    def set_host_slab_bytes(self, nbytes=0):
        """Slab size of the host-pointer entries (0: defaults); small values make a short record stream."""
        _check(self.lib, self.lib.dfk_set_host_slab_bytes(self._h, int(nbytes)))

    # ---- introspection ---------------------------------------------------------------------------------
    def lm_counters(self, reset=False) -> dict:
        c = LmCounters()
        _check(self.lib, self.lib.dfk_lm_counters_read(self._h, ctypes.byref(c), int(bool(reset))))
        return {k: int(getattr(c, k)) for k, _ in LmCounters._fields_}

    def profile_enable(self, on=True):
        _check(self.lib, self.lib.dfk_profile_enable(self._h, int(bool(on))))

    def profile_read(self, reset=False) -> dict:
        """Summed device milliseconds and region counts: demod launches and LM launches."""
        ms = (ctypes.c_double * PROFILE_KINDS)()
        n = (_i64 * PROFILE_KINDS)()
        _check(self.lib, self.lib.dfk_profile_read(self._h, ms, n, int(bool(reset))))
        return {"demod_ms": ms[0], "demod_regions": int(n[0]), "lm_ms": ms[1], "lm_regions": int(n[1]),
                "seed_ms": ms[2], "seed_regions": int(n[2]), "ekf_ms": ms[3], "ekf_regions": int(n[3])}

    def probe_fp64_tflops(self) -> float:
        v = ctypes.c_double()
        _check(self.lib, self.lib.dfk_probe_fp64(self._h, ctypes.byref(v)))
        return float(v.value)

    def launch_count(self) -> int:
        return int(self.lib.dfk_launch_count(self._h))


class dev_overrides:
    """``with dev_overrides(DFK_NO_TILE=1): ...`` -- kernel-selection overrides for tuning runs and A/B tests,
    set through the library's explicit call (it never reads the environment) and cleared on exit."""

    def __init__(self, **values):
        self.values = values

    def __enter__(self):
        lib = load_library()
        for k, v in self.values.items():
            _check(lib, lib.dfk_dev_set(k.encode(), int(v)))
        return self

    def __exit__(self, *exc):
        load_library().dfk_dev_clear()


def demod_path(R, w0) -> int:
    return int(load_library().dfk_demod_path(int(R), float(w0)))


def device_count() -> int:
    return int(load_library().dfk_device_count())


_ctx_cache = threading.local()


def get_context(device: int = 0) -> Context:
    """Per-thread, per-device cached context."""
    cache = getattr(_ctx_cache, "ctx", None)
    if cache is None:
        cache = _ctx_cache.ctx = {}
    if device not in cache:
        cache[device] = Context(device)
    return cache[device]
