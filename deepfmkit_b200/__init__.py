"""B200-native DFMI readout hot path: lock-in demodulation, batched LM NLS fit, EKF (sm_100a CUDA)."""
from . import fit  # noqa: F401  (module-level solver tunables, patched like the reference's fit.py)
from .core import DeepFitFramework, DeepFitObject, DeepRawObject  # noqa: F401
from .fitters import (BaseFitter, EKFFitter, StandardNLSFitter, ekf_fit_batch, ekf_smooth, nls_fit_batch,  # noqa: F401
                      rows_to_frame)

from .io import load_binary, load_raw, load_raw_device, parse_header  # noqa: F401,E402
from .spectra import lcsd, lcsd_conditioned, lpsd, vectorized_downsample, wiener_subtract  # noqa: F401,E402
from . import factories, helpers, physics, waveforms  # noqa: F401,E402
from .experiments import Experiment  # noqa: F401,E402
from .simulation import simulate, simulate_asd_batch  # noqa: F401,E402
from .montecarlo import crlb_sigma_m, nls_sweep, nls_sweep_sharded  # noqa: F401,E402
from . import workers  # noqa: F401,E402

__all__ = ["nls_sweep", "nls_sweep_sharded", "crlb_sigma_m", "BaseFitter", "StandardNLSFitter", "EKFFitter", "DeepFitFramework", "DeepRawObject", "DeepFitObject",
           "nls_fit_batch", "ekf_fit_batch", "ekf_smooth", "rows_to_frame", "fit", "lpsd", "lcsd", "lcsd_conditioned", "wiener_subtract", "vectorized_downsample",
           "load_raw", "load_raw_device", "load_binary", "parse_header", "Experiment", "simulate", "simulate_asd_batch", "factories", "physics",
           "waveforms", "helpers", "workers"]
