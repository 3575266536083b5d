"""The façade of the reference, ``DeepFitFramework`` (core.py:22-609), over the GPU fitters, generators and ingest.

Everything either side of the readout path is here under the reference's names: ``load_raw`` / ``load_fit`` /
``to_txt`` (the DFMSWPM ``raw_data`` and ``fit_data`` text formats), ``simulate`` (main and witness channel),
``new_sim`` / ``create_witness_channel``, ``fit`` and ``calc_lpsd``.  Plotting and the experimental W-DFMI fitters
stay with the reference (``fit`` hands those method names to the reference's classes when it is importable;
INTEGRATION.md shows the opposite direction too: the reference's own façade pointed at these fitters).  Call
signatures, default labels, the ``tau`` column, the error behaviour (log + ``None``) and the fields of the returned
objects are those of the reference.  ``DeepFitObject.calc_csd`` is this package's addition: the cross-spectral estimate
(CSD, coherence, transfer function) of one fit against another on the LPSD frequency plan; ``calc_conditioned`` is its
multi-witness counterpart (joint transfer functions, residual PSD, multiple coherence), and ``subtract_witnesses``
performs that subtraction in the time domain (least-squares FIR filters, the cleaned series).
"""
from __future__ import annotations

import logging

import numpy as np

from .fitters import EKFFitter, StandardNLSFitter

_HEADER_LINES = 13  # both DFMSWPM text formats: 12 '%' lines and the column names (core.py:280, 310)


def _header_values(path):
    """The digits of header lines 3..11 (core.py:146-147: every character that is not a digit or a dot is dropped)."""
    with open(path) as f:
        lines = [f.readline() for _ in range(11)]
    return ["".join(c for c in line if c in "1234567890.") for line in lines[2:11]]


def _reference_fitters():
    """The experimental W-DFMI / HW-DFMI fitters of the reference (bound to a general-purpose optimiser, outside this package), under
    the method names core.py:452-459 gives them -- available when the reference itself is importable as ``DeepFMKit``."""
    try:
        from DeepFMKit import fitters as ref
    except Exception:
        return {}
    names = {"wdfmi_ortho": "WDFMI_OrthogonalFitter", "wdfmi_nls": "WDFMI_NLSFitter", "wdfmi_seq": "WDFMI_SequentialFitter",
             "hwdfmi": "HWDFMI_Fitter"}
    return {method: getattr(ref, cls) for method, cls in names.items() if hasattr(ref, cls)}


class DeepRawObject:
    """One channel of raw data: what the fitters read (data.py:16-118 holds the full container).

    ``data`` is the one-column pandas frame of the reference.  A record that already lives on the GPU (io.load_raw,
    io.load_binary, the device generator) is carried as ``device_data`` -- a 1-D float64 CUDA tensor the fitters read
    in place -- and the frame is built from it only when ``data`` is asked for."""

    def __init__(self, data=None, f_samp=None, f_mod=None, label=None, sim=None, t0=0, device_data=None, column="ch0"):
        import pandas as pd
        if data is not None and not hasattr(data, "columns"):
            data = pd.DataFrame(np.asarray(data, dtype=np.float64).reshape(-1), columns=[column])
        self._data = data
        self.device_data = device_data
        self._column = column
        self.f_samp = f_samp
        self.f_mod = f_mod
        self.label = label
        self.sim = sim
        self.t0 = t0
        self.phi_sim = None
        self.raw_file = None

    @property
    def data(self):
        if self._data is None and self.device_data is not None:
            import pandas as pd
            self._data = pd.DataFrame(self.device_data.detach().cpu().numpy().reshape(-1), columns=[self._column])
        return self._data

    @data.setter
    def data(self, value):
        self._data = value
        self.device_data = None  # the frame is the truth once somebody assigns it

    def __len__(self):
        if self.device_data is not None:
            return int(self.device_data.shape[0])
        return 0 if self._data is None else int(self._data.shape[0])

    def info(self):
        """Log label and rates (data.py:43-57)."""
        logging.info("\nDeepRawObject\nLabel: {}\nStart time: {}\nSampling frequency: {}\nModulation frequency: {}\n".format(
            self.label, self.t0, self.f_samp, self.f_mod))

    def parse_header(self):
        """t0, f_samp, f_mod from the header of this object's ``raw_file``.  (data.py:88-110 takes them from one line
        too high -- the channel count becomes ``t0``, the start time ``f_samp`` -- which no caller relies on; the lines
        read here are those of the format, as core.py:129-174 reads them.)"""
        if self.raw_file is None:
            logging.error("No file specified !!")
            return
        v = _header_values(self.raw_file)
        self.t0, self.f_samp, self.f_mod = int(v[1]), float(v[2]), float(v[3])

    def to_txt(self, filename):
        """Write the channel as a one-column DFMSWPM text record under the header of data.py:60-85.

        The reference's writer repeats the FIRST sample on every row (``self.data.iloc[0][0]``, data.py:83); this one
        writes the samples, each with the shortest digits that read back bit-identically (``repr``), so that
        ``load_raw`` of the file returns the record."""
        lines = ["% fit_data", "% Message goes here", "% Number of channels: {}".format(1),
                 "% Start time: {}".format(self.t0), "% Sampling frequency: {}".format(self.f_samp),
                 "% Modulation frequency: {}".format(self.f_mod), "% n: {}".format(0), "% Downsampling factor: {}".format(0),
                 "% Fit data rate: {}".format(0), "% Initial amplitude: {}".format(0),
                 "% Initial modulation depth: {}".format(0), "%", "ch0 "]
        frame = self.data
        values = np.zeros(0) if frame is None else np.asarray(frame.iloc[:, 0], dtype=np.float64)
        with open(filename, "w") as f:
            f.write("\n".join(lines) + "\n")
            f.write("".join(repr(float(x)) + " \n" for x in values))


class DeepFitObject:
    """Result arrays + fit geometry, the fields core.py:372-386 fills."""

    def __init__(self):
        self.fit_file = None
        self.label = None
        self.n = self.R = self.fs = self.nbuf = None
        self.ndata = self.init_a = self.init_m = 0
        self.t0 = 0
        self.f_samp = self.f_mod = None
        self.ssq = self.amp = self.m = self.tau = self.phi = self.psi = self.dc = self.time = None
        # one-sigma errors, filled by fit(..., uncertainties=True) (not part of the fit_data text format)
        self.amp_err = self.m_err = self.phi_err = self.psi_err = self.tau_err = None
        # spectral-estimate settings and results (data.py:148-158)
        self.f = None
        self.Sxx = None
        self.olap = "default"
        self.bmin = 1
        self.Lmin = 0
        self.Jdes = 500
        self.Kdes = 100
        self.order = 0
        self.win = np.kaiser
        self.psll = 200

    def info(self):
        """Log label, rates and fit geometry (data.py:161-177)."""
        logging.info("\nDeepFitObject\nLabel: {}\nStart time: {}\nSampling frequency: {}\nModulation frequency: {}\n"
                     "Downsampling factor: {}\nn: {}\nFit data rate: {}\n".format(self.label, self.t0, self.f_samp, self.f_mod,
                                                                              self.R, self.n, self.fs))

    def to_txt(self, filename):
        """Save the fit in the DFMSWPM ``fit_data`` text format (data.py:180-213): twelve '%' header lines, the
        column names, then ``ssq amp m phi psi dc`` per buffer, every number as ``str`` of the float64 (shortest digits
        that round-trip) followed by one space -- byte for byte what the reference writes."""
        lines = ["% fit_data", "% Message goes here", "% Number of channels: {}".format(1),
                 "% Start time: {}".format(self.t0), "% Sampling frequency: {}".format(self.f_samp),
                 "% Modulation frequency: {}".format(self.f_mod), "% n: {}".format(int(self.n)),
                 "% Downsampling factor: {}".format(int(self.R)), "% Fit data rate: {}".format(self.fs),
                 "% Initial amplitude: {}".format(self.init_a), "% Initial modulation depth: {}".format(self.init_m), "%",
                 "ssq0 amp0 m0 phi0 psi0 dc0 "]
        cols = [np.asarray(getattr(self, c), dtype=np.float64) for c in ("ssq", "amp", "m", "phi", "psi", "dc")]
        with open(filename, "w") as f:
            f.write("\n".join(lines) + "\n")
            for row in zip(*cols):
                f.write("".join(str(v) + " " for v in row) + "\n")

    def parse_header(self):
        """t0, rates, n, R, fs from the header of this object's ``fit_file``.  (data.py:216-236 reads one line too high
        and fails on ``int('400.0')`` for any file ``to_txt`` wrote; the lines read here are those of the format, as
        core.py:129-174 reads them.)"""
        if self.fit_file is None:
            logging.error("No file specified !!")
            return
        v = _header_values(self.fit_file)
        self.t0, self.f_samp, self.f_mod = int(v[1]), float(v[2]), float(v[3])
        self.n, self.R, self.fs = int(v[4]), int(v[5]), float(v[6])

    def calc_lpsd(self):
        """LPSD of the fitted interferometric phase (data.py:239-244), on the device."""
        from .spectra import lpsd
        self.f, _, self.Sxx, _, _, _ = lpsd(self.phi, self.fs, self.olap, self.bmin, self.Lmin, self.Jdes, self.Kdes,
                                            self.order, self.win, self.psll, return_type="legacy")

    def calc_csd(self, other, column="phi"):
        """Cross-spectral estimate of this fit's ``column`` against ``other``'s on the device, with this object's
        spectral settings: the ``lcsd`` dict (f, Sxx, Syy, Sxy, coh, tf, enbw, navs), this fit as x and ``other`` as y.
        Stores nothing.  Both fits must have the same fit rate and the same number of buffers."""
        from .spectra import lcsd
        if self.fs != other.fs:
            raise ValueError(f"fit rates differ: {self.fs} and {other.fs}")
        x, y = getattr(self, column), getattr(other, column)
        if x is None or y is None:
            raise ValueError(f"both fits need a '{column}' series")
        if len(x) != len(y):
            raise ValueError(f"series lengths differ: {len(x)} and {len(y)}")
        return lcsd(x, y, self.fs, self.olap, self.bmin, self.Lmin, self.Jdes, self.Kdes, self.order, self.win,
                    self.psll)

    def calc_conditioned(self, witness_fits, column="phi"):
        """Conditioned spectra of this fit's ``column`` given the same column of every fit in ``witness_fits`` (one fit
        or a sequence of up to 64), on the device with this object's spectral settings: the ``lcsd_conditioned`` dict
        (f, enbw, navs, Sxx, Syy, Sxy, H, Sres, mcoh) with this fit as the one target.  Stores nothing.  Every fit must
        have this fit's rate and number of buffers."""
        from .spectra import lcsd_conditioned
        xs, y = self._witness_series(witness_fits, column)
        return lcsd_conditioned(xs, y, self.fs, self.olap, self.bmin, self.Lmin, self.Jdes, self.Kdes, self.order,
                                self.win, self.psll)

    def subtract_witnesses(self, witness_fits, taps, lead=None, ridge=0.0, column="phi"):
        """Time-domain witness subtraction of this fit's ``column`` on the device: the ``wiener_subtract`` dict (h,
        offsets, n0, lead, residual, var_y, var_res, explained, singular) with the same column of every fit in
        ``witness_fits`` (one fit or a sequence of up to 64) as witnesses and this fit as the one target.  Stores
        nothing.  Every fit must have this fit's rate and number of buffers."""
        from .spectra import wiener_subtract
        xs, y = self._witness_series(witness_fits, column)
        return wiener_subtract(xs, np.asarray(y, dtype=np.float64), taps, lead, ridge)

    def calc_stability(self, column="phi", kinds=("oadev", "mdev", "tdev", "ohdev"), taus="octave"):
        """Time-domain stability of this fit's ``column`` on the device: the ``stability`` dict (taus, m and, per kind,
        the deviation, its simple error and its term count) with the column as the averaged series (``data_type``
        "freq") at the fit rate, so the deviations are in the column's units.  Stores nothing."""
        from .spectra import stability
        x = getattr(self, column)
        if x is None:
            raise ValueError(f"this fit has no '{column}' series")
        return stability(np.asarray(x, dtype=np.float64), self.fs, kinds=kinds, taus=taus, data_type="freq")

    def _witness_series(self, witness_fits, column):
        """([Cx, N] witness columns, this fit's column) after checking that there is at least one witness fit and that
        every fit has this fit's rate and length."""
        if isinstance(witness_fits, DeepFitObject):
            witness_fits = [witness_fits]
        witness_fits = list(witness_fits)
        if not witness_fits:
            raise ValueError("need at least one witness fit")
        y = getattr(self, column)
        if y is None:
            raise ValueError(f"this fit has no '{column}' series")
        xs = []
        for w in witness_fits:
            if w.fs != self.fs:
                raise ValueError(f"fit rates differ: {self.fs} and {w.fs}")
            x = getattr(w, column)
            if x is None:
                raise ValueError(f"every witness fit needs a '{column}' series")
            if len(x) != len(y):
                raise ValueError(f"series lengths differ: {len(y)} and {len(x)}")
            xs.append(np.asarray(x, dtype=np.float64))
        return np.stack(xs), y


class DeepFitFramework:
    def __init__(self, raw_file=None, fit_file=None, raw_labels=None, fit_labels=None):
        """Fields and the load-on-construction behaviour of core.py:92-117."""
        self.raw_file = raw_file
        self.fit_file = fit_file
        self.lasers = {}
        self.ifos = {}
        self.sims = {}
        self.raws = {}
        self.fits = {}
        self.fits_df = {}
        self.channr = None
        self.n = None
        self.t0 = None
        self.R = None
        self.fs = None
        self.f_samp = None
        self.f_mod = None
        self.ndata = 10
        self.init_a = 1.6
        self.init_m = 6.0
        self.cfit = None
        if self.raw_file is not None:
            self.load_raw(labels=raw_labels)
        if self.fit_file is not None:
            self.load_fit(labels=fit_labels)

    def to_txt(self, filepath="./", labels=None):
        """One ``fit_data`` text file per fit, ``<filepath><label>.txt`` (core.py:119-127)."""
        for label in (labels if labels is not None else list(self.fits)):
            fit = self.fits[label]
            fit.to_txt(filepath + (label if labels is not None else fit.label) + ".txt")

    def parse_header(self, file_select="raw"):
        """Header of ``self.raw_file`` or ``self.fit_file`` (core.py:129-174)."""
        if file_select == "raw" and getattr(self, "raw_file", None) is not None:
            from .io import parse_header
            hdr = parse_header(self.raw_file)
            self.channr, self.t0, self.f_samp, self.f_mod = hdr["channels"], hdr["t0"], hdr["f_samp"], hdr["f_mod"]
        elif file_select == "fit" and getattr(self, "fit_file", None) is not None:
            v = _header_values(self.fit_file)
            self.channr, self.t0, self.f_samp, self.f_mod = int(v[0]), int(v[1]), float(v[2]), float(v[3])
            self.n, self.R, self.fs = int(v[4]), int(v[5]), float(v[6])
        else:
            logging.error("No files specified !!")
            return
        logging.info("Number of channels: {}".format(self.channr))
        logging.info("Starting time: {}".format(self.t0))
        logging.info("Sampling frequency: {}".format(self.f_samp))
        logging.info("Modulation frequency: {}".format(self.f_mod))
        if file_select == "fit":
            logging.info("n: {}".format(self.n))
            logging.info("Downsampling factor: {}".format(self.R))
            logging.info("Fit data rate: {}".format(self.fs))

    def load_fit(self, fit_file=None, labels=None):
        """Load a DFMSWPM ``fit_data`` file (core.py:288-332): six columns ``ssq amp m phi psi dc`` per channel under
        a 13-line header, one ``DeepFitObject`` per channel.  A results table of a few MB: read on the host, every
        number correctly rounded as ``numpy.genfromtxt`` reads it.  Default labels are ``<file>_ch<k>`` with the raw
        file's name as in the reference, or the fit file's when no raw file is loaded (the reference raises there)."""
        if fit_file is not None:
            self.fit_file = fit_file
        if self.fit_file is None:
            logging.error("No fit file specified !!")
            return
        self.parse_header(file_select="fit")
        if labels is None:
            stem = self.raw_file if self.raw_file is not None else self.fit_file
            labels = [stem + "_ch" + str(c) for c in range(self.channr)]
        else:
            assert len(labels) == self.channr
        with open(self.fit_file) as f:
            for _ in range(_HEADER_LINES):
                f.readline()
            rows = [line.split() for line in f if line.strip()]
        width = 6 * self.channr
        data = np.array([[float(v) for v in r] for r in rows if len(r) == width], dtype=np.float64).reshape(-1, width)
        if len(data) != len(rows):  # genfromtxt(invalid_raise=False) drops rows of the wrong width with a warning
            logging.warning(f"{self.fit_file}: {len(rows) - len(data)} rows did not have {width} columns and were skipped")
        for k in range(self.channr):
            fit = DeepFitObject()
            fit.fit_file = self.fit_file
            fit.nbuf = len(data)
            fit.n, fit.t0, fit.R, fit.fs = self.n, self.t0, self.R, self.fs
            fit.f_samp, fit.f_mod = self.f_samp, self.f_mod
            fit.ndata, fit.init_a, fit.init_m = self.ndata, self.init_a, self.init_m
            for j, col in enumerate(("ssq", "amp", "m", "phi", "psi", "dc")):
                setattr(fit, col, data[:, 6 * k + j].copy())
            fit.time = np.arange(0, fit.nbuf / self.fs, 1.0 / self.fs)
            fit.label = labels[k]
            self.fits[labels[k]] = fit

    def new_sim(self, label=None):
        """A default ``DFMIObject`` under ``label`` (a time stamp when omitted), core.py:248-257."""
        from .physics import DFMIObject, InterferometerConfig, LaserConfig
        if label is None:
            from datetime import datetime
            label = datetime.now().strftime("%Y%m%d_%H%M%S")
        self.sims[label] = DFMIObject(label, LaserConfig(), InterferometerConfig())
        return label

    def create_witness_channel(self, main_channel_label, witness_channel_label, m_witness=None, delta_l_witness=None):
        """A static witness interferometer on the main channel's laser (core.py:519-588): path difference from the
        target ``m_witness`` (default 0.1) or given directly, phase offset set so that it sits at mid-fringe."""
        from .physics import SPEED_OF_LIGHT, DFMIObject, InterferometerConfig
        if main_channel_label not in self.sims:
            raise KeyError(f"Main channel '{main_channel_label}' not found in framework.")
        if delta_l_witness is not None and m_witness is not None:
            raise ValueError("Please specify either delta_l_witness or m_witness, but not both.")
        main = self.sims[main_channel_label]
        laser = main.laser
        if m_witness is not None:
            m_target = m_witness
        elif delta_l_witness is not None:
            m_target = (2 * np.pi * laser.df * delta_l_witness) / SPEED_OF_LIGHT
        else:
            m_target = 0.1
        ifo = InterferometerConfig(label=f"{witness_channel_label}_ifo")
        ifo.arml_mod_amp = 0.0
        ifo.arml_mod_n = 0.0
        if laser.df == 0:
            raise ValueError("Cannot set 'm_witness' when laser 'df' is zero.")
        delta_l = (m_target * SPEED_OF_LIGHT) / (2 * np.pi * laser.df)
        ifo.ref_arml = 0.01
        ifo.meas_arml = ifo.ref_arml + delta_l
        f0 = SPEED_OF_LIGHT / laser.wavelength
        fringe = (2 * np.pi * f0 * delta_l) / SPEED_OF_LIGHT
        ifo.phi = ((np.pi / 2.0) + fringe) % (2 * np.pi)
        witness = DFMIObject(witness_channel_label, laser, ifo, f_samp=main.f_samp)
        witness.fit_n = main.fit_n
        self.sims[witness_channel_label] = witness
        logging.debug(f"Created witness channel '{witness_channel_label}' with final m_witness={witness.m:.3f}.")
        return witness

    def load_raw(self, raw_file=None, labels=None):
        """Load a raw_data file (core.py:259-286): parsed on the GPU, one ``DeepRawObject`` per channel whose samples
        stay on the device for the fitters."""
        from .io import load_raw
        if raw_file is not None:
            self.raw_file = raw_file
        if getattr(self, "raw_file", None) is None:
            logging.error("No raw file specified !!")
            return
        self.parse_header(file_select="raw")
        for raw in load_raw(self.raw_file, labels=labels):
            self.raws[raw.label] = raw

    def load_sim(self, sim):
        self.sims[sim.label] = sim

    def simulate(self, main_label, n_seconds, mode="asd", witness_label=None, snr_db=None, trial_num=0, verbose=False):
        """Simulate the channel ``self.sims[main_label]`` on the GPU (core.py:176-243 -> SignalGenerator.generate) and
        store the record in ``self.raws`` -- with ``witness_label``, the linked witness channel beside it ('asd' mode;
        the reference's 'snr' engine ignores the witness, physics.py:414-415, and so does this one)."""
        import time
        from .simulation import simulate
        t0 = time.time()
        if main_label not in self.sims:
            logging.error(f"Main simulation label '{main_label}' not found!")
            return
        witness_config = None
        if witness_label:
            if witness_label not in self.sims:
                logging.error(f"Witness simulation label '{witness_label}' not found!")
                return
            witness_config = self.sims[witness_label]
        if mode == "snr" and snr_db is None:
            logging.error("SNR mode requires a value for 'snr_db'.")
            logging.error("Simulation failed to generate data.")
            return
        if mode not in ("asd", "snr"):
            logging.error(f"Unknown simulation mode: '{mode}'")
            logging.error("Simulation failed to generate data.")
            return
        main_config = self.sims[main_label]
        if mode == "asd" and witness_config is not None:
            raws = simulate(main_config, n_seconds, mode=mode, trial_num=trial_num, witness=witness_config)
        else:
            raws = (simulate(main_config, n_seconds, mode=mode, snr_db=snr_db, trial_num=trial_num),)
        for raw in raws:
            self.raws[raw.label] = raw
        main_config.simtime = time.time() - t0

    def load_raw_object(self, raw: DeepRawObject, label=None):
        label = label or raw.label
        raw.label = label
        self.raws[label] = raw
        return raw

    def calc_lpsd(self, labels=None):
        """LPSD of phi for the fits under ``labels``, or for every fit (core.py:590-609)."""
        if labels is not None:
            for label in labels:
                try:
                    self.fits[label].calc_lpsd()
                except KeyError:
                    logging.warning("Specified label is invalid!")
        else:
            for fit in self.fits.values():
                fit.calc_lpsd()

    def fit_init(self, label, n):
        """(R, fs, nbuf) of a fitting run (core.py:390-422)."""
        raw = self.raws[label]
        R = int(raw.f_samp / raw.f_mod * n)
        fs = raw.f_samp / R
        nbuf = int(len(raw) / R)
        if nbuf == 0:
            logging.error("Check buffer size !! Calculated nbuf is zero.")
        return R, fs, nbuf

    def fit(self, main_label, method="nls", fit_label=None, **kwargs):
        fitter_map = {"nls": StandardNLSFitter, "ekf": EKFFitter}
        fitter_map.update(_reference_fitters())  # the W-DFMI family stays with the reference (core.py:452-459)
        if method not in fitter_map:
            logging.error(f"Unknown fit method: '{method}'. Available: {list(fitter_map.keys())}")
            return
        FitterClass = fitter_map[method]
        if main_label not in self.raws:
            logging.error(f"Invalid raw data label: '{main_label}' !!")
            return
        main_raw = self.raws[main_label]
        if fit_label is None:
            fit_label = f"{main_label}_{method}"
        n_cycles = kwargs.get("n")
        if n_cycles is None:
            sim = getattr(main_raw, "sim", None)
            sim_obj = self.sims.get(sim.label if sim else main_label)
            n_cycles = sim_obj.fit_n if sim_obj else 20
        R, fs, nbuf = self.fit_init(main_label, n_cycles)

        phi_sim = getattr(main_raw, "phi_sim", None)
        if phi_sim is not None and len(phi_sim) > 0:  # core.py:480-481: ground truth at the fit rate
            from .spectra import vectorized_downsample
            main_raw.phi_sim_downsamp = vectorized_downsample(phi_sim, R)

        fit_config = {"n": n_cycles}
        fitter_args = {"main_raw": main_raw}
        if "wdfmi" in method:  # core.py:492-496 (reference fitters only)
            witness_label = kwargs.get("witness_label")
            if not witness_label or witness_label not in self.raws:
                logging.error(f"W-DFMI method '{method}' requires a valid 'witness_label'.")
                return
            fitter_args["witness_raw"] = self.raws[witness_label]
        fitter = FitterClass(fit_config)
        results_df = fitter.fit(**fitter_args, **kwargs)
        if results_df is None or results_df.empty:
            logging.error(f"{FitterClass.__name__} returned no results.")
            return None
        sim = getattr(main_raw, "sim", None)
        results_df["tau"] = results_df["m"] / (2 * np.pi * sim.laser.df) if sim else 0.0  # core.py:506-507
        uncertainties = "m_err" in results_df.columns
        if uncertainties:  # the error of tau follows from m's exactly as tau does
            results_df["tau_err"] = results_df["m_err"] / (2 * np.pi * sim.laser.df) if sim else 0.0
        self.fits_df[fit_label] = results_df

        fit = DeepFitObject()
        fit.n, fit.R, fit.fs, fit.nbuf = n_cycles, R, fs, nbuf
        fit.ndata, fit.init_a, fit.init_m = fit_config.get("ndata", 0), 0, 0  # Q5: the reference stores zeros
        fit.t0 = getattr(main_raw, "t0", 0)
        fit.f_samp, fit.f_mod = main_raw.f_samp, main_raw.f_mod
        for col in ("ssq", "amp", "m", "tau", "phi", "psi", "dc"):
            setattr(fit, col, np.asarray(results_df[col], dtype=np.float64) if col != "tau" or sim
                    else np.zeros(len(results_df)))
        if uncertainties:
            for col in ("amp_err", "m_err", "tau_err", "phi_err", "psi_err"):
                setattr(fit, col, np.asarray(results_df[col], dtype=np.float64) if col != "tau_err" or sim
                        else np.zeros(len(results_df)))
        fit.time = np.arange(0, fit.ssq.shape[0] / fit.fs, 1.0 / fit.fs)
        fit.label = fit_label
        self.fits[fit_label] = fit
        return fit
