/*
 * dfk_b200.h -- C ABI of the B200-native DFMI readout hot path.
 *
 * This is the drop-in boundary for mdovale/DeepFMKit's readout path: every
 * entry point names the reference interface it replaces (file:line into the
 * upstream repo).  Plain pointers and sizes only; all floating point is IEEE
 * fp64, little endian, row-major.  The library is CUDA-only: there is no CPU
 * fallback, and every call fails with DFK_ERR_CUDA if no sm_100 device is
 * usable.
 *
 * Conventions
 *   - harmonic vector  qi[b] = [Q_1..Q_N, I_1..I_N]   (Q = cosine mean, I = sine mean, 1/R
 *     normalised) -- the layout of QI_data_mean in fitters.py:45-49
 *   - parameter vector [amp, m, phi, psi]              -- fit.py:93
 *   - result row       [amp, m, phi, psi, dc, ssq, fitok, aux] (8 doubles, DFK_ROW_STRIDE);
 *     columns 0..6 are the reference's result-frame columns (fitters.py:55-58), fitok stored
 *     as a double holding 0/1/2; aux = accepted LM steps (NLS) or 0 (EKF)
 *   - covariance row [C_aa, C_am, C_aphi, C_mm, C_mphi, C_phiphi, C_psipsi, s^2] (8 doubles,
 *     DFK_COV_STRIDE), one per result row and laid out like the rows: s^2 (J^T J)^-1 at the row's
 *     parameters, s^2 = ssq / (2N - 4) (see dfk_lm_cov)
 *   - "dev" pointers are device pointers on the context's device; "host" pointers are host
 *     memory (pinned memory is detected and copied from directly, pageable memory is staged)
 *   - all calls return 0 on success or a negative DFK_ERR_* code; dfk_last_error() gives the
 *     message for the calling thread.  Numerical failure of a fit is never an error: it is
 *     reported through fitok exactly as the reference does (fit.py:334-349).
 */
#ifndef DFK_B200_H
#define DFK_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DFK_ABI_VERSION 6
#define DFK_ROW_STRIDE 8
#define DFK_COV_STRIDE 8
#define DFK_MAX_HARMONICS 64

#define DFK_PROFILE_KINDS 4

/* Warm-start schedule of a record, the `seeded` argument of the NLS entries (fitters.py:370-428):
 *   DFK_SCHED_INDEPENDENT  every buffer is a cold start from init (single-buffer fits, workers.py:167-173)
 *   k >= 1                 buffer 0 from init; the buffers after it in k chunks (np.array_split), the first buffer of
 *                          a chunk started from buffer 0's result, every other from its predecessor's result:
 *                          StandardNLSFitter.fit(parallel=True, n_cores=k) (fitters.py:395-428); k = 1 is also the
 *                          sequential chain of parallel=False (fitters.py:370-393)
 *   DFK_SCHED_EACH         every buffer its own chunk (the pool schedule at n_cores >= nbuf - 1)
 * On the GPU all buffers are first fitted from their chunk's seed at once; buffers whose first descent fails are
 * then walked in record order from their predecessor's result, which is what the chain would have done. */
#define DFK_SCHED_INDEPENDENT 0
#define DFK_SCHED_EACH (-1)

#define DFK_OK 0
#define DFK_ERR_ARG (-1)
#define DFK_ERR_CUDA (-2)
#define DFK_ERR_NOMEM (-3)

/* Tunables of the reference solver; module globals in fit.py:5-16 that users patch at run
 * time, so the host shim reads them at call time and passes them here. */
typedef struct dfk_lm_opts {
    int32_t max_lma_steps;        /* fit.py:7   MAX_LMA_STEPS               (100)  */
    int32_t lanes_per_fit;        /* 0 = auto; 1,2,4,8,16,32 lanes cooperate on one fit */
    double conv_improve;          /* fit.py:8   LMA_CONVERGENCE_IMPROVE      (1e-9) */
    double conv_param;            /* fit.py:9   LMA_CONVERGENCE_PARAM_CHANGE (1e-9) */
    double fitok_threshold;       /* fit.py:10  FITOK_THRESHOLD              (1e-3) */
    double m_grid_min;            /* fit.py:12  M_GRID_MIN                   (5.0)  */
    double m_grid_max;            /* fit.py:13  M_GRID_MAX                   (30.0) */
    double m_grid_step;           /* fit.py:14  M_GRID_STEP                  (0.5)  */
    double bessel_amp_threshold;  /* fit.py:15  BESSEL_AMP_THRESHOLD         (0.05) */
    double sincos_amp_threshold;  /* fit.py:16  SINCOS_AMP_THRESHOLD         (0.1)  */
} dfk_lm_opts;

/* EKF settings; defaults of EKFFitter.fit (fitters.py:241-248). */
typedef struct dfk_ekf_opts {
    double init[4];     /* init_a, init_m, init_phi, init_psi   (1.6, 6.0, 0, 0) */
    double p0_diag[5];  /* initial covariance diagonal           (1,1,1,1,1)      */
    double q_diag[5];   /* process noise diagonal (1e-8,1e-8,1e-6,1e-6,1e-8)      */
    double r_val;       /* measurement variance; NaN = var(record) per channel (fitters.py:256) */
    double init_dc;     /* initial dc state; NaN = mean(record) per channel (fitters.py:253)    */
} dfk_ekf_opts;

/* Work counters of the LM kernels (for the FP64 flop accounting in bench.py). */
typedef struct dfk_lm_counters {
    uint64_t n_state;   /* model+Jacobian evaluations  (fit.py:68  coeffs)  */
    uint64_t n_ssq;     /* residual-only evaluations   (fit.py:152 ssqf)    */
    uint64_t n_solve;   /* damped normal-equation solves (fit.py:169 msolve) */
    uint64_t n_grid;    /* grid-search fallbacks       (fit.py:260)         */
    uint64_t n_bessel_steps; /* Miller recurrence steps over all evaluations */
} dfk_lm_counters;

/* Settings of the log-frequency spectral estimate; defaults of DeepFitObject (data.py:150-158). */
typedef struct dfk_lpsd_opts {
    double olap;     /* overlap fraction; < 0 = "default": the window's recommended overlap (data.py:150) */
    double bmin;     /* first usable (fractional) DFT bin                                  (1)   */
    int64_t lmin;    /* shortest segment                                                   (0)   */
    int32_t jdes;    /* desired number of frequencies                                      (500) */
    int32_t kdes;    /* desired number of averages                                         (100) */
    int32_t order;   /* detrending polynomial per segment: -1 none, 0 mean, 1, 2           (0)   */
    int32_t window;  /* 0 = Kaiser (np.kaiser, data.py:156), 1 = Hann                      (0)   */
    double psll;     /* Kaiser peak side-lobe level in dB                                  (200) */
} dfk_lpsd_opts;

/* Header of a DFMSWPM raw_data text file as parse_header reads it (core.py:129-174). */
typedef struct dfk_raw_header {
    int32_t channels;     /* "Number of channels" (line 2)        */
    int32_t pad_;
    int64_t t0;           /* "Start time" (line 3)                */
    double f_samp;        /* "Sampling frequency" (line 4)        */
    double f_mod;         /* "Modulation frequency" (line 5)      */
    int64_t data_offset;  /* byte offset of the first data row: after the 13 lines read_csv(skiprows=13) skips */
} dfk_raw_header;

/* Sample types of the binary ingest path. */
#define DFK_RAW_I16 0
#define DFK_RAW_I32 1
#define DFK_RAW_F32 2
#define DFK_RAW_F64 3

typedef struct dfk_ctx dfk_ctx;

/* ---- library / context ------------------------------------------------------------------ */
int dfk_abi_version(void);
const char* dfk_last_error(void);
int dfk_device_count(void);
/* One context per (thread, device): owns its streams (compute, copy, side) and device scratch. */
int dfk_create(int device, dfk_ctx** out);
int dfk_destroy(dfk_ctx* ctx);
/* Use a caller-owned stream (e.g. torch's current stream) for the device-pointer calls;
 * NULL restores the context's own stream. */
int dfk_set_stream(dfk_ctx* ctx, void* cuda_stream);
/* on != 0: issue the device-pointer calls on the legacy default stream (handle 0, what torch uses
 * unless told otherwise); on == 0: back to the context's own stream. */
int dfk_use_legacy_default_stream(dfk_ctx* ctx, int on);
int dfk_synchronize(dfk_ctx* ctx);
void dfk_default_lm_opts(dfk_lm_opts* o);
void dfk_default_ekf_opts(dfk_ekf_opts* o);

/* ---- device-pointer kernels --------------------------------------------------------------- */
/* Harmonic lock-in of nbuf contiguous buffers of R samples.
 * Replaces calculate_quadratures (fit.py:18-66) and the three mean() loops
 * (fitters.py:45-49, 380-384, 436-440) plus dc = mean(buffer) (fitters.py:57).
 * w0 is rad/sample exactly as the reference passes it (fitters.py:39).
 * qi_dev: nbuf x 2N, dc_dev: nbuf. */
int dfk_demod(dfk_ctx* ctx, const double* x_dev, int64_t nbuf, int64_t R, int32_t N, double w0,
              double* qi_dev, double* dc_dev);

/* Batched LM fit of (amp, m, phi, psi) on nbuf harmonic vectors.
 * Replaces fit.fit (fit.py:322-362) incl. coeffs/ssqf/msolve/_run_lma_fit/_find_best_initial_guess.
 * guess_dev: 4 doubles when guess_stride == 0 (one seed for all fits, fitters.py:404-417) or
 * nbuf x guess_stride.  dc_dev may be NULL.  rows_dev: nbuf x DFK_ROW_STRIDE. */
int dfk_lm_fit(dfk_ctx* ctx, const double* qi_dev, int64_t nbuf, int32_t N, const double* guess_dev,
               int64_t guess_stride, const double* dc_dev, const dfk_lm_opts* opts, double* rows_dev);

/* Parameter covariance of nbuf fitted rows (rows_dev: nbuf x DFK_ROW_STRIDE, e.g. from dfk_lm_fit) on their harmonic
 * vectors qi_dev (nbuf x 2N, from dfk_demod): the standard NLS estimate s^2 (J^T J)^-1, J^T J of the harmonic model at
 * the row's own amp, m, phi, psi and s^2 = ssq / (2N - 4) from the row's ssq.  The reference forms the same
 * inv(J^T J) sigma^2 only at the true parameters, for its Cramer-Rao bound (helpers.py:16-45, 60-96).
 * cov_dev: nbuf x DFK_COV_STRIDE = [C_aa, C_am, C_aphi, C_mm, C_mphi, C_phiphi, C_psipsi, s^2]; the psi cross terms are
 * identically zero.  The estimate takes the residual scatter as the noise level; a caller who knows the I/Q noise
 * variance sigma^2 rescales by sigma^2 / s^2.  Every row is computed whatever its fitok; filter on fitok as for the
 * parameters.  Degenerate rows: 2N - 4 <= 0 or a non-finite parameter -> all eight NaN; a singular amp/m/phi block
 * (e.g. amp = 0) -> its six entries NaN; a vanishing psi column -> C_psipsi NaN; ssq = 0 -> zeros. */
int dfk_lm_cov(dfk_ctx* ctx, const double* qi_dev, int64_t nbuf, int32_t N, const double* rows_dev, double* cov_dev);

/* Whole NLS readout of one device-resident record: demod, fit buffer 0 from init, fit the other
 * buffers on the schedule `seeded` names (DFK_SCHED_* above).  Replaces StandardNLSFitter._fit_sequential
 * (fitters.py:370-393) and _fit_parallel with its multiprocessing.Pool (fitters.py:395-428). */
int dfk_nls_fit_dev(dfk_ctx* ctx, const double* x_dev, int64_t nbuf, int64_t R, int32_t N, double w0,
                    const double init[4], int32_t seeded, const dfk_lm_opts* opts, double* rows_dev);
/* The same, plus the covariance row of every buffer (dfk_lm_cov on the record's harmonic vectors and the final rows)
 * in cov_dev: nbuf x DFK_COV_STRIDE.  Rows are those of dfk_nls_fit_dev.  (helpers.py:16-45, 60-96) */
int dfk_nls_fit_cov_dev(dfk_ctx* ctx, const double* x_dev, int64_t nbuf, int64_t R, int32_t N, double w0,
                        const double init[4], int32_t seeded, const dfk_lm_opts* opts, double* rows_dev, double* cov_dev);

/* A slab of a record whose buffer 0 lives elsewhere (another GPU): the slab is `chunks` chunks (>= 1, or
 * DFK_SCHED_EACH) whose first buffers start from seed[4], the fitted [amp, m, phi, psi] of the record's
 * buffer 0 -- what each Pool chunk receives as seed_guess in fitters.py:407-417.  Slabs are independent:
 * no inter-GPU traffic on the kernel path. */
int dfk_nls_fit_seeded_dev(dfk_ctx* ctx, const double* x_dev, int64_t nbuf, int64_t R, int32_t N, double w0,
                           const double seed[4], int32_t chunks, const dfk_lm_opts* opts, double* rows_dev);

/* The same for C channel records at once (additive API for multi-channel batches and Monte-Carlo
 * sweeps; the reference loops dff.fit(label) per channel, core.py:279-286).  Channel c is the
 * bufs_per_channel * R samples at x_dev + c * ld_c.  Cold starts use init[4], or, when init_dev is
 * not NULL, init_dev[c * init_stride .. +3] (per-channel guesses, e.g. init_m = m_true per grid point,
 * workers.py:167-173).  seeded != 0: buffer 0 of every channel is fitted cold, its other buffers start
 * from that result.  rows_dev: C x bufs_per_channel x DFK_ROW_STRIDE. */
int dfk_nls_fit_batch_dev(dfk_ctx* ctx, const double* x_dev, int64_t C, int64_t bufs_per_channel, int64_t ld_c,
                          int64_t R, int32_t N, double w0, const double init[4], const double* init_dev,
                          int64_t init_stride, int32_t seeded, const dfk_lm_opts* opts, double* rows_dev);
/* The same with covariance rows, cov_dev: C x bufs_per_channel x DFK_COV_STRIDE (helpers.py:16-45, 60-96). */
int dfk_nls_fit_batch_cov_dev(dfk_ctx* ctx, const double* x_dev, int64_t C, int64_t bufs_per_channel, int64_t ld_c,
                              int64_t R, int32_t N, double w0, const double init[4], const double* init_dev,
                              int64_t init_stride, int32_t seeded, const dfk_lm_opts* opts, double* rows_dev, double* cov_dev);

/* The same for a TIME-MAJOR record, sample (t, c) at x_dev[t * C + c] (interleaved channels: the layout acquisition
 * hardware and the DFMSWPM text format produce), without a transposition pass: an interleaved buffer folds like one
 * channel whose period is C times as long, and the per-channel harmonics are taken from the folded sums.  Needs a
 * foldable geometry (whole even number of samples per modulation period x C, whole periods per buffer) and fails with
 * DFK_ERR_ARG otherwise -- transpose with dfk_widen_dev then.  Units are channel-major as above:
 * rows_dev / qi_dev row c * bufs_per_channel + b. */
int dfk_demod_tm_dev(dfk_ctx* ctx, const double* x_dev, int64_t bufs_per_channel, int64_t C, int64_t R, int32_t N, double w0,
                     double* qi_dev, double* dc_dev);
int dfk_nls_fit_batch_tm_dev(dfk_ctx* ctx, const double* x_dev, int64_t C, int64_t bufs_per_channel, int64_t R, int32_t N,
                             double w0, const double init[4], const double* init_dev, int64_t init_stride, int32_t seeded,
                             const dfk_lm_opts* opts, double* rows_dev);
/* The same with covariance rows, cov_dev: C x bufs_per_channel x DFK_COV_STRIDE (helpers.py:16-45, 60-96). */
int dfk_nls_fit_batch_tm_cov_dev(dfk_ctx* ctx, const double* x_dev, int64_t C, int64_t bufs_per_channel, int64_t R, int32_t N,
                                 double w0, const double init[4], const double* init_dev, int64_t init_stride, int32_t seeded,
                                 const dfk_lm_opts* opts, double* rows_dev, double* cov_dev);

/* 5-state EKF over C independent channels, one thread per channel.
 * Replaces EKFFitter.fit (fitters.py:214-320).  Sample (t, c) is z_dev[t*ld_t + c*ld_c]
 * (time-major: ld_t = C, ld_c = 1; channel-major: ld_t = 1, ld_c = T).
 * rows_dev: C x nbuf x DFK_ROW_STRIDE with nbuf = T / R. */
int dfk_ekf_dev(dfk_ctx* ctx, const double* z_dev, int64_t T, int64_t C, int64_t ld_t, int64_t ld_c,
                int64_t R, double f_samp, double f_mod, const dfk_ekf_opts* opts, double* rows_dev);

/* The same filter fed slab by slab, for records that do not fit the GPU (cfg 4: 655 GB): samples
 * k0 .. k0+T-1 of every channel per call, k0 and T multiples of R.  state_dev (C x 32 doubles: x[5],
 * the upper triangle of P [15], r at index 30) carries the filter between calls; the call with k0 == 0
 * initialises it.  Initial dc and the default measurement variance are those of opts (init_dc, r_val);
 * where opts leaves them NaN they come from this first slab instead of the whole record -- the one
 * place the slab-wise result can depart from EKFFitter.fit on the full record (dfk_ekf_host computes the
 * whole-record moments in a first pass instead).
 * rows_dev: C x (T/R) x DFK_ROW_STRIDE for this slab. */
int dfk_ekf_stream_dev(dfk_ctx* ctx, const double* z_dev, int64_t T, int64_t C, int64_t ld_t, int64_t ld_c,
                       int64_t R, double f_samp, double f_mod, const dfk_ekf_opts* opts, int64_t k0,
                       double* state_dev, double* rows_dev);

/* 'snr'-mode synthetic record (physics.py:475-530) generated on the device with a counter-based
 * RNG: y = A(1 + C cos(phi0 + m cos(2 pi f_mod t + psi0))) + sigma N(0,1), sigma from snr_db.
 * Statistically (not bitwise) equivalent to the reference's MT19937 stream.  C channels,
 * channel-major [C][T]; channel c uses phi0 + c*dphi and seed + c. */
int dfk_synth_snr_dev(dfk_ctx* ctx, double* x_dev, int64_t T, int64_t C, double f_samp, double f_mod,
                      double m, double amp, double visibility, double phi0, double dphi, double psi0,
                      double snr_db, uint64_t seed);

/* Samples t0 .. t0+T-1 of the same streams, channel c written at x_dev + c * ld_c: any slab of a long
 * record can be produced on its own, on any GPU. */
int dfk_synth_snr_slab_dev(dfk_ctx* ctx, double* x_dev, int64_t T, int64_t C, int64_t ld_c, int64_t t0, double f_samp,
                           double f_mod, double m, double amp, double visibility, double phi0, double dphi,
                           double psi0, double snr_db, uint64_t seed);

/* Monte-Carlo sweep without records: realisations c0 .. c0+nbuf-1 of one grid point -- single 'snr'-mode records of R
 * samples, noise keyed by seed + index exactly as dfk_synth_snr_slab_dev keys channels -- are generated inside the
 * demodulation kernel's shared memory and reduced to their harmonic vectors qi_dev[nbuf x 2N] and means dc_dev[nbuf]
 * (run_efficiency_trial's simulate step, workers.py:132-189, fused with calculate_quadratures).  Bit-identical to
 * dfk_synth_snr_slab_dev followed by dfk_demod.  One period per record (R = f_samp / f_mod, a multiple of 4, <= 256)
 * takes the fused kernel; any other geometry generates into scratch and demodulates from there. */
int dfk_sweep_demod_dev(dfk_ctx* ctx, int64_t nbuf, int64_t c0, int64_t R, int32_t N, double f_samp, double f_mod, double m,
                        double amp, double visibility, double phi0, double psi0, double snr_db, uint64_t seed,
                        double* qi_dev, double* dc_dev);
/* The whole study of notebook 1.1_CRLB-test / BASELINE config 5 in one call: for every m_values[i] (host array),
 * ntrials realisations (indices trial0 .. trial0+ntrials-1, noise key seed + i * seed_stride + index) generated,
 * demodulated and fitted cold from [init_a, init_m, 0, 0] -- init_m = NaN starts every fit at its true m
 * (workers.py:167-173).  rows_dev: nm x ntrials x DFK_ROW_STRIDE. */
int dfk_nls_sweep_dev(dfk_ctx* ctx, const double* m_values, int32_t nm, int64_t ntrials, int64_t trial0, int64_t seed_stride,
                      int64_t R, int32_t N, double f_samp, double f_mod, double amp, double visibility, double phi0,
                      double psi0, double snr_db, uint64_t seed, double init_a, double init_m, const dfk_lm_opts* opts,
                      double* rows_dev);
/* The same with covariance rows, cov_dev: nm x ntrials x DFK_COV_STRIDE -- the notebook's inv(J^T J) sigma^2 of
 * helpers.py:16-45, 60-96 at every fitted realisation instead of at the truth only. */
int dfk_nls_sweep_cov_dev(dfk_ctx* ctx, const double* m_values, int32_t nm, int64_t ntrials, int64_t trial0,
                          int64_t seed_stride, int64_t R, int32_t N, double f_samp, double f_mod, double amp, double visibility,
                          double phi0, double psi0, double snr_db, uint64_t seed, double init_a, double init_m,
                          const dfk_lm_opts* opts, double* rows_dev, double* cov_dev);

/* ---- host-pointer entry points (what the reference-side shim binds) ---------------------- */
/* StandardNLSFitter.fit on one host record (fitters.py:330-428): nsamp samples, buffers of R,
 * slabs streamed host->device on a copy stream while the previous slab is demodulated and
 * fitted.  rows_host: (nsamp / R) x DFK_ROW_STRIDE. */
int dfk_nls_fit_host(dfk_ctx* ctx, const double* x_host, int64_t nsamp, int64_t R, int32_t N, double w0,
                     const double init[4], int32_t seeded, const dfk_lm_opts* opts, double* rows_host);
/* The same with covariance rows, cov_host: (nsamp / R) x DFK_COV_STRIDE.  Each slab's covariance comes from that slab's
 * harmonic vectors after its last LM launch; one more copy back beside the rows' (helpers.py:16-45, 60-96). */
int dfk_nls_fit_cov_host(dfk_ctx* ctx, const double* x_host, int64_t nsamp, int64_t R, int32_t N, double w0,
                         const double init[4], int32_t seeded, const dfk_lm_opts* opts, double* rows_host, double* cov_host);

/* dfk_nls_fit_seeded_dev for a host slab (same streaming as dfk_nls_fit_host): what each rank of a record sharded
 * over several GPUs calls on its own slab once buffer 0's result is known. */
int dfk_nls_fit_seeded_host(dfk_ctx* ctx, const double* x_host, int64_t nsamp, int64_t R, int32_t N, double w0,
                            const double seed[4], int32_t chunks, const dfk_lm_opts* opts, double* rows_host);

/* EKFFitter.fit on host records, channel-major [C][T]. rows_host: C x (T/R) x DFK_ROW_STRIDE.
 * A record larger than the device is streamed in slabs of whole buffers (twice when the whole-record
 * mean / variance are needed first), the filter state carried on the device from slab to slab. */
int dfk_ekf_host(dfk_ctx* ctx, const double* z_host, int64_t T, int64_t C, int64_t R, double f_samp,
                 double f_mod, const dfk_ekf_opts* opts, double* rows_host);

/* Slab size of the two host-pointer entries above (0 restores the defaults: 128 MiB NLS slabs, half the free
 * device memory for the EKF).  Lets a small record exercise the streaming path. */
int dfk_set_host_slab_bytes(dfk_ctx* ctx, int64_t bytes);

/* ---- raw-data ingest (SURVEY 8f-2) ------------------------------------------------------------- */
/* parse_header(file_select='raw') (core.py:129-174): of header lines 2..5 only the characters "0-9." are kept
 * and read as int, int, float, float (an exponent or a sign is therefore dropped, as in the reference); fails where
 * Python's int()/float() would raise.  Host only -- no GPU needed. */
int dfk_raw_parse_header(const char* path, dfk_raw_header* out);

/* load_raw (core.py:259-286) is pd.read_csv(raw_file, sep=' ', skiprows=13, usecols=[c], names=['ch<c>']) per
 * channel.  Here the data region of the file goes to the device once (file -> pinned staging buffers -> HBM, reads and
 * DMA overlapped) and is parsed there: dfk_text_load_* uploads the bytes, finds the rows (lines holding only blanks
 * are skipped) and reports their number, so that the caller can allocate the record; dfk_text_parse_dev converts
 * the wanted columns into out_dev (column c, row r at out_dev[c * ld_c + r]).  usecols: ascending file columns, or
 * NULL for 0..ncols-1.  Fields are converted exactly as the reference's pandas call converts them (pandas' C-parser
 * default, precise_xstrtod: 17 significant digits, one scaling by a power of ten -- not correctly rounded, and
 * reproduced bit for bit).  A missing or non-numeric field becomes NaN and is counted in *nbad_out.
 * The text stays resident (for further dfk_text_parse_dev calls) until the next load or dfk_text_release. */
int dfk_text_load_file(dfk_ctx* ctx, const char* path, int64_t byte_offset, int64_t* nbytes_out, int64_t* nrows_out);
int dfk_text_load_host(dfk_ctx* ctx, const char* text_host, int64_t nbytes, int64_t* nrows_out);
int dfk_text_parse_dev(dfk_ctx* ctx, int32_t ncols, const int32_t* usecols, double* out_dev, int64_t ld_c,
                       int64_t* nbad_out);
int dfk_text_release(dfk_ctx* ctx);

/* Binary fast path (additive: the reference reads text only): samples of type dtype (DFK_RAW_*), time-major
 * interleaved (sample (t, c) at t * C + c, what acquisition hardware writes) or channel-major (c * T + t), widened
 * to the fp64 channel-major record out_dev[c * ld_c + t] = scale * sample + offset.  The host and file entries
 * stream the source in slabs through the pinned staging buffers, copies overlapping the widening kernel; a 16-bit
 * record crosses PCIe at a quarter of the fp64 bytes. */
int dfk_widen_dev(dfk_ctx* ctx, const void* src_dev, int32_t dtype, int64_t T, int64_t C, int32_t time_major,
                  double scale, double offset, double* out_dev, int64_t ld_c);
int dfk_ingest_binary_host(dfk_ctx* ctx, const void* src_host, int32_t dtype, int64_t T, int64_t C, int32_t time_major,
                           double scale, double offset, double* out_dev, int64_t ld_c);
int dfk_ingest_binary_file(dfk_ctx* ctx, const char* path, int64_t byte_offset, int32_t dtype, int64_t T, int64_t C,
                           int32_t time_major, double scale, double offset, double* out_dev, int64_t ld_c);

/* ---- batched experiments (SURVEY 8f-3) ------------------------------------------------------------- */
/* One Monte-Carlo trial of the 'asd'-mode physics (physics.py:615-722), DFK_ASD_TRIAL_DOUBLES doubles:
 *   [0] amp  [1] visibility  [2] df  [3] 2 pi f_mod  [4] psi  [5] 2 pi c / wavelength  [6] ref_arml / c
 *   [7] meas_arml / c  [8] phi wavelength / (2 pi)  [9] arml_mod_amp  [10] 2 pi arml_mod_f  [11] arml_mod_psi
 *   [12] amp_n sqrt(fs/2)  [13] df_n sqrt(fs/2)  [14] noise key (the trial number)  [15] number of waveform terms
 *   (0: the waveform is row [16] of the tables)  [17 + 3k ..] harmonic h_k, amplitude a_k, phase p_k of term k < 6:
 *   g(theta) = sum_k a_k cos(h_k theta + p_k), normalised to max |g| = 1 over the trial.
 *   [35] != 0: the channel is dynamic (the main channel; a witness is static, physics.py:460)
 *   [36] row of the external noise series this trial reads (dfk_synth_asd_noise_dev), or < 0 for internal noise. */
#define DFK_ASD_TRIAL_DOUBLES 37
#define DFK_TRIAL_STATS_DOUBLES 6
/* The reference simulates every trial of an Experiment on its own (experiments.py:15-88 -> SignalGenerator.generate,
 * mode 'asd'); here all trials of a batch are produced at once, N samples each: y_dev[j * ld + i].  tables_dev:
 * ntables x N samples of host-evaluated waveforms for trials whose waveform is not a harmonic series.
 * truth_dev (may be NULL) receives the ground-truth interferometric phase (raw.phi_sim).  White amplitude and
 * modulation-depth noise only; statistically, not bitwise, the reference's MT19937 draws. */
int dfk_synth_asd_dev(dfk_ctx* ctx, const double* trials_dev, int64_t ntrials, int64_t N, double f_samp,
                      const double* tables_dev, int64_t ntables, double* y_dev, int64_t ld, double* truth_dev);
/* The same with pre-computed noise series, the engine's external_noise input (SignalGenerator.generate, physics.py:
 * 380-434; _run_simulation_physics :672-710): noise_dev[4] holds device pointers to noise_rows x N series -- laser
 * frequency [Hz], amplitude, modulation amplitude df [Hz], arm length [m] -- any of which may be NULL (taken as zero).
 * A trial whose record names a row ([36] >= 0) reads that row of each series INSTEAD of drawing white noise; the
 * arm-length series only if the trial is dynamic ([35]).  This is how coloured laser-frequency and arm-length noise,
 * which the reference takes from a third-party generator, enter: main and witness channel of a pair name the same row. */
#define DFK_NOISE_LASER_FREQUENCY 0
#define DFK_NOISE_AMPLITUDE 1
#define DFK_NOISE_DF 2
#define DFK_NOISE_ARMLENGTH 3
int dfk_synth_asd_noise_dev(dfk_ctx* ctx, const double* trials_dev, int64_t ntrials, int64_t N, double f_samp,
                            const double* tables_dev, int64_t ntables, const double* const* noise_dev, int64_t noise_rows,
                            double* y_dev, int64_t ld, double* truth_dev);
/* Per grid point and result column: nanmean, nanstd, nanmin, nanmax, "worst" (the trial farthest from the mean)
 * and the number of finite trials -- the aggregation at the end of Experiment.run (experiments.py:432-446).
 * values_dev[(p * ntrials + t) * col_stride + c]; out_dev[(p * ncols + c) * 6 + {0..5}].  center_dev (npoints x
 * ncols, may be NULL): measure "worst" from these values -- e.g. the true parameters -- instead of the mean.
 * ncols <= 8. */
int dfk_trial_stats_dev(dfk_ctx* ctx, const double* values_dev, int64_t npoints, int64_t ntrials, int32_t ncols,
                        int64_t col_stride, const double* center_dev, double* out_dev);

/* ---- post-fit step (SURVEY 8f-4) -------------------------------------------------------------- */
/* Block means: out[b] = mean(x[b*R .. b*R+R-1]), b < n / R; a tail shorter than R is dropped.
 * Replaces vectorized_downsample (dsp.py:3-56), the boxcar that brings the simulated ground-truth phase to the
 * fit rate.  The host entry streams the record in slabs like dfk_nls_fit_host. */
int dfk_downsample_dev(dfk_ctx* ctx, const double* x_dev, int64_t n, int64_t R, double* out_dev);
int dfk_downsample_host(dfk_ctx* ctx, const double* x_host, int64_t n, int64_t R, double* out_host);

void dfk_default_lpsd_opts(dfk_lpsd_opts* o);
/* The frequency plan of the estimate for a series of N samples at rate fs: frequencies f, resolutions r,
 * fractional bins m, segment lengths L, averages K (the LTPDA ltf_plan scheduler).  *nf receives the number of
 * frequencies; at most cap entries are written to each non-NULL array. */
int dfk_lpsd_plan(int64_t N, double fs, const dfk_lpsd_opts* opts, int32_t cap, int32_t* nf, double* f, double* r,
                  double* m, int64_t* L, int64_t* K);
/* Log-frequency power spectrum / spectral density of C device-resident series (Troebs & Heinzel 2006).
 * Replaces the spectools.lpsd call of calc_lpsd (core.py:590-609, data.py:239-244) on fit.phi.  Sample i of series c
 * is x_dev[c * ld_c + i * stride] -- stride = DFK_ROW_STRIDE reads a column of a row table in place.
 * Host outputs: f_host[nf], ps_host / psd_host [C x nf] (power spectrum; one-sided density, the reference's Sxx),
 * enbw_host[nf], navs_host[nf]; any may be NULL.  Fails if the plan needs more than cap frequencies. */
int dfk_lpsd_dev(dfk_ctx* ctx, const double* x_dev, int64_t N, int64_t stride, int64_t C, int64_t ld_c, double fs,
                 const dfk_lpsd_opts* opts, int32_t cap, int32_t* nf_out, double* f_host, double* ps_host,
                 double* psd_host, double* enbw_host, int64_t* navs_host);
/* Log-frequency cross-spectral density of Cx device-resident series x against Cy series y on the plan of
 * dfk_lpsd_plan with the same options (the LTPDA log-frequency CSD, Troebs & Heinzel 2006): same frequencies, segments,
 * detrending and window as dfk_lpsd_dev.  Sample i of series a of x is x_dev[a * ldx + i * stride], likewise for y;
 * stride = DFK_ROW_STRIDE reads a column of a row table in place.  Every series has N samples; Cx, Cy >= 1 and
 * Cx + Cy <= 65535.
 * For frequency row j (K_j segments, window w, S2_j = sum w^2) and segment s of series u let
 * A_{u,s} = sum_n w_n v_n e^{+i p_j n}, v the detrended segment: the complex conjugate of the usual DFT X.  Then
 *     Sxy[a,b,j] = 2 / (fs S2_j) * (1 / K_j) * sum_s A_{x_a,s} conj(A_{y_b,s})
 * is the one-sided CSD in scipy's convention, E[conj(X) Y]; Sxx, Syy are the same sum on one series, i.e. the psd of
 * dfk_lpsd_dev (equal up to the order of the segment sum).  If y(t) = x(t - tau), arg Sxy = -2 pi f tau.
 * Host outputs: f_host[nf], sxx_host [Cx x nf], syy_host [Cy x nf], sxy_host [Cx x Cy x nf x 2] (re, im interleaved),
 * enbw_host[nf], navs_host[nf] (K_j); any may be NULL.  Coherence |Sxy|^2 / (Sxx Syy) is identically 1 where K_j = 1.
 * Fails if the plan needs more than cap frequencies.  Two kernel launches; synchronises like dfk_lpsd_dev. */
int dfk_lcsd_dev(dfk_ctx* ctx, const double* x_dev, int64_t Cx, int64_t ldx, const double* y_dev, int64_t Cy, int64_t ldy,
                 int64_t N, int64_t stride, double fs, const dfk_lpsd_opts* opts, int32_t cap, int32_t* nf_out,
                 double* f_host, double* sxx_host, double* syy_host, double* sxy_host, double* enbw_host,
                 int64_t* navs_host);

/* ---- introspection ------------------------------------------------------------------------ */
/* Counters accumulated by the LM kernels since the last reset (device -> host copy, syncs). */
int dfk_lm_counters_read(dfk_ctx* ctx, dfk_lm_counters* out, int32_t reset);
/* Device-time accounting per kernel class for the roofline report: with profiling on, the entry
 * points record CUDA event pairs on the launching stream around the demodulation launch (index 0),
 * around the LM launches (index 1), on the side stream around the cold seed fits that overlap the
 * demodulation (index 2), and around the EKF kernel (index 3).  dfk_profile_read synchronises and
 * returns the summed milliseconds and the number of timed regions of each class. */
int dfk_profile_enable(dfk_ctx* ctx, int32_t on);
int dfk_profile_read(dfk_ctx* ctx, double ms_total[DFK_PROFILE_KINDS], int64_t launches[DFK_PROFILE_KINDS],
                     int32_t reset);
/* Measured fp64 FMA throughput of the device in TFLOP/s (8 independent DFMA chains per thread, best of 3):
 * the denominator for the LM kernel's fraction of the FP64 roofline. */
int dfk_probe_fp64(dfk_ctx* ctx, double* tflops_out);
/* Development overrides of kernel choice and geometry for tuning runs and kernel A/B tests, e.g.
 * dfk_dev_set("DFK_NO_TILE", 1) (names: csrc/dfk_b200.cu).  Process-wide, set only by these calls -- the library
 * never reads the environment.  dfk_dev_clear() drops them all. */
int dfk_dev_set(const char* name, int32_t value);
void dfk_dev_clear(void);
/* Kernel launches issued through this context since creation (bench.py's gpu_launches). */
int64_t dfk_launch_count(dfk_ctx* ctx);
/* Which demod path the given geometry selects: 1 = a folded TMA kernel (fold / tile / single-period),
 * 0 = the direct kernel (incommensurate period or a buffer that is not a whole number of fold lengths). */
int dfk_demod_path(int64_t R, double w0);
/* Bessel J_0..J_nmax(x) by the device's Miller recurrence, evaluated on the device (testing). */
int dfk_bessel_dev(dfk_ctx* ctx, const double* x_dev, int64_t n, int32_t nmax, double* out_dev);

#ifdef __cplusplus
}
#endif
#endif /* DFK_B200_H */
