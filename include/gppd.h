/*
 * gppd.h -- C ABI of libgppd.so: the B200 (sm_100a) implementation of
 * GPPupilDemodulation.jl's `demodulateall` hot path.
 *
 * The reference has no native interface for this path (it is plain Julia); its
 * only FFI idiom is `ccall(...)::Cint` + `fits_assert_ok(status)`
 * (reference src/FitsUtils.jl:42-58).  This header follows that idiom: every
 * entry point returns an int status (0 = OK), takes plain pointers and sizes,
 * never keeps a caller pointer after it returns, and never throws.  The Julia
 * side binds it with `ccall` (see INTEGRATION.md and julia/GPPDB200.jl).
 *
 * Layout conventions (all little-endian host order unless stated):
 *   complex128 = two consecutive doubles (re, im) == Julia ComplexF64
 *   data / out of the *_f64 calls: N x 40 column-major == Julia
 *       Matrix{ComplexF64}(N, 40): channel c (0-based) starts at 2*N*c doubles
 *   VOLT of the *_f32 calls: 80 x N column-major in Julia == N rows of 80
 *       floats in memory; channel c = (VOLT[2c], VOLT[2c+1]) of each row
 *       (reference src/GPPupilDemodulation.jl:148)
 *   params: 6 doubles per fitted diode (c.re, c.im, a.re, a.im, b, phi), diode
 *       order = channel order 0..31 (reference idx(), src/Modulation.jl:17-22)
 *   state: int8 MetState values OFF=0 LOW=1 NORMAL=2 HIGH=3 TRANSIENT=-1
 *       (reference src/Faint.jl:1)
 */
#ifndef GPPD_H
#define GPPD_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GPPD_VERSION 122 /* 0.1.22: + GPPD_COVARIANCE / gppd_covariances, GPPD_FP32, GPPD_CENTER_ELLIPSE / gppd_ellipses; 0.1.21: + gppd_file_* (native ingest); 0.1.20: gppd_options.group_mask, gppd_demodulate_f64_dev (0.1.10: gppd_submit_fits_rows,
                            gppd_centres, gppd_set_split_chains, gppd_debug_harmonics, GPPD_CENTER_EMPIRICAL) */

/* ---- status codes ------------------------------------------------------ */
#define GPPD_OK 0
#define GPPD_ERR_ARG 1        /* bad argument (NULL, n < 2, ...) */
#define GPPD_ERR_CUDA 2       /* a CUDA call failed; see gppd_last_error() */
#define GPPD_ERR_NO_DEVICE 3  /* no usable sm_100 device: there is no CPU fallback */
#define GPPD_ERR_NOMEM 4
#define GPPD_ERR_UNSUPPORTED 5
#define GPPD_ERR_IO 6          /* file could not be read / written; see gppd_last_error() */

/* ---- option flags ------------------------------------------------------ */
#define GPPD_ONLYHIGH 1u    /* demodulateall(onlyhigh=true)   src/Modulation.jl:348 */
#define GPPD_FITOFFSETS 2u  /* demodulateall(fitoffsets=true) src/Modulation.jl:349 */
#define GPPD_NO_RECENTER 4u /* demodulateall(recenter=false)  src/Modulation.jl:346 */
#define GPPD_KEEPRAW 8u     /* processmetrology(keepraw=true) src/GPPupilDemodulation.jl:163 */
#define GPPD_BIG_ENDIAN 16u /* table buffers are raw FITS (big-endian) bytes */
#define GPPD_CENTER_EMPIRICAL 32u /* processmetrology(offsets=true), `--center empirical`:
                               the centres are fitted here, one algebraic least-squares
                               circle per channel over the table's samples (the HIGH
                               samples of a FAINT table), compute_offsets,
                               src/GPPupilDemodulation.jl:105-125,153-154.  Table entry
                               points only; their `offsets` argument is then ignored and
                               GPPD_FITOFFSETS is off.  (The reference itself throws on
                               this path: its `Circle` type is undefined.) */
#define GPPD_CENTER_ELLIPSE 0x80u /* (= 128) `--center ellipse`: offset AND ellipse
                               (Heydemann) correction of each of the 40 channels, for quadrature detectors whose two outputs
                               differ in gain (ratio r) or are not exactly in quadrature (error
                               alpha).  Per channel, over the samples compute_offsets uses (all
                               rows, or the HIGH rows of a FAINT table): the algebraic
                               least-squares conic A u^2 + B uv + C v^2 + D u + E v + F = 0 with
                               A + C = 1 (solved on samples shifted to their centroid and scaled
                               to unit rms radius); centre [2A B; B 2C] (x0, y0) = -(D, E),
                               r = sqrt(C/A), alpha = asin(B / (2 sqrt(AC))), i.e. the forward
                               model x = x0 + U1, y = y0 + (U2 cos alpha - U1 sin alpha) / r.
                               Every row, in every state, is then corrected in float64 with
                               every operation rounded (no FMA):
                                   m21 = tan alpha, m22 = r / cos alpha
                                   x' = x - x0,  y' = m21 x' + m22 (y - y0)
                               (the x-axis scale is kept: |a| stays in volts of the x output),
                               and the corrected channels replace the centred ones everywhere
                               downstream (NoOffsets fit, FC phasor, FAINT statistics, output
                               VOLT including the FC columns; keepraw: columns 1..80 stay raw).
                               A channel falls back to the empirical circle centre and the
                               identity shape (status 1) when it has fewer than 5 samples, the
                               Cholesky factorisation of the 5x5 normal matrix meets a pivot
                               <= 1e-12 of its diagonal entry, A <= 0 or C <= 0, or the axis
                               ratio exceeds 10 (4AC - B^2 <= 4 * 0.01 / 1.01^2); with no circle
                               either, to centre 0 and the identity (status 0).  Table entry
                               points only (gppd_demodulate_f64* return GPPD_ERR_UNSUPPORTED);
                               their `offsets` argument is ignored; with GPPD_FITOFFSETS or
                               GPPD_CENTER_EMPIRICAL the call fails with GPPD_ERR_ARG.
                               GPPD_FP32 has no effect in this mode (the array path the
                               corrected channels take has no FP32 form).  gppd_ellipses
                               returns the fitted maps. */

#define GPPD_FP32 64u /* OPTIONAL reduced precision, off by default: the harmonic sums of the fit are
                         formed from float32 stream values and harmonics rounded to 23-bit fixed
                         point (harm_tc32_kernels.cu) instead of 48-bit.  Times, phases, the
                         optimiser and the demodulation stay FP64; fitted parameters agree with the
                         FP64 path to ~1e-6 (bound tested: 1e-5, BASELINE north_star "optional FP32
                         path").  Applies where the tensor-core harmonic kernel does (dense
                         METROLOGY-table entry points, harmonic evaluator); ignored elsewhere. */

#define GPPD_COVARIANCE 0x100u /* (= 256) the statistical uncertainty of every fit: after the
                               fit, one extra streaming pass (csrc/cov_kernels.cu, FP64 whatever
                               GPPD_FP32 says) forms the Gauss-Newton covariance of the REPORTED
                               parameters at the reported values; gppd_covariances returns it.
                               Nothing else a call returns changes.  Definition, per fit:
                                 model  m_n = c + a p_n exp(j b s_n),  p_n = power_state FCphasor_n,
                                        s_n = sin(fl(fl(omega t_n) + phi)), cs_n = cos of the same
                                        rounded argument, weight w_n (1 in bright mode); n runs over
                                        the job's valid rows (onlyhigh, TRANSIENT), N_valid of them
                                 theta  = (c.re, c.im, a.re, a.im, b, phi) in params order; without
                                        GPPD_FITOFFSETS the model has no c: k = 4 and rows / columns
                                        0-1 of the result are 0 (k = 6 otherwise)
                                 J_n    = dm/dtheta = (1, j, g, j g, j a s g, j a b cs g),
                                        g = p e^{j b s}
                                 H      = Re sum w conj(J_n) J_n^T  (k x k)
                                 s^2    = sum w |m_n - d_n|^2 / (2 N_valid - k)
                                 cov    = s^2 H^-1
                               evaluated at the exported (b, phi) (after the sign normalisation
                               b < 0 -> -b, phi +- pi), so that entries pairing b with another
                               parameter have the sign of the reported parametrisation.  All 36
                               entries of a fit are NaN when 2 N_valid <= k, when the Cholesky
                               factorisation of the diagonally scaled H meets a pivot <= 1e-12,
                               when the fit's group is outside group_mask, or when the fit itself
                               has a NaN.  In ellipse mode it is the covariance of the fit to the
                               corrected channels (the maps are treated as exact).  With this flag
                               a batch of the table entry points runs as one launch sequence
                               (gppd_set_split_chains has no effect), so that every fit's result
                               is on the slot gppd_covariances reads. */
#define GPPD_COV_STRIDE 36    /* doubles per fit: a 6 x 6 matrix, row-major */

/* which evaluator computes chi2(b, phi) inside the fit */
#define GPPD_METHOD_AUTO 0     /* harmonic when its validity conditions hold, else direct */
#define GPPD_METHOD_DIRECT 1   /* O(N) pass per objective call (the reference's formulation) */
#define GPPD_METHOD_HARMONIC 2 /* Jacobi-Anger sums once, O(K) per objective call */

typedef struct gppd_handle_s *gppd_handle;

typedef struct gppd_options {
    uint32_t flags;     /* GPPD_* bits */
    int32_t method;     /* GPPD_METHOD_* */
    int32_t maxfun;     /* NEWUOA objective-call cap; 0 => 60 (30n, OptimPackNextGen default) */
    int32_t has_xinit;  /* 0: init=:auto (8-point phase scan), 1: use xinit */
    double xinit[2];    /* demodulateall(init=[b, phi])       src/Modulation.jl:345,362 */
    double rhobeg;      /* 0 => 1.0   (src/Modulation.jl:335) */
    double rhoend;      /* 0 => 1e-3  (src/Modulation.jl:335) */
    uint32_t group_mask; /* which of the 8 (telescope, side) groups of src/Modulation.jl:387 to
                            process: bit g = group g = diode channels 4g..4g+3 + FC channel 32+g
                            (g = 0..3: FT T1..T4, 4..7: SC T1..T4); 0 => all 8.  The groups are
                            independent (:387-390), so one demodulateall call can be split over
                            GPUs by groups with no exchange: a call with a partial mask reads
                            and writes only the columns of its groups (the others' output
                            columns, params, chi2 and info entries are left untouched).
                            gppd_demodulate_f64 / gppd_demodulate_f64_dev only; the table
                            entry points return GPPD_ERR_UNSUPPORTED for a partial mask.
                            A call with 5 or more groups forms the harmonic sums on the int8
                            tensor cores, one with fewer on the per-group FP64 kernel (less
                            work); the two agree to 2e-14, so sharded and unsharded calls give
                            the same bits when made with the same kernel (environment
                            GPPD_TENSOR_MIN_GROUPS = 1 or 9) and the same fits up to NEWUOA's
                            rounding-level ties otherwise (DESIGN.md sections 2 and 6). */
    uint32_t reserved;  /* 0 */
} gppd_options;

/* per-fit diagnostics (optional output, 4 int32 per diode) */
#define GPPD_INFO_STRIDE 4 /* [0]=objective calls, [1]=NEWUOA status of the last
                              run, [2]=evaluator used (GPPD_METHOD_*), [3]=second
                              NEWUOA run taken (the "bad minima" retry, :411) */

/* optional trace of every objective call of every fit: GPPD_TRACE_MAX entries
 * of (b, phi, chi2) per diode, in call order; entry count = info[0] */
#define GPPD_TRACE_MAX 160

/* ---- library / handle -------------------------------------------------- */
int gppd_version(void);
const char *gppd_strerror(int status);
/* message of the last failure on this thread (CUDA error string etc.) */
const char *gppd_last_error(void);

/* Opens CUDA device `device`, creates the handle's streams and scratch.
 * Fails with GPPD_ERR_NO_DEVICE when no sm_100 GPU is present. */
int gppd_create(int device, gppd_handle *out);
int gppd_destroy(gppd_handle h);

/* Page-locked host buffers for the ingest layer (FitsUtils reads table
 * columns straight into these so that uploads run at PCIe rate). */
int gppd_alloc_pinned(gppd_handle h, uint64_t bytes, void **out);
int gppd_free_pinned(gppd_handle h, void *p);

/* ---- small host-side helpers (no GPU work) ------------------------------ */
/* reference idx(), src/Modulation.jl:17-22: side 0=FT 16=SC, telescope 1..4,
 * diode 1..4 or 5=FC; returns the 1-based channel number, or -1 */
int gppd_idx(int side, int telescope, int diode);
/* the phase-scan grid range(-pi, pi, 8), src/Modulation.jl:360 */
int gppd_phirange(double *phi8);

/* ---- buildstates, src/Faint.jl:21-73 ----------------------------------- */
/* timer1 = HIGH series, timer2 = LOW series (the FaintStates constructor swap,
 * src/Faint.jl:12-19, is done by the caller). */
int gppd_buildstates(gppd_handle h, int64_t n, const double *t,
                     const double *timer1, int64_t n1, const double *timer2,
                     int64_t n2, int64_t lag, double preswitchdelay,
                     double postswitchdelay, int8_t *state_out);

/* ---- demodulateall, src/Modulation.jl:344-435 --------------------------- */
/*
 * One call = `nwin` independent demodulateall calls over consecutive row
 * windows of `nwindow` rows (the loop of src/GPPupilDemodulation.jl:204-225);
 * nwindow <= 0 or >= n means one call over all n rows.
 *   t      [n]            seconds (absolute, as the reference passes them)
 *   data   [n x 40]       complex128, column-major
 *   state  [n] or NULL    faintparam = Vector{MetState} / nothing
 *   out    [n x 40]       complex128, column-major (columns 32..39 = input)
 *   params [nwin x 32 x 6], chi2 [nwin x 32]
 *   info   [nwin x 32 x GPPD_INFO_STRIDE] or NULL
 *   trace  [nwin x 32 x GPPD_TRACE_MAX x 3] or NULL
 * nwin = ceil(n / nwindow); gppd_num_windows() computes it.
 */
int64_t gppd_num_windows(int64_t n, int64_t nwindow);
int gppd_demodulate_f64(gppd_handle h, int64_t n, int64_t nwindow, const double *t,
                        const double *data, const int8_t *state,
                        const gppd_options *opt, double *out, double *params,
                        double *chi2, int32_t *info, double *trace);

/*
 * Device-resident variant: t, data, state, out, params, chi2, info are DEVICE pointers on
 * the handle's GPU (same layouts as above; info may be NULL), `stream` a cudaStream_t
 * passed as void* (NULL = the slot's own stream).  No host<->device copies and no
 * synchronisation: the caller orders and synchronises the stream.  This is the entry
 * point for exposures too long to stage through host memory (1e8 rows = 64 GB of
 * complex128 per direction) and for sharding one call over GPUs with
 * gppd_options.group_mask.  Scratch comes from pipeline slot `slot`.
 */
int gppd_demodulate_f64_dev(gppd_handle h, int slot, void *stream, int64_t n, int64_t nwindow,
                            const double *d_t, const double *d_data, const int8_t *d_state,
                            const gppd_options *opt, double *d_out, double *d_params,
                            double *d_chi2, int32_t *d_info);

/* ---- processmetrology on arrays, src/GPPupilDemodulation.jl:128-255 ----- */
/*
 * Table-level fast path: everything between reading the METROLOGY columns and
 * writing them back, on the device.
 *   time_us [n] int32, mjd               TIME column and MJD-OBS          (:139)
 *   volt    [n x 80] float32             VOLT column                       (:147)
 *   offsets [40] complex128 or NULL      centres to subtract; NULL => fit  (:150-157)
 *   timer1/timer2                        FAINT timers (n1 = 0 => bright)   (:141-145)
 *   window_s                             --window seconds; <= 0 => whole   (:192)
 *   volt_out [n x 80] (or n x 144 with GPPD_KEEPRAW) float32               (:163-171,253)
 *   params/chi2/info as above with nwin = *nwin_out windows; the caller sizes
 *   them with gppd_table_windows()
 *   state_out [n] int8 or NULL           STATE column                      (:248)
 */
int gppd_table_windows(int64_t n, const int32_t *time_us, double mjd,
                       double window_s, int64_t *nwindow_rows, int64_t *nwin);
int gppd_process_table_f32(gppd_handle h, int64_t n, const int32_t *time_us,
                           double mjd, const float *volt, const double *offsets,
                           const double *timer1, int64_t n1, const double *timer2,
                           int64_t n2, double window_s, const gppd_options *opt,
                           float *volt_out, double *params, double *chi2,
                           int32_t *info, int8_t *state_out);

/*
 * Asynchronous variant for pipelines over many files: the call enqueues the
 * upload, the kernels and the download on pipeline slot `slot`
 * (0 <= slot < gppd_num_slots()) and returns; gppd_wait(h, slot) blocks until
 * that slot's results are in the caller's buffers.  Buffers must stay valid
 * until then.  Uploads are truly asynchronous only from pinned memory
 * (gppd_alloc_pinned); pageable memory works but serialises.
 */
int gppd_num_slots(gppd_handle h);
int gppd_submit_table_f32(gppd_handle h, int slot, int64_t n,
                          const int32_t *time_us, double mjd, const float *volt,
                          const double *offsets, const double *timer1, int64_t n1,
                          const double *timer2, int64_t n2, double window_s,
                          const gppd_options *opt, float *volt_out, double *params,
                          double *chi2, int32_t *info, int8_t *state_out);
int gppd_wait(gppd_handle h, int slot);

/*
 * Raw FITS binary-table records (what FitsUtils.jl's Dict(hdu) reads and FITScopy!
 * writes, reference src/FitsUtils.jl:31-37,95-156): `rows` holds the n records of the
 * METROLOGY BINTABLE as stored in the file (big-endian, row_bytes = NAXIS1 bytes each),
 * TIME (int32, "1J") at byte time_off and VOLT (80 float32, "80E") at byte volt_off of
 * a record, at any alignment.  Byte-swapping, de-interleaving and re-packing are done
 * on the device.  rows_out receives the records of the output table: the input record
 * with its VOLT field replaced by the demodulated 80 floats (144 with GPPD_KEEPRAW, the
 * record then grows by 256 bytes: row_bytes_out = row_bytes + 256), every other byte
 * copied.  Asynchronous on pipeline slot `slot` like gppd_submit_table_f32; the
 * other arguments are as for gppd_process_table_f32.
 */
int gppd_submit_fits_rows(gppd_handle h, int slot, int64_t n, const void *rows,
                          int64_t row_bytes, int64_t time_off, int64_t volt_off, double mjd,
                          const double *offsets, const double *timer1, int64_t n1,
                          const double *timer2, int64_t n2, double window_s,
                          const gppd_options *opt, void *rows_out, double *params,
                          double *chi2, int32_t *info, int8_t *state_out);

/*
 * ---- native file ingest / egress, src/FitsUtils.jl:31-37,95-156 ----------------------
 * The record path without the host language touching a byte of the table: the library
 * reads the n METROLOGY records of a (plain, uncompressed) FITS file straight into the
 * slot's pinned staging buffer on its own reader threads -- chunk by chunk, each chunk
 * uploaded while the next one is being read --, runs the batch of gppd_submit_fits_rows
 * on them, brings the output records back into pinned memory, and its writer threads
 * assemble the output file (FITScopy!: every other HDU copied, the METROLOGY table and
 * its header replaced).  The host language keeps what is cheap and its own: header
 * parsing / gating (src/GPPupilDemodulation.jl:358-392) and the text of the new header.
 *
 *   gppd_file_submit   returns at once; the job runs on the handle's I/O threads.  It
 *                      first waits for the slot's previous file to be written.
 *   gppd_file_wait     blocks until the fit results are there and copies them out
 *                      (params [nwin x 32 x 6], chi2 [nwin x 32], info / state may be NULL).
 *   gppd_file_write    returns at once; a writer thread writes the segments in order:
 *                        GPPD_SEG_COPY     `length` bytes of the INPUT file from `offset`
 *                        GPPD_SEG_BYTES    `length` bytes from `bytes` (copied at call time)
 *                        GPPD_SEG_RECORDS  the n output records (each followed by its
 *                                          `extra_row_bytes` bytes of `extra`, if any: the
 *                                          per-row columns of window mode, :239-249), then
 *                                          zero padding to a multiple of 2880 bytes
 *                      `extra` must stay valid until the slot's next gppd_file_submit or
 *                      gppd_file_drain returns.
 *   gppd_file_drain    waits for every pending job of the handle; returns the first error.
 * Errors of the asynchronous parts are reported by the next wait / drain on the slot.
 */
#define GPPD_SEG_COPY 0
#define GPPD_SEG_BYTES 1
#define GPPD_SEG_RECORDS 2
typedef struct gppd_file_segment {
    int32_t kind;       /* GPPD_SEG_* */
    int32_t reserved;
    int64_t offset;     /* GPPD_SEG_COPY: byte offset in the input file */
    int64_t length;     /* GPPD_SEG_COPY / GPPD_SEG_BYTES */
    const void *bytes;  /* GPPD_SEG_BYTES */
} gppd_file_segment;

int gppd_file_submit(gppd_handle h, int slot, const char *path, int64_t data_offset, int64_t n,
                     int64_t row_bytes, int64_t time_off, int64_t volt_off, double mjd,
                     const double *offsets, const double *timer1, int64_t n1,
                     const double *timer2, int64_t n2, double window_s, const gppd_options *opt);
int gppd_file_wait(gppd_handle h, int slot, double *params, double *chi2, int32_t *info,
                   int8_t *state_out);
int gppd_file_write(gppd_handle h, int slot, const char *out_path, const gppd_file_segment *segs,
                    int32_t nsegs, const void *extra, int64_t extra_row_bytes);
int gppd_file_drain(gppd_handle h);

/*
 * Device-resident variant (all pointers are device pointers on the handle's
 * GPU; `stream` is a cudaStream_t passed as void*, NULL = the slot's own
 * stream).  No host<->device copies, no synchronisation: the caller orders
 * and synchronises the stream.  nwindow_rows as in gppd_demodulate_f64.
 * Scratch comes from pipeline slot `slot`.
 */
int gppd_process_table_f32_dev(gppd_handle h, int slot, void *stream, int64_t n,
                               int64_t nwindow_rows, const int32_t *d_time_us,
                               double mjd, const float *d_volt,
                               const double *d_offsets, const double *timer1,
                               int64_t n1, const double *timer2, int64_t n2,
                               const gppd_options *opt, float *d_volt_out,
                               double *d_params, double *d_chi2, int32_t *d_info,
                               int8_t *d_state_out);

/*
 * Batch of tables (a night, or a chunk of one) in ONE launch sequence: every
 * pass covers all tables, so the GPU stays full even though one table holds
 * only 32 fits.  Arrays have `ntables` entries; pointer arrays hold device
 * pointers, timer arrays hold HOST pointers (NULL entry / NULL array = bright
 * table); nwindow_rows may be NULL (whole-table fits); d_info / d_state_out may
 * be NULL.  d_offsets (40 complex128, shared) may be NULL (fit the centres).
 */
int gppd_process_tables_f32_dev(gppd_handle h, int slot, void *stream, int64_t ntables,
                                const int64_t *n, const int64_t *nwindow_rows,
                                const int32_t *const *d_time_us, const double *mjd,
                                const float *const *d_volt, const double *d_offsets,
                                const double *const *timer1, const int64_t *n1,
                                const double *const *timer2, const int64_t *n2,
                                const gppd_options *opt, float *const *d_volt_out,
                                double *const *d_params, double *const *d_chi2,
                                int32_t *const *d_info, int8_t *const *d_state_out);

/*
 * The centres the last GPPD_CENTER_EMPIRICAL call on pipeline slot `slot` fitted and
 * subtracted: centres [ntables][40] complex128 (ntables = 1 for the single-table entry
 * points).  Waits for the slot's own stream (after a *_dev call on a caller-supplied
 * stream the caller synchronises that stream first).  A channel without a circle (fewer
 * than 3 samples, or all on one line) has centre 0.
 */
int gppd_centres(gppd_handle h, int slot, int64_t ntables, double *centres);

/*
 * The maps the last GPPD_CENTER_ELLIPSE call on pipeline slot `slot` fitted and applied:
 * ell [ntables][40][GPPD_ELLIPSE_STRIDE] = (x0, y0, r, alpha, m21, m22) and, unless NULL,
 * status [ntables][40] = 2 (ellipse), 1 (no ellipse: circle centre, identity shape) or
 * 0 (no circle either: centre 0, identity).  Waits like gppd_centres.
 */
#define GPPD_ELLIPSE_STRIDE 6
int gppd_ellipses(gppd_handle h, int slot, int64_t ntables, double *ell, int32_t *status);

/*
 * The parameter covariances (GPPD_COVARIANCE) of the last call on pipeline slot `slot`:
 * cov [nfits][6][6] in params order (table, then window, then diode).  GPPD_ERR_ARG when
 * that call ran without the flag or had fewer than nfits fits.  Waits like gppd_centres;
 * after gppd_file_submit, call it once gppd_file_wait has returned.
 */
int gppd_covariances(gppd_handle h, int slot, int64_t nfits, double *cov);

/*
 * Test hook: the harmonic-sum table of the last batch of pipeline slot `slot`
 * (value-major, [value][fit]; see csrc/gppd_device.cuh), so that the tests can hold the
 * two implementations of the sums (FP64 DMMA, int8 tensor cores) against each other.
 */
int gppd_debug_harmonics(gppd_handle h, int slot, double *htab, int64_t nvals);

/* Experiment hook: 16 cycle counters of the tensor-core harmonic kernel, non-zero only in
 * builds with -DTC_PROFILE (csrc/harm_tc_kernels.cu says what each one is). */
int gppd_debug_counters(gppd_handle h, uint64_t *out16, int reset);

/*
 * Batches that hold both FAINT and bright tables run as two concurrent launch sequences
 * (the latency-bound tail of one chain's fit and its HBM-bound demodulation overlap the
 * other chain's harmonic pass; results do not depend on it).  on = 0 keeps one launch
 * sequence per batch, e.g. to time the passes one by one (gppd_pass_times); the default
 * is on unless the environment has GPPD_SPLIT_CHAINS=0.
 */
int gppd_set_split_chains(gppd_handle h, int on);

/* number of kernels this library has launched on the handle so far */
int64_t gppd_launch_count(gppd_handle h);

/* Per-pass device timing (CUDA events on the launching stream around each pass
 * of the launch sequence).  ms[p] / counts[p] accumulate over all slots since
 * the last reset; gppd_pass_times waits for the recorded events. */
#define GPPD_PASS_SEGMENT 0 /* FAINT segmentation (buildstates)          */
#define GPPD_PASS_BASIS 1   /* per-row sin/cos basis + job ranges (+ the centre fits and the
                               ellipse correction of --center empirical / ellipse) */
#define GPPD_PASS_STATS 2   /* per-state mean/variance (FAINT)            */
#define GPPD_PASS_FIT 3     /* the modulation fit (NEWUOA + objective)    */
#define GPPD_PASS_DEMOD 4   /* demodulation + repack (+ the ellipse mode's repack) */
#define GPPD_PASS_EXPORT 5  /* parameter export                           */
#define GPPD_PASS_HARMONICS 6 /* Jacobi-Anger harmonic sums (harmonic evaluator) */
#define GPPD_PASS_FALLBACK 7  /* direct re-fit of the fits the harmonic evaluator gave up on */
#define GPPD_NPASS 8
int gppd_enable_timing(gppd_handle h, int on);
/* measured FP64 FMA throughput of the device in TFLOP/s (the better of a DFMA and an
 * mma.sync.m8n8k4.f64 micro-benchmark; both use the same FP64 units): the denominator
 * of the harmonic pass's FP64 roofline */
int gppd_measure_fp64_peak(gppd_handle h, double *tflops);
int gppd_pass_times(gppd_handle h, double *ms, int64_t *counts, int reset);

#ifdef __cplusplus
}
#endif
#endif /* GPPD_H */
