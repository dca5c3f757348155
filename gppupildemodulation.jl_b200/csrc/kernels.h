// kernels.h -- host-callable launchers of the device passes.  Every pass is
// batched: one launch covers all tables (or all jobs / fits) of a batch.
#pragma once
#include "gppd_device.cuh"

namespace gppd {

constexpr int SEG_EVENT_BYTES = 24;

// where one table's fit results go in the caller's layout
struct ExportDesc {
    int fit0, nfits;      // this table's fits in the batch result array
    double *params;       // [nfits][6]
    double *chi2;         // [nfits]
    int *info;            // [nfits][4] or nullptr
};

// FAINT segmentation (reference buildstates, src/Faint.jl:21-73)
void launch_segmentation(const Launcher &L, const TableDesc *d_tabs, int ntables,
                         long long max_rows, int max_timers);

// per-row basis + per-job theta range / valid count / first row of each state
// (d_nvalid: 5 ints per job)
void launch_basis(const Launcher &L, const TableDesc *d_tabs, int ntables, long long max_rows,
                  int max_jobs_per_table, int njobs, unsigned flags,
                  unsigned long long *d_thkeys, int *d_nvalid, JobInfo *d_jobs);

// per-state (mean |d|, 1 / var |d|) table (reference compute_mean_var_power,
// src/Faint.jl:89-100): d_part = per-segment partials, d_table = [njobs*8][16] double2
// d_faint_jobs: the nfaint jobs (batch job indices) whose table has states
void launch_stats(const Launcher &L, const TableDesc *d_tabs, const JobInfo *d_jobs, int njobs,
                  const int *d_faint_jobs, int nfaint, const int *d_jobcnt, unsigned flags, int P,
                  double *d_part, double *d_table, bool dense);

// `--center empirical` (reference compute_offsets, src/GPPupilDemodulation.jl:105-125):
// algebraic circle fit of each of the 40 channels of every kind-0 table whose
// tv.offsets is set, over all rows or the HIGH rows of a table with states; writes the
// 40 centres INTO tv.offsets.  d_part: [ntables][circle_max_segments][CIRC_VALS][40]
constexpr int CIRC_SEG_ROWS = 4096;
constexpr int CIRC_VALS = 10;
int circle_max_segments(long long max_rows);
void launch_circle(const Launcher &L, const TableDesc *d_tabs, int ntables, long long max_rows,
                   double *d_part);

// `--center ellipse` (GPPD_CENTER_ELLIPSE, centre_kernels.cu).  On kind-0 descriptors whose
// tv.t / tv.data point at the corrected arrays and ov.out at the demodulated ones:
//   launch_ellipse_fit    the ten circle sums + five fourth-order ones over the same fixed
//                         segments (d_part: [ntables][circle_max_segments][ELL_VALS][40]),
//                         then one conic per channel -> d_ell [ntables][40][ELL_STRIDE]
//                         = (x0, y0, r, alpha, m21, m22), d_status [ntables][40]
//   launch_ellipse_apply  TIME + VOLT rows -> t [n] f64 and corrected data [40][n] complex128
//   launch_repack_arrays  demodulated out [40][n] complex128 -> float32 VOLT rows of ov
constexpr int ELL_VALS = 15;
constexpr int ELL_STRIDE = 6;
void launch_ellipse_fit(const Launcher &L, const TableDesc *d_tabs, int ntables, long long max_rows,
                        double *d_part, double *d_ell, int *d_status);
void launch_ellipse_apply(const Launcher &L, const TableDesc *d_tabs, int ntables, long long max_rows,
                          const double *d_ell);
void launch_repack_arrays(const Launcher &L, const TableDesc *d_tabs, int ntables, long long max_rows, bool keepraw);

// Jacobi-Anger harmonic sums of every fit + reduction into the harmonic table
int harm_max_segments(long long max_rows_per_job);   // fixed 6144-row segments
int stats_max_segments(long long max_rows_per_job);  // fixed 1024-row segments
// tensor: the int8 tensor-core kernel (harm_tc_kernels.cu; dense METROLOGY tables only)
// instead of the FP64 DMMA kernel (harm_kernels.cu; any layout)
void launch_harmonics(const Launcher &L, const TableDesc *d_tabs, const JobInfo *d_jobs, int njobs,
                      unsigned flags, int P, int SP, const double *d_spart1,
                      const double *d_spart2, double *d_partZ, double *d_partY, double *d_htab,
                      int tensor);   // 0: FP64 DMMA kernel, 1: int8 tensor cores on tables, 2: on complex128 arrays
void tc_profile_read(unsigned long long *out16, int reset);   // TC_PROFILE experiment builds
int harm_tc_min_rows();   // shortest job the tensor kernel is used for (1; GPPD_HARMONICS=dmma: never)
void launch_harmonics_tc32(const Launcher &L, const TableDesc *d_tabs, const JobInfo *d_jobs, int njobs,
                           unsigned flags, int P, const double *d_spart2, double *d_partZ, double *d_partY);
void launch_harmonics_tc(const Launcher &L, const TableDesc *d_tabs, const JobInfo *d_jobs, int njobs,
                         unsigned flags, int P, const double *d_spart2, double *d_partZ, double *d_partY,
                         bool arrays);

// the fit, harmonic evaluator (one thread per fit)
void launch_fit_harmonic(const Launcher &L, const TableDesc *d_tabs, const JobInfo *d_jobs,
                         const double *d_htab, int nfits, const FitOptions &opt,
                         FitResult *d_results, double *d_trace, int *d_fbq);

// the fit, direct evaluator (one block per fit); scratch = false: only the fits the
// harmonic evaluator queued in d_fbq ([0] = count, [1..] = fit numbers) run,
// recomputing z / y from the table
void launch_fit_direct(const Launcher &L, const TableDesc *d_tabs, const JobInfo *d_jobs,
                       int nfits, int SP, const double *d_spart1, const double *d_spart2,
                       const FitOptions &opt, bool scratch, FitResult *d_results, double *d_trace,
                       const int *d_fbq);

// demodulation + repack (reference src/Modulation.jl:417-425)
void launch_demod(const Launcher &L, const TableDesc *d_tabs, int ntables, long long max_rows,
                  const FitResult *d_results, unsigned flags, bool arrays);

// FitResult -> params / chi2 / info in the caller's layout
void launch_export(const Launcher &L, const ExportDesc *d_exps, int ntables, int max_fits,
                   const FitResult *d_results, unsigned flags);

// GPPD_COVARIANCE (cov_kernels.cu): per (job, FIXED segment of COV_SEG_ROWS rows) the 21 entries
// of the upper triangle of H and sum w |r|^2 of each of the job's 32 fits -> d_part
// [njobs][P][COV_VALS][32]; then per fit the covariance, 36 doubles -> d_cov [nfits][36].
// d_stats: the per-state (mean, weight) table of the statistics pass (tables with states).
constexpr int COV_SEG_ROWS = 4096;
constexpr int COV_SSE = 21;
constexpr int COV_VALS = 22;
int cov_max_segments(long long max_rows_per_job);
void launch_covariance(const Launcher &L, const TableDesc *d_tabs, const JobInfo *d_jobs, int njobs,
                       const FitResult *d_results, const double *d_stats, unsigned flags, int P, double *d_part,
                       double *d_cov);

// raw FITS binary-table records <-> dense little-endian TIME / VOLT arrays
void launch_unpack_rows(const Launcher &L, const void *d_rows, long long n, long long row_bytes,
                        long long time_off, long long volt_off, int32_t *d_time, float *d_volt);
void launch_pack_rows(const Launcher &L, const void *d_rows, long long n, long long row_bytes,
                      long long volt_off, const float *d_volt_out, int out_floats, void *d_rows_out,
                      long long row_bytes_out);

// measured FP64 FMA throughput of the device (TFLOP/s), for the fit's roofline
double measure_dfma_tflops(cudaStream_t stream, double *d_scratch);

}  // namespace gppd
