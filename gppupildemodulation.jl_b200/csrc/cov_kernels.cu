// cov_kernels.cu -- GPPD_COVARIANCE: the Gauss-Newton covariance of every fit's reported
// parameters (definition: include/gppd.h).  One streaming pass over the valid rows after the
// fit, in two launches:
//
//   k_cov_seg    one block per (job, FIXED segment of COV_SEG_ROWS rows); lane = diode (the 32
//                fits of the job), warp w takes rows w, w + 8, ... of the segment.  Per row and
//                fit: the model g = p e^{j b s}, the six real 2-vectors of the Jacobian and the
//                21 entries of the upper triangle of H plus sum w |r|^2, accumulated in FP64.
//                The 8 warps' sums are added in warp order and written as one partial per
//                (fit, segment).
//   k_cov_final  one thread per fit: the segments added in index order, the Cholesky
//                factorisation of the diagonally scaled H, its inverse, times s^2.
//
// Fixed segments and in-order sums: a fit's covariance does not depend on the batch it is
// in nor on the launch shape, like every other partial sum of the library.
#include "fit_math.cuh"
#include "gppd_device.cuh"
#include "kernels.h"

namespace gppd {

constexpr int COV_THREADS = 256;
constexpr int COV_WARPS = COV_THREADS / 32;

int cov_max_segments(long long max_rows_per_job) {
    return (int)((max_rows_per_job + COV_SEG_ROWS - 1) / COV_SEG_ROWS);
}

// the parameters as exported (k_export's sign normalisation of b < 0)
__device__ __forceinline__ void exported_b_phi(const FitResult &r, double &b, double &phi) {
    b = r.b;
    phi = r.phi;
    if (b < 0) {
        b = -b;
        phi += (phi < 0 ? PI_F64 : -PI_F64);
    }
}

// index of (k, l), k <= l, in the packed upper triangle of a 6 x 6 matrix
__host__ __device__ constexpr int tri6(int k, int l) { return k * 6 - k * (k - 1) / 2 + (l - k); }

__global__ void __launch_bounds__(COV_THREADS)
k_cov_seg(const TableDesc *tabs, const JobInfo *jobs, const FitResult *results, const double *stats,
          unsigned flags, int P, double *part) {
    __shared__ double red[COV_WARPS][COV_VALS][32];
    const int job = blockIdx.x, seg = blockIdx.y;
    const JobInfo ji = jobs[job];
    const int i0 = seg * COV_SEG_ROWS;
    if (i0 >= ji.nrows) return;
    const int i1 = (i0 + COV_SEG_ROWS < ji.nrows) ? i0 + COV_SEG_ROWS : ji.nrows;
    const TableDesc &tb = tabs[ji.table];
    const TableView &tv = tb.tv;
    const int8_t *state = tb.state;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int group = lane >> 2, fcch = fc_channel(group);
    const bool active = group_on(flags, group);

    const FitResult r = results[(long long)job * NDIODE + lane];
    double b, phi;
    exported_b_phi(r, b, phi);
    const PhaseQ pq = make_phaseq(phi, ji.thmin, ji.thmax);
    const double cre = r.cre, cim = r.cim, are = r.are, aim = r.aim;
    double2 mw[4];
#pragma unroll
    for (int s = 0; s < 4; ++s)
        mw[s] = state ? stats_mean_weight(stats, job * NGROUP + group, lane & 3, s) : make_double2(1.0, 1.0);

    double acc[COV_VALS];
#pragma unroll
    for (int v = 0; v < COV_VALS; ++v) acc[v] = 0.0;
    if (active) {
        for (int i = i0 + warp; i < i1; i += COV_WARPS) {
            const long long row = ji.row0 + i;
            double w = 1.0, m = 1.0;
            if (state) {
                const int st = state[row];
                if (!row_valid(st, flags)) continue;     // (warp-uniform: one row per warp)
                m = mw[st & 3].x;
                w = mw[st & 3].y;
            }
            const double2 d = row_sample(tv, row, lane);
            const double2 fc = fc_phasor(row_sample(tv, row, fcch));
            const double2 sc = tb.basis[row];
            // s, cs = sin, cos of fl(theta + phi)
            double s, cs;
            if (pq.uniform) {
                s = fma(sc.x, pq.cq, sc.y * pq.sq);
                cs = fma(sc.y, pq.cq, -(sc.x * pq.sq));
            } else {
                const double th = row_theta(tv, row);
                const double qn = __dadd_rn(th, phi) - th;
                double sqn, cqn;
                sincos(qn, &sqn, &cqn);
                s = fma(sc.x, cqn, sc.y * sqn);
                cs = fma(sc.y, cqn, -(sc.x * sqn));
            }
            double su, cu;
            sincos_moderate(b * s, &su, &cu);
            const double pr = m * fc.x, pi = m * fc.y;
            const double gr = fma(pr, cu, -(pi * su)), gi = fma(pr, su, pi * cu);   // g = p e^{j b s}
            const double Gr = fma(are, gr, -(aim * gi)), Gi = fma(are, gi, aim * gr);  // a g
            const double rr = (cre + Gr) - d.x, ri = (cim + Gi) - d.y;               // m - d
            // the Jacobian columns as real 2-vectors (re, im)
            const double bcs = b * cs;
            const double vx[6] = {1.0, 0.0, gr, -gi, s * -Gi, bcs * -Gi};
            const double vy[6] = {0.0, 1.0, gi, gr, s * Gr, bcs * Gr};
#pragma unroll
            for (int k = 0; k < 6; ++k)
#pragma unroll
                for (int l = k; l < 6; ++l)
                    acc[tri6(k, l)] = fma(w, fma(vx[k], vx[l], vy[k] * vy[l]), acc[tri6(k, l)]);
            acc[COV_SSE] = fma(w, fma(rr, rr, ri * ri), acc[COV_SSE]);
        }
    }
#pragma unroll
    for (int v = 0; v < COV_VALS; ++v) red[warp][v][lane] = acc[v];
    __syncthreads();
    double *out = part + ((long long)job * P + seg) * COV_VALS * 32;
    for (int e = threadIdx.x; e < COV_VALS * 32; e += COV_THREADS) {
        const int v = e >> 5, l = e & 31;
        double t = 0.0;
#pragma unroll
        for (int k = 0; k < COV_WARPS; ++k) t += red[k][v][l];
        out[e] = t;
    }
}

__global__ void k_cov_final(const JobInfo *jobs, const FitResult *results, const double *part, int P, int nfits,
                            unsigned flags, double *cov) {
    const int fit = blockIdx.x * blockDim.x + threadIdx.x;
    if (fit >= nfits) return;
    const int job = fit / NDIODE, lane = fit % NDIODE;
    const JobInfo ji = jobs[job];
    const bool offs = (flags & 2u) != 0;
    const int k0 = offs ? 0 : 2, k = 6 - k0;
    double *out = cov + (long long)fit * 36;

    const int nseg = (ji.nrows + COV_SEG_ROWS - 1) / COV_SEG_ROWS;
    double sum[COV_VALS];
#pragma unroll
    for (int v = 0; v < COV_VALS; ++v) sum[v] = 0.0;
    for (int s = 0; s < nseg; ++s) {
        const double *p = part + ((long long)job * P + s) * COV_VALS * 32 + lane;
#pragma unroll
        for (int v = 0; v < COV_VALS; ++v) sum[v] += p[v * 32];
    }
    const FitResult r = results[fit];
    bool ok = group_on(flags, lane >> 2) && 2 * ji.nvalid > k;
    ok = ok && !isnan(r.b) && !isnan(r.phi) && !isnan(r.cre) && !isnan(r.cim) && !isnan(r.are) && !isnan(r.aim);

    // scaled H = D H D, D = diag(1 / sqrt(H_ii)), factorised as L L^T
    double D[6], L[6][6];
    for (int i = 0; i < 6; ++i) {
        const double h = sum[tri6(i, i)];
        D[i] = (i >= k0 && h > 0.0) ? 1.0 / sqrt(h) : 0.0;
        if (i >= k0 && !(h > 0.0)) ok = false;
    }
    for (int i = 0; i < 6; ++i)
        for (int j = 0; j < 6; ++j) L[i][j] = 0.0;
    for (int j = k0; j < 6 && ok; ++j) {
        double piv = sum[tri6(j, j)] * D[j] * D[j];
        for (int m = k0; m < j; ++m) piv -= L[j][m] * L[j][m];
        if (!(piv > 1e-12)) {
            ok = false;
            break;
        }
        L[j][j] = sqrt(piv);
        for (int i = j + 1; i < 6; ++i) {
            double a = sum[tri6(j, i)] * D[i] * D[j];
            for (int m = k0; m < j; ++m) a -= L[i][m] * L[j][m];
            L[i][j] = a / L[j][j];
        }
    }
    // L^-1 (lower triangular), then (D H D)^-1 = L^-T L^-1
    double M[6][6];
    for (int i = 0; i < 6; ++i)
        for (int j = 0; j < 6; ++j) M[i][j] = 0.0;
    if (ok) {
        for (int j = k0; j < 6; ++j) {
            M[j][j] = 1.0 / L[j][j];
            for (int i = j + 1; i < 6; ++i) {
                double a = 0.0;
                for (int m = j; m < i; ++m) a += L[i][m] * M[m][j];
                M[i][j] = -a / L[i][i];
            }
        }
    }
    const double s2 = ok ? sum[COV_SSE] / (double)(2 * ji.nvalid - k) : 0.0;
    double C[36];
    for (int i = 0; i < 6; ++i) {
        for (int j = i; j < 6; ++j) {
            double a = 0.0;
            for (int m = j; m < 6; ++m) a += M[m][i] * M[m][j];
            const double c = s2 * (D[i] * (a * D[j]));
            C[6 * i + j] = C[6 * j + i] = c;
            if (i >= k0 && isnan(c)) ok = false;
        }
    }
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    for (int e = 0; e < 36; ++e) out[e] = ok ? C[e] : nan;
}

void launch_covariance(const Launcher &L, const TableDesc *d_tabs, const JobInfo *d_jobs, int njobs,
                       const FitResult *d_results, const double *d_stats, unsigned flags, int P, double *d_part,
                       double *d_cov) {
    if (njobs <= 0) return;
    k_cov_seg<<<dim3((unsigned)njobs, (unsigned)P), COV_THREADS, 0, L.stream>>>(d_tabs, d_jobs, d_results, d_stats,
                                                                                flags, P, d_part);
    const int nfits = njobs * NDIODE;
    k_cov_final<<<(nfits + 127) / 128, 128, 0, L.stream>>>(d_jobs, d_results, d_part, P, nfits, flags, d_cov);
    *L.counter += 2;
}

}  // namespace gppd
