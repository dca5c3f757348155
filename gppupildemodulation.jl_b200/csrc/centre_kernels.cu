// centre_kernels.cu -- `--center empirical`: one circle per channel.
//
// Reference: compute_offsets, src/GPPupilDemodulation.jl:105-125 -- for each of the 40
// channels `fit(Circle, re, im)` over all samples of the table, or over its HIGH samples
// when the table has FAINT states, and processmetrology subtracts the circle centres
// (:153-154).  `Circle` is not defined in the reference's environment, so the reference
// throws there; this is the algebraic (Kasa) least-squares circle the call was written
// for: minimise sum (x^2 + y^2 - 2 x0 x - 2 y0 y - c)^2, a linear problem in
// (x0, y0, c), i.e. ten moment sums per channel and a 2x2 solve.
//
// The sums are taken relative to a pivot on the circle (the channel's sample of the
// table's first row), which keeps every moment at the scale of the radius whatever the
// distance of the circle from the origin, and over FIXED row segments added in index
// order, so a table's centres do not depend on the batch it is in.
//
// `--center ellipse` (GPPD_CENTER_ELLIPSE) generalises the circle to the conic
// A u^2 + B uv + C v^2 + D u + E v + F = 0 with A + C = 1 (Heydemann correction of
// quadrature detectors with a gain mismatch and a quadrature phase error): the same
// segment pass with five more (fourth-order) moments, a 5x5 Cholesky solve per channel,
// then k_ellipse_apply maps every row onto the circle, x' = x - x0,
// y' = tan(alpha) x' + r / cos(alpha) (y - y0), into complex128 arrays that the ordinary
// array path demodulates; k_repack_arrays turns its output back into VOLT rows.
#include "kernels.h"

namespace gppd {

constexpr int CIRC_LANES = 8;                       // rows in flight per block iteration
constexpr int CIRC_THREADS = CIRC_LANES * NCHAN;    // thread = (row lane, channel)
constexpr int CIRC_UNROLL = 8;

int circle_max_segments(long long max_rows) {
    return (int)((max_rows + CIRC_SEG_ROWS - 1) / CIRC_SEG_ROWS);
}

// centred sample (u, v) -> the ten moments
struct Moments {
    double n, u, v, uu, uv, vv, uuu, uuv, uvv, vvv;
};

// the five fourth-order moments of the ellipse fit
struct Moments4 {
    double uuuu, uuuv, uuvv, uvvv, vvvv;
};

__device__ __forceinline__ void add_sample(Moments &m, double u, double v) {
    const double uu = u * u, vv = v * v;
    m.n += 1.0;
    m.u += u;
    m.v += v;
    m.uu += uu;
    m.uv = fma(u, v, m.uv);
    m.vv += vv;
    m.uuu = fma(uu, u, m.uuu);
    m.uuv = fma(uu, v, m.uuv);
    m.uvv = fma(u, vv, m.uvv);
    m.vvv = fma(vv, v, m.vvv);
}

__device__ __forceinline__ void add_sample4(Moments4 &m, double u, double v) {
    const double uu = u * u, vv = v * v, uv = u * v;
    m.uuuu = fma(uu, uu, m.uuuu);
    m.uuuv = fma(uu, uv, m.uuuv);
    m.uuvv = fma(uu, vv, m.uuvv);
    m.uvvv = fma(uv, vv, m.uvvv);
    m.vvvv = fma(vv, vv, m.vvvv);
}

// grid (segment, table); a row is 40 consecutive float2 = one coalesced 320-byte read
// of the 40 threads of a row lane.  NV = CIRC_VALS (circle) or ELL_VALS (ellipse: the
// same ten sums, then the five fourth-order ones)
template <int NV>
__global__ void __launch_bounds__(CIRC_THREADS) k_circle_seg(const TableDesc *tabs, int P,
                                                             double *part) {
    __shared__ double s_m[CIRC_LANES][NV][NCHAN];
    const TableDesc &tb = tabs[blockIdx.y];
    if (tb.tv.kind != 0 || !tb.tv.offsets) return;
    const long long n = tb.tv.n;
    const long long r0 = (long long)blockIdx.x * CIRC_SEG_ROWS;
    if (r0 >= n) return;
    const long long r1 = min(n, r0 + (long long)CIRC_SEG_ROWS);
    const int lane = threadIdx.x / NCHAN, ch = threadIdx.x - lane * NCHAN;
    const int8_t *state = tb.state;
    TableView tv = tb.tv;
    tv.offsets = nullptr;                      // raw volts
    const double2 piv = row_sample(tv, 0, ch);

    Moments m = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    Moments4 m4 = {0, 0, 0, 0, 0};
    for (long long r = r0 + lane; r < r1; r += CIRC_LANES * CIRC_UNROLL) {
        double2 d[CIRC_UNROLL];
        int use[CIRC_UNROLL];
#pragma unroll
        for (int j = 0; j < CIRC_UNROLL; ++j) {
            const long long rr = r + (long long)j * CIRC_LANES;
            use[j] = rr < r1;
            if (use[j]) {
                d[j] = row_sample(tv, rr, ch);
                if (state) use[j] = state[rr] == ST_HIGH;   // cmplxV[state .== HIGH, ch], :108
            }
        }
#pragma unroll
        for (int j = 0; j < CIRC_UNROLL; ++j)
            if (use[j]) {
                add_sample(m, d[j].x - piv.x, d[j].y - piv.y);
                if constexpr (NV == ELL_VALS) add_sample4(m4, d[j].x - piv.x, d[j].y - piv.y);
            }
    }
    double *sm = &s_m[lane][0][ch];
    sm[0 * NCHAN] = m.n;   sm[1 * NCHAN] = m.u;   sm[2 * NCHAN] = m.v;   sm[3 * NCHAN] = m.uu;
    sm[4 * NCHAN] = m.uv;  sm[5 * NCHAN] = m.vv;  sm[6 * NCHAN] = m.uuu; sm[7 * NCHAN] = m.uuv;
    sm[8 * NCHAN] = m.uvv; sm[9 * NCHAN] = m.vvv;
    if constexpr (NV == ELL_VALS) {
        sm[10 * NCHAN] = m4.uuuu; sm[11 * NCHAN] = m4.uuuv; sm[12 * NCHAN] = m4.uuvv;
        sm[13 * NCHAN] = m4.uvvv; sm[14 * NCHAN] = m4.vvvv;
    }
    __syncthreads();
    // lanes added in lane order: [table][segment][value][channel]
    double *dst = part + ((size_t)blockIdx.y * P + blockIdx.x) * (NV * NCHAN);
    for (int i = threadIdx.x; i < NV * NCHAN; i += CIRC_THREADS) {
        double acc = 0.0;
#pragma unroll
        for (int l = 0; l < CIRC_LANES; ++l) acc += (&s_m[l][0][0])[i];
        dst[i] = acc;
    }
}

// Kasa circle centre from the first ten sums (centred moments, 2x2 solve); false when the
// channel has fewer than 3 samples or they lie on one line
__device__ __forceinline__ bool kasa_centre(const double *s, double2 piv, double2 &centre) {
    const double N = s[0];
    if (!(N >= 3.0)) return false;
    const double mu = s[1] / N, mv = s[2] / N;
    const double cuu = s[3] - N * mu * mu;
    const double cuv = s[4] - N * mu * mv;
    const double cvv = s[5] - N * mv * mv;
    const double cuuu = s[6] - 3.0 * mu * s[3] + 2.0 * N * mu * mu * mu;
    const double cvvv = s[9] - 3.0 * mv * s[5] + 2.0 * N * mv * mv * mv;
    const double cuuv = s[7] - 2.0 * mu * s[4] - mv * s[3] + 2.0 * N * mu * mu * mv;
    const double cuvv = s[8] - 2.0 * mv * s[4] - mu * s[5] + 2.0 * N * mu * mv * mv;
    const double det = cuu * cvv - cuv * cuv;
    if (!(det > 1.0e-12 * cuu * cvv && det > 0.0)) return false;
    const double bu = 0.5 * (cuuu + cuvv), bv = 0.5 * (cvvv + cuuv);
    const double uc = (bu * cvv - bv * cuv) / det;
    const double vc = (bv * cuu - bu * cuv) / det;
    centre = make_double2(piv.x + (mu + uc), piv.y + (mv + vc));
    return true;
}

// one thread per (table, channel): segments in index order, then the 2x2 solve.  A
// channel with fewer than 3 samples, or whose samples lie on one line, has no circle:
// its centre is 0 (the channel is left as it is).
__global__ void k_circle_solve(const TableDesc *tabs, int ntables, int P, const double *part) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ntables * NCHAN) return;
    const int t = i / NCHAN, ch = i - t * NCHAN;
    const TableDesc &tb = tabs[t];
    if (tb.tv.kind != 0 || !tb.tv.offsets) return;
    const int nseg = (int)((tb.tv.n + CIRC_SEG_ROWS - 1) / CIRC_SEG_ROWS);
    double s[CIRC_VALS];
#pragma unroll
    for (int k = 0; k < CIRC_VALS; ++k) s[k] = 0.0;
    for (int p = 0; p < nseg; ++p) {
        const double *src = part + ((size_t)t * P + p) * (CIRC_VALS * NCHAN) + ch;
#pragma unroll
        for (int k = 0; k < CIRC_VALS; ++k) s[k] += src[k * NCHAN];
    }
    TableView tv = tb.tv;
    tv.offsets = nullptr;
    double2 centre = make_double2(0.0, 0.0);     // stays 0 without a circle
    kasa_centre(s, row_sample(tv, 0, ch), centre);
    const_cast<double2 *>(tb.tv.offsets)[ch] = centre;
}

void launch_circle(const Launcher &L, const TableDesc *d_tabs, int ntables, long long max_rows,
                   double *d_part) {
    const int P = circle_max_segments(max_rows);
    k_circle_seg<CIRC_VALS><<<dim3(P, ntables), CIRC_THREADS, 0, L.stream>>>(d_tabs, P, d_part);
    k_circle_solve<<<(ntables * NCHAN + 127) / 128, 128, 0, L.stream>>>(d_tabs, ntables, P, d_part);
    *L.counter += 2;
}


// ===========================================================================
// `--center ellipse`
// ===========================================================================

// One thread per (table, channel).  The pivot-relative sums S_pq = sum u^p v^q (p + q <= 4)
// are moved to the centroid analytically (binomial expansion) and scaled to unit rms radius;
// on these the fit A (u^2 - v^2) + B uv + D u + E v + F = -v^2 is a 5x5 normal system,
// solved by Cholesky.  Output per channel: ell[6] = (x0, y0, r, alpha, m21, m22) and the
// status 2 (ellipse), 1 (no ellipse: Kasa centre, identity shape) or 0 (no circle either:
// centre 0, identity).
__global__ void k_ellipse_solve(const TableDesc *tabs, int ntables, int P, const double *part,
                                double *ell, int *status) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ntables * NCHAN) return;
    const int t = i / NCHAN, ch = i - t * NCHAN;
    const TableDesc &tb = tabs[t];
    const int nseg = (int)((tb.tv.n + CIRC_SEG_ROWS - 1) / CIRC_SEG_ROWS);
    double s[ELL_VALS];
#pragma unroll
    for (int k = 0; k < ELL_VALS; ++k) s[k] = 0.0;
    for (int p = 0; p < nseg; ++p) {
        const double *src = part + ((size_t)t * P + p) * (ELL_VALS * NCHAN) + ch;
#pragma unroll
        for (int k = 0; k < ELL_VALS; ++k) s[k] += src[k * NCHAN];
    }
    TableView tv = tb.tv;
    tv.offsets = nullptr;
    const double2 piv = row_sample(tv, 0, ch);
    double2 centre = make_double2(0.0, 0.0);
    int st = kasa_centre(s, piv, centre) ? 1 : 0;
    double r = 1.0, alpha = 0.0, m21 = 0.0, m22 = 1.0;
    const double N = s[0];
    if (N >= 5.0) {
        // S[p][q] from the sums (order of the partial layout), then central moments
        double S[5][5] = {};
        S[0][0] = s[0];  S[1][0] = s[1];  S[0][1] = s[2];
        S[2][0] = s[3];  S[1][1] = s[4];  S[0][2] = s[5];
        S[3][0] = s[6];  S[2][1] = s[7];  S[1][2] = s[8];  S[0][3] = s[9];
        S[4][0] = s[10]; S[3][1] = s[11]; S[2][2] = s[12]; S[1][3] = s[13]; S[0][4] = s[14];
        const double mu = s[1] / N, mv = s[2] / N;
        const double binom[5][5] = {{1, 0, 0, 0, 0}, {1, 1, 0, 0, 0}, {1, 2, 1, 0, 0}, {1, 3, 3, 1, 0}, {1, 4, 6, 4, 1}};
        double pu[5], pv[5];
        pu[0] = pv[0] = 1.0;
        for (int k = 1; k < 5; ++k) {
            pu[k] = pu[k - 1] * -mu;
            pv[k] = pv[k - 1] * -mv;
        }
        double M[5][5] = {};
        for (int p = 0; p <= 4; ++p)
            for (int q = 0; p + q <= 4; ++q) {
                double c = 0.0;
                for (int a = 0; a <= p; ++a)
                    for (int b = 0; b <= q; ++b) c += binom[p][a] * binom[q][b] * pu[p - a] * pv[q - b] * S[a][b];
                M[p][q] = c;
            }
        const double rms2 = (M[2][0] + M[0][2]) / N;
        if (rms2 > 0.0) {
            // scaled, per-sample moments: M[p][q] / (N rms^(p+q))
            const double h = 1.0 / sqrt(rms2);
            double hp[5];
            hp[0] = 1.0 / N;
            for (int k = 1; k < 5; ++k) hp[k] = hp[k - 1] * h;
            for (int p = 0; p <= 4; ++p)
                for (int q = 0; p + q <= 4; ++q) M[p][q] *= hp[p + q];
            M[1][0] = M[0][1] = 0.0;      // centroid frame (exactly, up to rounding)
            // features (x^2 - y^2, xy, x, y, 1), target -y^2
            double G[5][5], g[5];
            G[0][0] = M[4][0] - 2.0 * M[2][2] + M[0][4];
            G[0][1] = M[3][1] - M[1][3];
            G[0][2] = M[3][0] - M[1][2];
            G[0][3] = M[2][1] - M[0][3];
            G[0][4] = M[2][0] - M[0][2];
            G[1][1] = M[2][2];
            G[1][2] = M[2][1];
            G[1][3] = M[1][2];
            G[1][4] = M[1][1];
            G[2][2] = M[2][0];
            G[2][3] = M[1][1];
            G[2][4] = M[1][0];
            G[3][3] = M[0][2];
            G[3][4] = M[0][1];
            G[4][4] = 1.0;
            g[0] = -(M[2][2] - M[0][4]);
            g[1] = -M[1][3];
            g[2] = -M[1][2];
            g[3] = -M[0][3];
            g[4] = -M[0][2];
            for (int a = 0; a < 5; ++a)
                for (int b = 0; b < a; ++b) G[a][b] = G[b][a];
            // Cholesky G = L L' (lower triangle of L in place of G's)
            double L[5][5] = {};
            bool ok = true;
            for (int k = 0; k < 5 && ok; ++k) {
                double d = G[k][k];
                for (int j = 0; j < k; ++j) d -= L[k][j] * L[k][j];
                if (!(d > 1.0e-12 * G[k][k])) {
                    ok = false;
                    break;
                }
                L[k][k] = sqrt(d);
                for (int a = k + 1; a < 5; ++a) {
                    double e = G[a][k];
                    for (int j = 0; j < k; ++j) e -= L[a][j] * L[k][j];
                    L[a][k] = e / L[k][k];
                }
            }
            if (ok) {
                double z[5], x[5];
                for (int a = 0; a < 5; ++a) {
                    double e = g[a];
                    for (int j = 0; j < a; ++j) e -= L[a][j] * z[j];
                    z[a] = e / L[a][a];
                }
                for (int a = 4; a >= 0; --a) {
                    double e = z[a];
                    for (int j = a + 1; j < 5; ++j) e -= L[j][a] * x[j];
                    x[a] = e / L[a][a];
                }
                const double A = x[0], B = x[1], C = 1.0 - x[0], D = x[2], E = x[3];
                const double det = 4.0 * A * C - B * B;
                if (A > 0.0 && C > 0.0 && det > 4.0 * 0.01 / (1.01 * 1.01)) {
                    const double xs = (B * E - 2.0 * C * D) / det;      // [2A B; B 2C] (x, y) = -(D, E)
                    const double ys = (B * D - 2.0 * A * E) / det;
                    const double rms = sqrt(rms2);
                    centre = make_double2(piv.x + (mu + xs * rms), piv.y + (mv + ys * rms));
                    r = sqrt(C / A);
                    alpha = asin(B / (2.0 * sqrt(A * C)));
                    m21 = tan(alpha);
                    m22 = r / cos(alpha);
                    st = 2;
                }
            }
        }
    }
    double *e = ell + (size_t)i * ELL_STRIDE;
    e[0] = centre.x;
    e[1] = centre.y;
    e[2] = r;
    e[3] = alpha;
    e[4] = m21;
    e[5] = m22;
    status[i] = st;
}

void launch_ellipse_fit(const Launcher &L, const TableDesc *d_tabs, int ntables, long long max_rows,
                        double *d_part, double *d_ell, int *d_status) {
    const int P = circle_max_segments(max_rows);
    k_circle_seg<ELL_VALS><<<dim3(P, ntables), CIRC_THREADS, 0, L.stream>>>(d_tabs, P, d_part);
    k_ellipse_solve<<<(ntables * NCHAN + 127) / 128, 128, 0, L.stream>>>(d_tabs, ntables, P, d_part, d_ell,
                                                                         d_status);
    *L.counter += 2;
}

// ---------------------------------------------------------------------------
// Streaming transposes through shared memory: a tile of TR_ROWS rows is read as whole rows
// (coalesced 16-byte loads when the rows allow it) and written as per-channel runs, or the
// other way round.  Tile pitch 81 floats: the 32 rows a warp reads of one channel fall in 32
// different banks.
constexpr int TR_ROWS = 64, TR_THREADS = 256, TR_PITCH = 81;

// rows [r0, r0 + nr) of a VOLT table (80 float32 per row, either byte order) -> s_v
__device__ __forceinline__ void load_volt_tile(const TableView &tv, long long r0, int nr, float *s_v) {
    const bool vec = ((reinterpret_cast<unsigned long long>(tv.volt) | (unsigned long long)tv.volt_stride) & 15ull) == 0;
    if (vec) {
        for (int i = threadIdx.x; i < nr * 20; i += TR_THREADS) {
            const int r = i / 20, j = i - r * 20;
            uint4 w = __ldg(reinterpret_cast<const uint4 *>(reinterpret_cast<const char *>(tv.volt) +
                                                          (r0 + r) * tv.volt_stride) + j);
            if (tv.big_endian) {
                w.x = bswap32(w.x); w.y = bswap32(w.y); w.z = bswap32(w.z); w.w = bswap32(w.w);
            }
            float *d = s_v + r * TR_PITCH + 4 * j;
            d[0] = __uint_as_float(w.x); d[1] = __uint_as_float(w.y);
            d[2] = __uint_as_float(w.z); d[3] = __uint_as_float(w.w);
        }
    } else {
        for (int i = threadIdx.x; i < nr * 80; i += TR_THREADS) {
            const int r = i / 80, j = i - r * 80;
            s_v[r * TR_PITCH + j] = load_f32(reinterpret_cast<const float *>(reinterpret_cast<const char *>(tv.volt) +
                                                                             (r0 + r) * tv.volt_stride) + j,
                                             tv.big_endian);
        }
    }
}

// TIME + VOLT rows -> t (f64, the two roundings of row_time) and the corrected channels
// data[40][n] complex128: x' = x - x0, y' = m21 x' + m22 (y - y0), every operation rounded
// (no FMA).  tv: the kind-0 input, whose t / data fields point at the outputs.
__global__ void __launch_bounds__(TR_THREADS) k_ellipse_apply(const TableDesc *tabs, const double *ell) {
    __shared__ float s_v[TR_ROWS * TR_PITCH];
    __shared__ double s_e[NCHAN][4];
    const TableView &tv = tabs[blockIdx.y].tv;
    const long long n = tv.n, r0 = (long long)blockIdx.x * TR_ROWS;
    if (r0 >= n) return;
    const int nr = (int)min((long long)TR_ROWS, n - r0);
    if (threadIdx.x < NCHAN) {
        const double *e = ell + ((size_t)blockIdx.y * NCHAN + threadIdx.x) * ELL_STRIDE;
        s_e[threadIdx.x][0] = e[0];
        s_e[threadIdx.x][1] = e[1];
        s_e[threadIdx.x][2] = e[4];
        s_e[threadIdx.x][3] = e[5];
    }
    load_volt_tile(tv, r0, nr, s_v);
    if ((int)threadIdx.x < nr) const_cast<double *>(tv.t)[r0 + threadIdx.x] = row_time(tv, r0 + threadIdx.x);
    __syncthreads();
    double2 *data = const_cast<double2 *>(tv.data);
    for (int i = threadIdx.x; i < NCHAN * TR_ROWS; i += TR_THREADS) {
        const int ch = i / TR_ROWS, r = i - ch * TR_ROWS;
        if (r >= nr) continue;
        const double x = (double)s_v[r * TR_PITCH + 2 * ch], y = (double)s_v[r * TR_PITCH + 2 * ch + 1];
        const double xp = __dsub_rn(x, s_e[ch][0]);
        const double yp = __dadd_rn(__dmul_rn(s_e[ch][2], xp), __dmul_rn(s_e[ch][3], __dsub_rn(y, s_e[ch][1])));
        data[(long long)ch * n + r0 + r] = make_double2(xp, yp);
    }
}

void launch_ellipse_apply(const Launcher &L, const TableDesc *d_tabs, int ntables, long long max_rows,
                          const double *d_ell) {
    const dim3 grid((unsigned)((max_rows + TR_ROWS - 1) / TR_ROWS), ntables);
    k_ellipse_apply<<<grid, TR_THREADS, 0, L.stream>>>(d_tabs, d_ell);
    *L.counter += 1;
}

// demodulated out[40][n] complex128 -> float32 VOLT rows (ov): 80 floats = the 40 channels,
// or with keepraw 144 = the 80 raw input floats (bits copied) then the 32 diode channels;
// rounding to nearest (Float32.(...)), in the byte order of ov.
template <bool KEEPRAW>
__global__ void __launch_bounds__(TR_THREADS) k_repack_arrays(const TableDesc *tabs) {
    constexpr int NCH = KEEPRAW ? NDIODE : NCHAN, W = KEEPRAW ? 144 : 80;
    __shared__ float s_o[TR_ROWS * TR_PITCH];
    const TableDesc &tb = tabs[blockIdx.y];
    const long long n = tb.tv.n, r0 = (long long)blockIdx.x * TR_ROWS;
    if (r0 >= n) return;
    const int nr = (int)min((long long)TR_ROWS, n - r0);
    const double2 *out = tb.ov.out;
    for (int i = threadIdx.x; i < NCH * TR_ROWS; i += TR_THREADS) {
        const int ch = i / TR_ROWS, r = i - ch * TR_ROWS;
        if (r >= nr) continue;
        const double2 o = __ldg(out + (long long)ch * n + r0 + r);
        s_o[r * TR_PITCH + 2 * ch] = __double2float_rn(o.x);
        s_o[r * TR_PITCH + 2 * ch + 1] = __double2float_rn(o.y);
    }
    __syncthreads();
    const int be = tb.ov.big_endian;
    for (int i = threadIdx.x; i < nr * W; i += TR_THREADS) {
        const int r = i / W, j = i - r * W;
        uint32_t *row = reinterpret_cast<uint32_t *>(reinterpret_cast<char *>(tb.ov.volt) + (r0 + r) * tb.ov.volt_stride);
        if (KEEPRAW && j < 80) {
            row[j] = __ldg(reinterpret_cast<const uint32_t *>(reinterpret_cast<const char *>(tb.tv.volt) +
                                                              (r0 + r) * tb.tv.volt_stride) + j);
        } else {
            store_f32(reinterpret_cast<float *>(row + j), s_o[r * TR_PITCH + (j - (KEEPRAW ? 80 : 0))], be);
        }
    }
}

void launch_repack_arrays(const Launcher &L, const TableDesc *d_tabs, int ntables, long long max_rows, bool keepraw) {
    const dim3 grid((unsigned)((max_rows + TR_ROWS - 1) / TR_ROWS), ntables);
    if (keepraw) k_repack_arrays<true><<<grid, TR_THREADS, 0, L.stream>>>(d_tabs);
    else k_repack_arrays<false><<<grid, TR_THREADS, 0, L.stream>>>(d_tabs);
    *L.counter += 1;
}

}  // namespace gppd
