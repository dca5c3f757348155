// fit_math.cuh -- arithmetic shared by the fit evaluators: closed-form linear
// parameters and chi2 from the reduced sums (reference src/Modulation.jl:140-145,
// :174-215, :325), Bessel coefficients for the Jacobi-Anger evaluator, and the
// per-state (mean, weight) lookup (reference src/Faint.jl:89-100).
#pragma once
#include "gppd_device.cuh"

namespace gppd {

// Constant (b, phi independent) sums of one fit.
struct FitConsts {
    double sw, sdd, sgg;   // sum w, sum w|d-mu|^2, sum w |p|^2
    double sdr, sdi;       // sum w (d - mu)
    double mur, mui;       // reference point mu (fitoffsets only), else 0
    double nvalid;
};

// Linear parameters and chi2 from the sums.  With g = p e (p = power * FCphasor,
// e = exp(j b sin(.))):  S_gd = sum w conj(g) (d - mu),  S_g = sum w g.
//   no offsets:  a = S_gd / S_gg,                         chi2 N = S_dd - |S_gd|^2 / S_gg
//   offsets:     [S_w  S_g; conj(S_g)  S_gg] [c'; a] = [S_d'; S_gd]  (Cramer, like the
//                reference's StaticArrays 2x2 solve), c = c' + mu,
//                chi2 N = S_dd - Re(conj(c') S_d' + conj(a) S_gd)
// which is sum w |c + a g - d|^2 at the least-squares (c, a) (reference :325).
__device__ __forceinline__ double solve_linear(const FitConsts &k, bool offs, double sgdr,
                                               double sgdi, double sgr, double sgi, double &cre,
                                               double &cim, double &are, double &aim) {
    if (!offs) {
        are = sgdr / k.sgg;
        aim = sgdi / k.sgg;
        cre = 0.0;
        cim = 0.0;
        double num = fma(sgdr, sgdr, sgdi * sgdi);
        return (k.sdd - num / k.sgg) / k.nvalid;
    }
    double det = fma(k.sw, k.sgg, -fma(sgr, sgr, sgi * sgi));
    double t1r = fma(sgr, sgdr, -(sgi * sgdi)), t1i = fma(sgr, sgdi, sgi * sgdr);
    double cpr = (k.sgg * k.sdr - t1r) / det, cpi = (k.sgg * k.sdi - t1i) / det;
    double t2r = fma(sgr, k.sdr, sgi * k.sdi), t2i = fma(sgr, k.sdi, -(sgi * k.sdr));
    are = (k.sw * sgdr - t2r) / det;
    aim = (k.sw * sgdi - t2i) / det;
    cre = cpr + k.mur;
    cim = cpi + k.mui;
    double proj = fma(cpr, k.sdr, cpi * k.sdi) + fma(are, sgdr, aim * sgdi);
    return (k.sdd - proj) / k.nvalid;
}

// J_0(b) .. J_HK(b) by Miller's backward recurrence J_{k-1} = (2k/b) J_k - J_{k+1}
// from k = BESSEL_M = 40 (far in the decaying region for |b| <= HARM_BMAX: the
// result is within 2.3e-16 absolute of the true values, as with any higher start),
// normalised with J_0 + 2 sum J_{2k} = 1.  Valid for either sign of b.  The
// recurrence grows like (2k/b)^k, so |b| < 1e-4 uses the first terms of the power
// series instead (the rest is below 1e-19).
constexpr int BESSEL_M = 40;
constexpr double BESSEL_TINY = 1.0e-4;

// value for order k of the tiny-|b| series, x = b/2
__device__ __forceinline__ double bessel_tiny(double b, int k) {
    const double x = 0.5 * b, x2 = x * x;
    if (k == 0) return 1.0 - x2;
    if (k == 1) return x * (1.0 - 0.5 * x2);
    if (k == 2) return 0.5 * x2;
    if (k == 3) return x2 * x * (1.0 / 6.0);
    return 0.0;
}

// Two recurrence steps (k even -> orders k-1 and k-2), shared by both evaluators.
#define GPPD_BESSEL_STEP2(k, kd, tb, jp, jc, seven, ON_ODD, ON_EVEN)   \
    {                                                                  \
        const double j1 = fma((kd) * (tb), jc, -(jp)); /* J_{k-1} */   \
        const double j0 = fma(((kd) - 1.0) * (tb), j1, -(jc)); /* J_{k-2} */ \
        ON_ODD(k - 1, j1);                                             \
        ON_EVEN(k - 2, j0);                                            \
        jp = j1;                                                       \
        jc = j0;                                                       \
        if (k - 2 > 0) seven += j0;                                    \
        kd -= 2.0;                                                     \
    }

__device__ __forceinline__ void bessel_j(double b, double *J) {
    if (fabs(b) < BESSEL_TINY) {
#pragma unroll
        for (int k = 0; k <= HK; ++k) J[k] = bessel_tiny(b, k);
        return;
    }
    const double tb = 2.0 / b;
    double jp = 0.0, jc = 1.0e-280, seven = 0.0, kd = (double)BESSEL_M;
#define GPPD_STORE(kk, v) if ((kk) <= HK) J[kk] = (v)
#pragma unroll
    for (int k = BESSEL_M; k >= 2; k -= 2) GPPD_BESSEL_STEP2(k, kd, tb, jp, jc, seven, GPPD_STORE, GPPD_STORE)
#undef GPPD_STORE
    const double inv = 1.0 / (jc + 2.0 * seven);   // jc = J_0
#pragma unroll
    for (int k = 0; k <= HK; ++k) J[k] *= inv;
}

// J_lane(b) for lane <= HK: every lane of a warp runs the same recurrence (uniform
// control flow, no array) and keeps the term of its own order.
__device__ __forceinline__ double bessel_j_lane(double b, int lane) {
    if (fabs(b) < BESSEL_TINY) return bessel_tiny(b, lane);
    const double tb = 2.0 / b;
    double jp = 0.0, jc = 1.0e-280, seven = 0.0, kd = (double)BESSEL_M, mine = 0.0;
#define GPPD_KEEP(kk, v) if ((kk) == lane) mine = (v)
#pragma unroll 4
    for (int k = BESSEL_M; k >= 2; k -= 2) GPPD_BESSEL_STEP2(k, kd, tb, jp, jc, seven, GPPD_KEEP, GPPD_KEEP)
#undef GPPD_KEEP
    return mine * (1.0 / (jc + 2.0 * seven));
}

// sin and cos of a moderate argument (|x| < 1e5), relative error below 2^-52 (at most 1.5 ulp,
// where the reduced argument is near +-pi/4) and, near the zeros of sin and cos, absolute error
// below 2^-52 |result| + 1e-28 (|k| |pi/2 - hi - lo| < 63 662 * 1.5e-33): two-constant Cody-Waite
// reduction by pi/2 with FMAs (exact first step) and the fdlibm kernel polynomials in
// Horner/FMA form.  About a third of the instructions of the general-purpose
// sincos(), which carries a Payne-Hanek path.  Every operation is an explicit fma or
// a single multiply, so the result does not depend on the -fmad setting.  The
// coefficients live in constant memory: as literals every one of them costs two
// extra (uniform-register move) instructions per use.
__constant__ double c_sincos[16] = {
    6.36619772367581382433e-01,   // 0: 2/pi
    1.57079632679489655800e+00,   // 1: pi/2, high part
    6.12323399573676603587e-17,   // 2: pi/2, low part
    1.58969099521155010221e-10,   // 3: S6
    -2.50507602534068634195e-08,  // 4: S5
    2.75573137070700676789e-06,   // 5: S4
    -1.98412698298579493134e-04,  // 6: S3
    8.33333333332248946124e-03,   // 7: S2
    -1.66666666666666324348e-01,  // 8: S1
    -1.13596475577881948265e-11,  // 9: C6
    2.08757232129817482790e-09,   // 10: C5
    -2.75573143513906633035e-07,  // 11: C4
    2.48015872894767294178e-05,   // 12: C3
    -1.38888888888741095749e-03,  // 13: C2
    4.16666666666666019037e-02,   // 14: C1
    0.0};

__device__ __forceinline__ void sincos_moderate(double x, double *sn, double *cs) {
    if (!(fabs(x) < 1.0e5)) {
        sincos(x, sn, cs);
        return;
    }
    const double fn = rint(x * c_sincos[0]);
    const int k = (int)fn;
    double r = fma(-fn, c_sincos[1], x);
    r = fma(-fn, c_sincos[2], r);
    const double z = r * r;
    double ps = fma(z, c_sincos[3], c_sincos[4]);
    ps = fma(z, ps, c_sincos[5]);
    ps = fma(z, ps, c_sincos[6]);
    ps = fma(z, ps, c_sincos[7]);
    ps = fma(z, ps, c_sincos[8]);
    const double ks = fma(z * r, ps, r);
    double pc = fma(z, c_sincos[9], c_sincos[10]);
    pc = fma(z, pc, c_sincos[11]);
    pc = fma(z, pc, c_sincos[12]);
    pc = fma(z, pc, c_sincos[13]);
    pc = fma(z, pc, c_sincos[14]);
    pc = fma(z, pc, -0.5);
    const double kc = fma(z, pc, 1.0);
    // quadrant: swap for odd k, then flip signs through the high words
    const bool odd = k & 1;
    const double s0 = odd ? kc : ks, c0 = odd ? ks : kc;
    const int sflip = (k & 2) << 30, cflip = ((k + 1) & 2) << 30;
    *sn = __hiloint2double(__double2hiint(s0) ^ sflip, __double2loint(s0));
    *cs = __hiloint2double(__double2hiint(c0) ^ cflip, __double2loint(c0));
}

// sin and cos of the demodulation phase psi for the float32 table path: |error| < 2e-10,
// i.e. 2^-32 -- the result is rounded to float32 (2^-24) right after, so a full-precision
// double sincos would buy nothing.  psi = b sin(.) is a few radians at most: one-constant
// Cody-Waite reduction by pi/2 (the quotient through the 1.5 * 2^52 rounding trick: no
// conversion instruction, the XU pipe issues one warp instruction every 8 cycles) and the
// leading terms of the fdlibm kernel polynomials.
// The caller guarantees |x| < 1e4 (|psi| <= |b|: checked once per fit, not per row).
__device__ __forceinline__ void sincos_demod(double x, double *sn, double *cs) {
    const double t = fma(x, c_sincos[0], 6755399441055744.0);      // 1.5 * 2^52: low word = rint(x 2/pi)
    const int k = __double2loint(t);
    const double fn = t - 6755399441055744.0;
    const double r = fma(-fn, c_sincos[1], x);                     // |fn| pi/2_lo < 1e-12
    const double z = r * r;
    double ps = fma(z, c_sincos[4], c_sincos[5]);                  // S5, S4
    ps = fma(z, ps, c_sincos[6]);
    ps = fma(z, ps, c_sincos[7]);
    ps = fma(z, ps, c_sincos[8]);
    const double ks = fma(z * r, ps, r);
    double pc = fma(z, c_sincos[11], c_sincos[12]);                // C4, C3
    pc = fma(z, pc, c_sincos[13]);
    pc = fma(z, pc, c_sincos[14]);
    pc = fma(z, pc, -0.5);
    const double kc = fma(z, pc, 1.0);
    const bool odd = k & 1;
    const double s0 = odd ? kc : ks, c0 = odd ? ks : kc;
    const int sflip = (k & 2) << 30, cflip = ((k + 1) & 2) << 30;
    *sn = __hiloint2double(__double2hiint(s0) ^ sflip, __double2loint(s0));
    *cs = __hiloint2double(__double2hiint(c0) ^ cflip, __double2loint(c0));
}

// sin and cos of theta = fl(omega t) ~ 3e10 (any |x| < 2^40): two-constant Cody-Waite
// reduction by 2 pi done with FMAs.  k = rint(x / 2 pi) < 2^38 and x is a multiple of
// its ulp >= 2^-13... so x - k * fl(2 pi) is a multiple of 2^-50 below 8 in magnitude:
// the first FMA is exact, the second rounds once; the reduced argument is within one
// ulp of x mod 2 pi.  The general-purpose sincos() spends ~300 instructions on its
// Payne-Hanek path for such arguments.
__device__ __forceinline__ void sincos_large(double x, double *sn, double *cs) {
    if (!(fabs(x) < 1.099511627776e12)) {   // 2^40
        sincos(x, sn, cs);
        return;
    }
    const double k = rint(x * 1.59154943091895345554e-01);          // 1 / (2 pi)
    double r = fma(-k, 6.28318530717958623200e+00, x);               // fl(2 pi)
    r = fma(-k, 2.44929359829470641435e-16, r);                      // 2 pi - fl(2 pi)
    sincos_moderate(r, sn, cs);
}

// Per-state statistics of one (job, group) (reference compute_mean_var_power,
// src/Faint.jl:89-100): the statistics pass leaves, per (job, group), a table of 16
// (mean |d|, weight = 1 / var |d|) pairs indexed [diode * 4 + state].
//   part[(jg*P + p)*STATS_VALS + ...]: per FIXED segment of STATS_SEG_ROWS rows,
//       [0..3] row count per state, [4..19] sum (|d| - pivot), [20..35] sum (|d| - pivot)^2
//       per (diode, state); the pivot is |d| at the job's first row of the state
//   table[jg*16 + diode*4 + state] = (mean, weight), segments added in index order,
// so the values are deterministic and independent of the batch the job is in.
constexpr int STATS_SEG_ROWS = 1024;
__host__ __device__ inline int stats_segments(long long nrows) {
    return (int)((nrows + STATS_SEG_ROWS - 1) / STATS_SEG_ROWS);
}
__device__ __forceinline__ double2 stats_mean_weight(const double *table, int jg, int dio, int st) {
    return reinterpret_cast<const double2 *>(table)[jg * 16 + dio * 4 + st];
}

}  // namespace gppd
