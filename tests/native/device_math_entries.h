// One extern "C" entry point per device math primitive of csrc/fit_math.cuh and
// csrc/gppd_device.cuh, applied element by element to host arrays.  Included by
// device_math.cu (nvcc: one kernel launch per call) and device_math_host.cpp (g++: a loop),
// which each define Stage:
//   in(p, n) / out(p, n)  the array the element functions see for host array p of n elements
//   run(f, n)             f(i) for i = 0 .. n-1, then the outputs back in the host arrays;
//                         returns 0 or a CUDA error code
// so both builds run the same element functions on the same inputs.
#pragma once

namespace dm {

// which: 0 sincos_large, 1 sincos_moderate, 2 sincos_demod
struct SinCosOp {
    int which;
    const double *x;
    double *s, *c;
    __device__ void operator()(long long i) const {
        if (which == 0) gppd::sincos_large(x[i], s + i, c + i);
        else if (which == 1) gppd::sincos_moderate(x[i], s + i, c + i);
        else gppd::sincos_demod(x[i], s + i, c + i);
    }
};

struct FcPhasorOp {
    const double *x, *y;
    double *px, *py;
    __device__ void operator()(long long i) const {
        const double2 p = gppd::fc_phasor(make_double2(x[i], y[i]));
        px[i] = p.x;
        py[i] = p.y;
    }
};

// make_phaseq (hence phase_quantum) of (phi, thmin, thmax); sin_arg of the row theta with
// the row's basis from sincos_large (as k_basis makes it), once with the job's PhaseQ and
// once with uniform = 0 (the per-row branch)
struct PhaseOp {
    const double *theta, *phi, *thmin, *thmax;
    double *q, *cq, *sq, *s_job, *s_row;
    int *uniform;
    __device__ void operator()(long long i) const {
        gppd::PhaseQ pq = gppd::make_phaseq(phi[i], thmin[i], thmax[i]);
        double sn, cs;
        gppd::sincos_large(theta[i], &sn, &cs);
        const double2 sc = make_double2(sn, cs);
        q[i] = pq.q;
        cq[i] = pq.cq;
        sq[i] = pq.sq;
        uniform[i] = pq.uniform;
        s_job[i] = gppd::sin_arg(pq, phi[i], theta[i], sc);
        pq.uniform = 0;
        s_row[i] = gppd::sin_arg(pq, phi[i], theta[i], sc);
    }
};

// J[25 i + k] = J_k(b[i]), k = 0..HK
struct BesselOp {
    const double *b;
    double *J;
    __device__ void operator()(long long i) const { gppd::bessel_j(b[i], J + (gppd::HK + 1) * i); }
};
// one element per (b, lane): J[25 i + lane] = bessel_j_lane(b[i], lane)
struct BesselLaneOp {
    const double *b;
    double *J;
    __device__ void operator()(long long e) const {
        const long long i = e / (gppd::HK + 1);
        const int lane = (int)(e % (gppd::HK + 1));
        J[e] = gppd::bessel_j_lane(b[i], lane);
    }
};

// row_time / row_theta of a METROLOGY table (kind 0) with int32 TIME in either byte order
struct RowTimeOp {
    gppd::TableView tv;
    double *t, *theta;
    __device__ void operator()(long long i) const {
        t[i] = gppd::row_time(tv, i);
        theta[i] = gppd::row_theta(tv, i);
    }
};

}  // namespace dm

extern "C" {

static int dm_sincos(int which, const double *x, double *s, double *c, long long n) {
    Stage st;
    return st.run(dm::SinCosOp{which, st.in(x, n), st.out(s, n), st.out(c, n)}, n);
}
int dm_sincos_large(const double *x, double *s, double *c, long long n) { return dm_sincos(0, x, s, c, n); }
int dm_sincos_moderate(const double *x, double *s, double *c, long long n) { return dm_sincos(1, x, s, c, n); }
int dm_sincos_demod(const double *x, double *s, double *c, long long n) { return dm_sincos(2, x, s, c, n); }

int dm_fc_phasor(const double *x, const double *y, double *px, double *py, long long n) {
    Stage st;
    return st.run(dm::FcPhasorOp{st.in(x, n), st.in(y, n), st.out(px, n), st.out(py, n)}, n);
}

int dm_phase(const double *theta, const double *phi, const double *thmin, const double *thmax,
             double *q, double *cq, double *sq, int *uniform, double *s_job, double *s_row, long long n) {
    Stage st;
    dm::PhaseOp op;
    op.theta = st.in(theta, n);
    op.phi = st.in(phi, n);
    op.thmin = st.in(thmin, n);
    op.thmax = st.in(thmax, n);
    op.q = st.out(q, n);
    op.cq = st.out(cq, n);
    op.sq = st.out(sq, n);
    op.uniform = st.out(uniform, n);
    op.s_job = st.out(s_job, n);
    op.s_row = st.out(s_row, n);
    return st.run(op, n);
}

int dm_bessel_j(const double *b, double *J, long long n) {
    Stage st;
    return st.run(dm::BesselOp{st.in(b, n), st.out(J, (gppd::HK + 1) * n)}, n);
}
int dm_bessel_j_lane(const double *b, double *J, long long n) {
    Stage st;
    return st.run(dm::BesselLaneOp{st.in(b, n), st.out(J, (gppd::HK + 1) * n)}, (gppd::HK + 1) * n);
}

int dm_row_time(const int32_t *time_us, int big_endian, double tmjd, double *t, double *theta, long long n) {
    Stage st;
    gppd::TableView tv = {};
    tv.kind = 0;
    tv.big_endian = big_endian;
    tv.n = n;
    tv.time_us = st.in(time_us, n);
    tv.time_stride = 4;
    tv.tmjd = tmjd;
    return st.run(dm::RowTimeOp{tv, st.out(t, n), st.out(theta, n)}, n);
}

}  // extern "C"
