"""The device math primitives every kernel is built on (csrc/fit_math.cuh,
csrc/gppd_device.cuh), each on its own against a high-precision reference: mpmath at 50
digits, exact rationals, or numpy float64 where the primitive is a fixed sequence of IEEE
operations.  The pipeline tests cannot see their errors (1e-9 parameter parity, float32
output, tensor-core sums held to the DMMA kernel's), so the bounds the code's comments state
are checked here, at the edges of every range.

Three builds of the same headers (tests/native): g++ -ffp-contract=off (CPU tests) and nvcc
with the library's flags, -fmad=true and -fmad=false (GPU tests).  On the GPU the builds must
also agree bit for bit wherever the arithmetic is explicit, and sqrt4 must be sqrt().
The end-to-end test at the bottom runs demodulateall with FC channels of extreme magnitude."""
import ctypes as C
import functools
import os
import shutil
import subprocess
from fractions import Fraction

import mpmath as mp
import numpy as np
import pytest

from fitref import MIN_COINCIDE, compare_fits

mp.mp.dps = 50

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "gppupildemodulation.jl_b200", "csrc")
NATIVE = os.path.join(ROOT, "tests", "native")
BUILD = os.path.join(NATIVE, "build")
_NVCC = shutil.which("nvcc")
CUDA_HOME = os.environ.get("CUDA_HOME") or (os.path.dirname(os.path.dirname(_NVCC)) if _NVCC else "/usr/local/cuda")
HEADERS = [os.path.join(CSRC, "fit_math.cuh"), os.path.join(CSRC, "gppd_device.cuh"),
           os.path.join(NATIVE, "device_math_entries.h"), os.path.join(NATIVE, "cuda_host_shim.h")]

TWO52, TWO51 = 2.0 ** -52, 2.0 ** -51
HK = 24
HARM_BMAX = 5.0


def _build(out, src, cmd):
    """(re)build ``out`` from ``src`` when it is missing or older than a source or header"""
    if not os.path.exists(out) or os.path.getmtime(out) < max(os.path.getmtime(p) for p in HEADERS + [src]):
        os.makedirs(BUILD, exist_ok=True)
        tmp = out + ".tmp%d" % os.getpid()
        subprocess.run(cmd + ["-o", tmp, src], check=True)
        os.replace(tmp, out)
    return out


@functools.lru_cache(maxsize=None)
def _lib(kind):
    """kind: 'host' (g++), 'fmad' / 'nofmad' (nvcc -fmad=true / false, sm_100a)"""
    if kind == "host":
        path = _build(os.path.join(BUILD, "libdevice_math_host.so"), os.path.join(NATIVE, "device_math_host.cpp"),
                      ["g++", "-O2", "-fPIC", "-shared", "-ffp-contract=off",
                       "-I", os.path.join(CUDA_HOME, "include"), "-I", CSRC])
    else:
        nvcc = _NVCC or os.path.join(CUDA_HOME, "bin", "nvcc")
        path = _build(os.path.join(BUILD, "libdevice_math_%s.so" % kind), os.path.join(NATIVE, "device_math.cu"),
                      [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17",
                       "-Xcompiler", "-fPIC,-ffp-contract=off", "-fmad=%s" % ("true" if kind == "fmad" else "false"),
                       "-shared", "-I", CSRC])
    return Prims(C.CDLL(path), kind)


_dp, _ip, _i32p = C.POINTER(C.c_double), C.POINTER(C.c_int), C.POINTER(C.c_int32)


def _p(a, typ=_dp):
    return a.ctypes.data_as(typ)


def _f64(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64).ravel())


class Prims:
    """The entry points of one build over numpy arrays."""

    def __init__(self, lib, kind):
        self.lib, self.kind = lib, kind

    def _call(self, name, *args):
        rc = getattr(self.lib, name)(*args)
        assert rc == 0, "%s: CUDA error %d" % (name, rc)

    def sincos(self, which, x):
        x = _f64(x)
        s, c = np.empty_like(x), np.empty_like(x)
        self._call("dm_sincos_" + which, _p(x), _p(s), _p(c), C.c_longlong(x.size))
        return s, c

    def fc_phasor(self, x, y):
        x, y = _f64(x), _f64(y)
        px, py = np.empty_like(x), np.empty_like(x)
        self._call("dm_fc_phasor", _p(x), _p(y), _p(px), _p(py), C.c_longlong(x.size))
        return px, py

    def phase(self, theta, phi, thmin, thmax):
        theta, phi, thmin, thmax = (_f64(v) for v in np.broadcast_arrays(theta, phi, thmin, thmax))
        n = theta.size
        r = {k: np.empty(n) for k in ("q", "cq", "sq", "s_job", "s_row")}
        r["uniform"] = np.empty(n, dtype=np.int32)
        self._call("dm_phase", _p(theta), _p(phi), _p(thmin), _p(thmax), _p(r["q"]), _p(r["cq"]), _p(r["sq"]),
                   _p(r["uniform"], _ip), _p(r["s_job"]), _p(r["s_row"]), C.c_longlong(n))
        return r

    def bessel(self, b, lane=False):
        b = _f64(b)
        J = np.empty((b.size, HK + 1))
        self._call("dm_bessel_j_lane" if lane else "dm_bessel_j", _p(b), _p(J), C.c_longlong(b.size))
        return J

    def row_time(self, time_us, big_endian, tmjd):
        raw = np.ascontiguousarray(np.asarray(time_us, dtype=">i4" if big_endian else "<i4")).view(np.int32)
        t, th = np.empty(raw.size), np.empty(raw.size)
        self._call("dm_row_time", _p(raw, _i32p), C.c_int(int(big_endian)), C.c_double(tmjd), _p(t), _p(th),
                   C.c_longlong(raw.size))
        return t, th

    def sqrt4(self, h):
        h = _f64(h)
        assert h.size % 4 == 0
        r = np.empty_like(h)
        self._call("dm_sqrt4", _p(h), _p(r), C.c_longlong(h.size))
        return r

    def sqrt(self, h):
        h = _f64(h)
        r = np.empty_like(h)
        self._call("dm_sqrt", _p(h), _p(r), C.c_longlong(h.size))
        return r


BUILDS = ["host", pytest.param("fmad", marks=pytest.mark.gpu), pytest.param("nofmad", marks=pytest.mark.gpu)]


@pytest.fixture(scope="module", params=BUILDS)
def prims(request):
    return _lib(request.param)


@pytest.fixture(scope="module")
def host():
    return _lib("host")


@pytest.fixture(scope="module")
def dev():
    return _lib("fmad"), _lib("nofmad")


def same_bits(a, b):
    """bitwise equality; any NaN equals any NaN (its sign and payload are not specified)"""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    nan = np.isnan(a) & np.isnan(b)
    return nan | (a.view(np.int64) == b.view(np.int64))


def assert_same_bits(a, b, what=""):
    ok = same_bits(a, b)
    if not ok.all():
        i = np.flatnonzero(~ok)[:5]
        raise AssertionError("%s: %d values differ, e.g. %s vs %s" % (what, (~ok).sum(), np.asarray(a).ravel()[i],
                                                                      np.asarray(b).ravel()[i]))


def mp_err(got, ref):
    """|got - ref| as a float64, ref an mpf"""
    return float(abs(mp.mpf(float(got)) - ref))


def neighbours(v, k=1):
    """v and its k nearest doubles on each side"""
    v = np.asarray(v, dtype=np.float64).ravel()
    out = [v]
    lo = hi = v
    for _ in range(k):
        lo, hi = np.nextafter(lo, -np.inf), np.nextafter(hi, np.inf)
        out += [lo, hi]
    return np.concatenate(out)


def nearest_multiples(unit, ks):
    """the doubles nearest k * unit (unit an mpf), k in ks"""
    return np.array([float(mp.mpf(int(k)) * unit) for k in ks])


SPECIALS = np.array([0.0, -0.0, np.inf, -np.inf, np.nan])


def check_sincos_bound(x, s, c, bound, what):
    """bound(ref) -> allowed |error| for each of sin, cos (finite x); non-finite x gives NaN"""
    worst = 0.0
    for xi, si, ci in zip(x, s, c):
        if not np.isfinite(xi):
            assert np.isnan(si) and np.isnan(ci), (what, xi, si, ci)
            continue
        X = mp.mpf(float(xi))
        for got, ref in ((si, mp.sin(X)), (ci, mp.cos(X))):
            e = mp_err(got, ref)
            lim = bound(ref)
            assert e <= lim, "%s: x = %r: got %r, error %.3g > %.3g" % (what, float(xi), float(got), e, lim)
            worst = max(worst, e / lim)
    return worst


# ---- sincos_large --------------------------------------------------------------------

def large_inputs():
    rng = np.random.default_rng(11)
    # theta as the product builds it: fl(OMEGA * fl(fl(TIME * 1e-6) + fl(86400 * MJD)))
    mjd = rng.uniform(50_000, 70_000, 3000)
    mjd[:20] = np.round(mjd[:20])
    time_us = rng.integers(-2 ** 31, 2 ** 31, mjd.size)
    time_us[:4] = [-2 ** 31, -1, 0, 2 ** 31 - 1]
    theta = 6.283185 * (time_us.astype(np.float64) * 1e-6 + 86400.0 * mjd)
    # the doubles nearest k pi/2 and k 2 pi over that range, and their neighbours
    kq = rng.integers(int(2.6e10 / (np.pi / 2)), int(3.9e10 / (np.pi / 2)), 300)
    kf = rng.integers(int(2.6e10 / (2 * np.pi)), int(3.9e10 / (2 * np.pi)), 300)
    adv = neighbours(np.concatenate([nearest_multiples(mp.pi / 2, kq), nearest_multiples(2 * mp.pi, kf)]))
    # relative timestamps: negative and small theta, and exact multiples near zero
    small = np.concatenate([rng.uniform(-100, 100, 500), rng.uniform(-1e6, 1e6, 500), -theta[:300],
                            neighbours(nearest_multiples(mp.pi / 2, np.arange(-40, 41)))])
    # both sides of the switch to sincos() at 2^40
    edge = neighbours(np.array([2.0 ** 40, -2.0 ** 40]), 2)
    return np.concatenate([theta, adv, small, edge, rng.uniform(2 ** 39, 2 ** 41, 200), SPECIALS])


def test_sincos_large_reference(prims):
    """|sincos_large(x) - (sin x, cos x)| <= 2^-51 for theta over MJD 50 000-70 000 and the whole
    int32 TIME range, the doubles nearest multiples of pi/2 and 2 pi, relative timestamps, both
    sides of 2^40 (beyond it sincos()), and non-finite x -> NaN"""
    x = large_inputs()
    s, c = prims.sincos("large", x)
    check_sincos_bound(x, s, c, lambda ref: TWO51, "sincos_large")


# ---- sincos_moderate -----------------------------------------------------------------

def moderate_bound(ref):
    # relative 2^-52 (1.5 ulp at most, near r = +-pi/4), and near the zeros of sin and cos the
    # error of the reduced argument: |k| |pi/2 - hi - lo| < 63 662 * 1.5e-33 < 1e-28
    return TWO52 * abs(ref) + 1e-28


def moderate_inputs():
    rng = np.random.default_rng(12)
    kmax = 63_662                               # |k pi/2| < 1e5
    kq = np.concatenate([np.arange(-400, 401), rng.integers(-kmax, kmax + 1, 1500), [-kmax, kmax]])
    k4 = np.concatenate([np.arange(-400, 401), rng.integers(-kmax, kmax + 1, 1500)])
    mult = neighbours(np.concatenate([nearest_multiples(mp.pi / 2, kq), nearest_multiples(mp.pi / 4, k4)]))
    mult = mult[np.abs(mult) < 1e5]
    rnd = np.concatenate([rng.uniform(-1e5, 1e5, 4000), rng.uniform(-8, 8, 2000),
                          np.ldexp(rng.uniform(-1, 1, 500), rng.integers(-1074, 0, 500))])
    return np.concatenate([mult, rnd, neighbours(np.array([1e5, -1e5]), 2), SPECIALS])


def test_sincos_moderate_reference(prims):
    """|sincos_moderate(x) - (sin x, cos x)| <= 2^-52 |sin x| + 1e-28 for |x| < 1e5: random x,
    the doubles nearest k pi/2 and k pi/4 for |k| up to 63 662 and their neighbours, tiny x;
    beyond 1e5 sincos() takes over (2 ulp); non-finite x -> NaN"""
    x = moderate_inputs()
    s, c = prims.sincos("moderate", x)
    inside = np.abs(x) < 1e5
    check_sincos_bound(x[inside], s[inside], c[inside], moderate_bound, "sincos_moderate")
    check_sincos_bound(x[~inside], s[~inside], c[~inside],
                       lambda ref: 2 * np.spacing(abs(float(ref))), "sincos() beyond 1e5")


# ---- sincos_demod --------------------------------------------------------------------

def demod_inputs():
    rng = np.random.default_rng(13)
    k = np.arange(-5730, 5731)                  # every quadrant boundary k pi/2 with |k pi/2| < 9e3
    bounds = neighbours(nearest_multiples(mp.pi / 2, k))
    bounds = np.concatenate([bounds, nearest_multiples(mp.pi / 4, 2 * k + 1)])
    return np.concatenate([bounds[np.abs(bounds) < 9e3], rng.uniform(-9e3, 9e3, 4000), rng.uniform(-4, 4, 2000),
                           [0.0, -0.0, 8999.999, -8999.999]])


def test_sincos_demod_reference(prims):
    """|sincos_demod(x) - (sin x, cos x)| <= 2e-10 for |x| < 9e3 (the caller's guard), both
    signs, every quadrant boundary and the midpoints between them, +-0"""
    x = demod_inputs()
    s, c = prims.sincos("demod", x)
    # float64 reference is enough at this bound; mpmath checks a sample below
    err = np.maximum(np.abs(s - np.sin(x)), np.abs(c - np.cos(x)))
    assert err.max() <= 2e-10 - 1e-15, (err.max(), x[np.argmax(err)])
    check_sincos_bound(x[::50], s[::50], c[::50], lambda ref: 2e-10, "sincos_demod")


# ---- fc_phasor -----------------------------------------------------------------------

def fc_inputs():
    rng = np.random.default_rng(14)
    ang = rng.uniform(-np.pi, np.pi, 2000)
    mag = 10.0 ** rng.uniform(-300, 300, ang.size)
    normal = np.stack([mag * np.cos(ang), mag * np.sin(ang)], 1)
    sub = 10.0 ** rng.uniform(-323, -308, (400, 2)) * rng.choice([-1.0, 1.0], (400, 2))
    low = 10.0 ** rng.uniform(-308, -299, (400, 2)) * rng.choice([-1.0, 1.0], (400, 2))
    huge = 10.0 ** rng.uniform(300, 308, (400, 2)) * rng.choice([-1.0, 1.0], (400, 2))
    big = np.finfo(float).max
    edges = [(1e-310, 0.0), (0.0, 1e-310), (1e-310, 1e-310), (-1e-310, 1e-320), (5e-324, -5e-324),
             (1e300, 0.0), (1e300, 1e300), (big, big), (big, -big), (-big, 1.0), (1e308, 1e308),
             (1.0, 1e-20), (-1.0, 1e-20), (-1.0, -1e-20), (3.0, 4.0)]
    zeros = [(x, y) for x in (0.0, -0.0) for y in (0.0, -0.0)]
    infs = [(x, y) for x in (np.inf, -np.inf, 1.0, -1.0, 0.0, -0.0) for y in (np.inf, -np.inf, 1.0, -1.0, 0.0, -0.0)
            if np.isinf(x) or np.isinf(y)]
    nans = [(np.nan, 1.0), (1.0, np.nan), (np.nan, np.nan), (np.inf, np.nan), (np.nan, -np.inf), (0.0, np.nan)]
    pts = np.concatenate([normal, sub, low, huge, np.array(edges + zeros + infs + nans)])
    return pts[:, 0].copy(), pts[:, 1].copy()


def fc_reference(x, y):
    """exp(1im * angle(x + 1im y)): for finite nonzero input the exact unit vector (x, y) / |(x, y)|;
    zeros and infinities through atan2's conventions ((-0, +0) -> angle pi -> (-1, 1.2e-16))"""
    if np.isfinite(x) and np.isfinite(y) and (x != 0 or y != 0):
        X, Y = mp.mpf(float(x)), mp.mpf(float(y))
        h = mp.sqrt(X * X + Y * Y)
        return X / h, Y / h
    a = mp.mpf(float(np.arctan2(y, x)))
    return mp.cos(a), mp.sin(a)


def test_fc_phasor_reference(prims):
    """fc_phasor within 2 ulp of the unit phasor (2^-51) plus 2 ulp of its angle (the atan2 branch
    rounds the angle, as the reference's angle() does) of exp(1im * angle(fc)): normal, subnormal
    (fc_phasor used to return Inf/NaN there), tiny, huge (x*x overflows), zero and infinite
    components; NaN in either component gives NaN"""
    x, y = fc_inputs()
    px, py = prims.fc_phasor(x, y)
    for xi, yi, gx, gy in zip(x, y, px, py):
        if np.isnan(xi) or np.isnan(yi):
            assert np.isnan(gx) and np.isnan(gy), (xi, yi, gx, gy)
            continue
        rx, ry = fc_reference(xi, yi)
        e = max(mp_err(gx, rx), mp_err(gy, ry))
        assert e <= TWO51 + 2 * np.spacing(abs(np.arctan2(yi, xi))), "fc_phasor(%r, %r) = (%r, %r), error %.3g" % (xi, yi, gx, gy, e)


def test_fc_phasor_signed_zeros(prims):
    """angle(0) conventions of atan2, as the reference's exp(1im*angle(fc))"""
    x = np.array([0.0, -0.0, 0.0, -0.0])
    y = np.array([0.0, 0.0, -0.0, -0.0])
    px, py = prims.fc_phasor(x, y)
    assert (px == [1.0, -1.0, 1.0, -1.0]).all()
    assert py[0] == 0.0 and py[2] == 0.0
    assert abs(py[1] - 1.2246467991473532e-16) <= 1e-31 and abs(py[3] + 1.2246467991473532e-16) <= 1e-31


def test_fc_phasor_normal_range_per_component(prims):
    """in the normal range the phasor is (x, y) / hypot(x, y): each component within a relative
    3 * 2^-52 of its own value, even the small one of a phasor next to an axis (hypot() is within
    2 ulp on the device, then one division and one multiplication round; 2.4 ulp seen there)"""
    rng = np.random.default_rng(15)
    ang = np.concatenate([rng.uniform(-np.pi, np.pi, 1000), [1e-20, np.pi - 1e-12, -np.pi / 2 + 1e-15]])
    mag = 10.0 ** rng.uniform(-290, 290, ang.size)
    x, y = mag * np.cos(ang), mag * np.sin(ang)
    px, py = prims.fc_phasor(x, y)
    for xi, yi, gx, gy in zip(x, y, px, py):
        rx, ry = fc_reference(xi, yi)
        for g, r in ((gx, rx), (gy, ry)):
            assert mp_err(g, r) <= 3 * TWO52 * (1 + TWO52) * abs(float(r)), (xi, yi, g, r)


# ---- phase_quantum / make_phaseq / sin_arg --------------------------------------------

def ulp_of(e_biased):
    return 2.0 ** (e_biased - 1023 - 52)


def phase_jobs():
    """(thmin, thmax, phi) triples at the edges of phase_quantum's conditions"""
    rng = np.random.default_rng(16)
    jobs = []
    # absolute timestamps: theta ~ 3e10 (binade [2^34, 2^35), ulp 2^-18), random phi, |phi| <= 10
    for _ in range(150):
        thmin = rng.uniform(2.0 ** 34, 2.0 ** 35 - 1e4)
        jobs.append((thmin, thmin + rng.uniform(0, 5e3), rng.uniform(-10, 10)))
    u = 2.0 ** -18
    base = 2.5e10
    for m in (-3, 0, 1, 7, 40):
        jobs.append((base, base + 0.01, (m + 0.5) * u))             # exact tie: uniform = 0
        jobs.append((base, base + 0.01, (m + 0.5) * u + u / 1024))  # not a tie
        jobs.append((base + u, base + 0.01, (m + 0.5) * u))         # tie, odd thmin
    jobs += [(base, base, 0.5 * u), (base + u, base + u, 0.5 * u), (base, base + u, -0.5 * u)]
    # ranges that straddle a binade, and phi that moves the ends across one
    e34 = 2.0 ** 34
    jobs += [(e34 - 10, e34 + 10, 0.3), (e34, e34 + 10, -1e-3), (e34 + 1e-3, e34 + 10, -2e-3),
             (e34, e34 + 100, 0.0), (2 * e34 - 10, 2 * e34 - 1, 9.5), (2 * e34 - 10, 2 * e34 - 1, 5.0)]
    # relative timestamps: small theta of every sign, thmin <= 0
    jobs += [(-5.0, 10.0, 0.7), (0.0, 3.0, 0.2), (-0.0, 3.0, 0.2), (1.0, 1.9, 0.3), (1.0, 1.9, -0.3),
             (100.0, 127.0, 1.0 / 3), (1e3, 1.5e3, -2.0)]
    # tiny theta: biased exponent <= 52 (the ulp grid would be subnormal)
    jobs += [(1e-300, 1.5e-300, 1e-310), (2.0 ** -975, 2.0 ** -975 * 1.5, 2.0 ** -1020),
             (2.0 ** -969, 2.0 ** -969 * 1.5, 2.0 ** -1015)]
    return jobs


def grid_points(thmin, thmax, rng, nmax=100_000):
    """every theta of [thmin, thmax] (one binade) when there are fewer than nmax, else a sample
    with both ends"""
    u = np.spacing(thmin)
    n = int(round((thmax - thmin) / u)) + 1
    if n <= nmax:
        return thmin + u * np.arange(n, dtype=np.float64)
    return np.concatenate([[thmin, thmax], thmin + u * rng.integers(0, n, 4000).astype(np.float64)])


def test_phase_quantum_uniform_is_exact(prims):
    """whenever make_phaseq says uniform, fl(theta + phi) - theta = q for thmin, thmax and every
    theta of the job's grid between them (a sample when there are 1e5 or more); an exact tie
    phi = (m + 1/2) ulp is never uniform"""
    rng = np.random.default_rng(17)
    jobs = phase_jobs()
    thmin = np.array([j[0] for j in jobs])
    thmax = np.array([j[1] for j in jobs])
    phi = np.array([j[2] for j in jobs])
    r = prims.phase(thmin, phi, thmin, thmax)
    n_uniform = 0
    for i, (a, b, p) in enumerate(jobs):
        if r["uniform"][i]:
            n_uniform += 1
            th = grid_points(a, b, rng)
            assert np.exp2(np.floor(np.log2(th))).min() == np.exp2(np.floor(np.log2(th))).max()
            dq = (th + p) - th
            assert (dq == r["q"][i]).all(), ("uniform but q varies", a, b, p, r["q"][i], np.unique(dq)[:4])
        ex = int(np.frexp(a)[1]) + 1022 if a > 0 else 0
        if a > 0 and ex > 0:
            rem = Fraction(p) / Fraction(ulp_of(ex))
            if rem.denominator == 2:
                assert not r["uniform"][i], ("tie taken as uniform", a, b, p)
    assert n_uniform >= 140


def test_phase_quantum_rejects(prims):
    """the cases phase_quantum must leave to the per-row branch"""
    e34 = 2.0 ** 34
    u = 2.0 ** -18
    cases = [(e34 - 10, e34 + 10, 0.3),            # straddles a binade
             (e34, e34 + 10, -1e-3),               # thmin + phi drops below 2^34
             (2 * e34 - 10, 2 * e34 - 1, 9.5),     # thmax + phi reaches 2^35
             (-5.0, 10.0, 0.7), (0.0, 3.0, 0.2), (-0.0, 3.0, 0.2),   # thmin <= 0
             (1e-300, 1.5e-300, 1e-310),           # exponent <= 52
             (2.5e10, 2.5e10 + 0.01, 0.5 * u), (2.5e10 + u, 2.5e10 + 0.01, 3.5 * u)]  # ties
    r = prims.phase([c[0] for c in cases], [c[2] for c in cases], [c[0] for c in cases], [c[1] for c in cases])
    assert not r["uniform"].any(), r["uniform"]


def test_sin_arg_reference(prims):
    """both branches of sin_arg against sin(fl(theta + phi)) in mpmath, |error| <= 4.5e-16, with
    the row's (sin, cos) from sincos_large as k_basis makes it"""
    rng = np.random.default_rng(18)
    th, ph, lo, hi = [], [], [], []
    for a, b, p in phase_jobs():
        for t in np.concatenate([[a, b], a + (b - a) * rng.uniform(0, 1, 6)]):
            t = min(max(t, a), b)
            th.append(t), ph.append(p), lo.append(a), hi.append(b)
    th, ph = np.array(th), np.array(ph)
    r = prims.phase(th, ph, lo, hi)
    for i in range(th.size):
        ref = mp.sin(mp.mpf(float(th[i] + ph[i])))
        for which in ("s_job", "s_row"):
            e = mp_err(r[which][i], ref)
            assert e <= 4.5e-16, (which, th[i], ph[i], r["uniform"][i], e)
    # (cos q, sin q) of a uniform job, from sincos(): its 2 ulp
    for i in np.flatnonzero(r["uniform"]):
        Q = mp.mpf(float(r["q"][i]))
        for got, ref in ((r["cq"][i], mp.cos(Q)), (r["sq"][i], mp.sin(Q))):
            assert mp_err(got, ref) <= 2 * np.spacing(abs(float(ref))), (r["q"][i], got)


# ---- Bessel coefficients ------------------------------------------------------------

def bessel_inputs():
    rng = np.random.default_rng(19)
    tiny = neighbours(np.array([1e-4, -1e-4]), 3)
    return np.concatenate([rng.uniform(-5, 5, 300), np.geomspace(1e-4, 5, 120), -np.geomspace(1e-4, 5, 60), tiny,
                           [0.0, -0.0, 5.0, -5.0, 1e-300, -1e-300, 1e-12, 3e-5, 4.999999999999999]])


def test_bessel_reference(prims):
    """bessel_j and bessel_j_lane within 2.3e-16 of J_k(b), k = 0..24, b in [-5, 5] including both
    sides of the switch to the power series at |b| = 1e-4; the lane form equals bessel_j bit for bit"""
    b = bessel_inputs()
    J = prims.bessel(b)
    JL = prims.bessel(b, lane=True)
    assert_same_bits(JL, J, "bessel_j_lane vs bessel_j")
    worst = 0.0
    for i, bi in enumerate(b):
        B = mp.mpf(float(bi))
        for k in range(HK + 1):
            e = mp_err(J[i, k], mp.besselj(k, B))
            assert e <= 2.3e-16, "J_%d(%r) = %r, error %.3g" % (k, float(bi), J[i, k], e)
            worst = max(worst, e)
    assert worst > 0.0


def test_jacobi_anger_truncation():
    """the HK = 24 harmonics the evaluator keeps: 2 sum_{k > 24} |J_k(b)| < 1.3e-15 for |b| <= HARM_BMAX
    (the tail grows with |b|: checked on a grid up to and at HARM_BMAX)"""
    for b in np.linspace(0.5, HARM_BMAX, 10):
        tail = 2 * mp.fsum(abs(mp.besselj(k, mp.mpf(b))) for k in range(HK + 1, 80))
        assert tail < 1.3e-15, (b, tail)


# ---- row_time / row_theta --------------------------------------------------------------

@pytest.mark.parametrize("big_endian", [False, True])
def test_row_time_theta(prims, big_endian):
    """row_time = float64(TIME) * 1e-6 + tmjd and row_theta = 6.283185 * t, two and one IEEE
    roundings (no FMA), bit for bit, in either byte order of the TIME column.  With tmjd = 86400 MJD
    the sum's ulp is 2^30 times the product's, so a fused multiply-add would round differently for
    almost no TIME; small tmjd values (relative times) make the difference common."""
    rng = np.random.default_rng(20)
    tm = np.concatenate([[-2 ** 31, -1, 0, 1, 2 ** 31 - 1], rng.integers(-2 ** 31, 2 ** 31, 20000)]).astype(np.int32)
    for tmjd in (0.0, 86400.0 * 59949.0, 86400.0 * 59949.01, 86400.0 * 70000.123, 1.0 / 3, -0.3, 1234.5678):
        t, th = prims.row_time(tm, big_endian, tmjd)
        ref_t = tm.astype(np.float64) * 1e-6 + tmjd
        assert_same_bits(t, ref_t, "row_time")
        assert_same_bits(th, 6.283185 * ref_t, "row_theta")


# ---- the device builds against the host build, and each other ---------------------------------

def _all_outputs(p):
    """every entry point over its test inputs (sqrt4 / sqrt aside)"""
    out = {}
    for which, x in (("large", large_inputs()), ("moderate", moderate_inputs()), ("demod", demod_inputs())):
        out[which] = (x, p.sincos(which, x))
    out["fc"] = p.fc_phasor(*fc_inputs())
    jobs = phase_jobs()
    rng = np.random.default_rng(21)
    th = np.concatenate([[a, b, a + (b - a) * rng.uniform()] for a, b, _ in jobs])
    rep = lambda k: np.repeat([j[k] for j in jobs], 3)
    out["phase"] = p.phase(np.clip(th, rep(0), rep(1)), rep(2), rep(0), rep(1))
    b = bessel_inputs()
    out["bessel"] = (p.bessel(b), p.bessel(b, lane=True))
    tm = np.concatenate([[-2 ** 31, -1, 0, 1, 2 ** 31 - 1], rng.integers(-2 ** 31, 2 ** 31, 20000)])
    out["time"] = [p.row_time(tm, be, tmjd) for be in (False, True) for tmjd in (86400.0 * 59949.01, 1.0 / 3)]
    return out


@pytest.mark.gpu
def test_device_equals_host_where_explicit(host, dev):
    """wherever the arithmetic is explicit (fma / _rn / rint / IEEE division) the device computes
    the host build's bits: the three sincos inside their ranges, both Bessel forms, phase_quantum,
    sin_arg of uniform jobs (given the same cos q, sin q, which come from sincos()), row_time,
    row_theta.  The sincos() / hypot / atan2 fallbacks are held to the references above only."""
    h = _all_outputs(host)
    for d in dev:
        o = _all_outputs(d)
        for which, lim in (("large", 2.0 ** 40), ("moderate", 1e5), ("demod", 9e3)):
            x, (hs, hc) = h[which]
            _, (ds, dc) = o[which]
            m = np.abs(x) < lim
            assert_same_bits(ds[m], hs[m], "sin " + which)
            assert_same_bits(dc[m], hc[m], "cos " + which)
        assert_same_bits(o["bessel"][0], h["bessel"][0], "bessel_j")
        assert_same_bits(o["bessel"][1], h["bessel"][1], "bessel_j_lane")
        hp, dp_ = h["phase"], o["phase"]
        assert (hp["uniform"] == dp_["uniform"]).all()
        assert_same_bits(dp_["q"], hp["q"], "phase_quantum q")
        m = (hp["uniform"] == 1) & same_bits(hp["cq"], dp_["cq"]) & same_bits(hp["sq"], dp_["sq"])
        assert m.any()
        assert_same_bits(dp_["s_job"][m], hp["s_job"][m], "sin_arg, uniform job")
        for (ht, hth), (dt, dth) in zip(h["time"], o["time"]):
            assert_same_bits(dt, ht, "row_time")
            assert_same_bits(dth, hth, "row_theta")


@pytest.mark.gpu
def test_fmad_setting_does_not_change_results(dev):
    """every entry point gives the same bits under nvcc -fmad=true and -fmad=false (the product
    compiles stream_kernels.cu one way and fit_kernels.cu the other)"""
    a, b = (_all_outputs(d) for d in dev)
    for which in ("large", "moderate", "demod"):
        for u, v in zip(a[which][1], b[which][1]):
            assert_same_bits(u, v, which)
    for u, v in zip(a["fc"], b["fc"]):
        assert_same_bits(u, v, "fc_phasor")
    for k in a["phase"]:
        assert_same_bits(a["phase"][k], b["phase"][k], "phase " + k)
    for u, v in zip(a["bessel"], b["bessel"]):
        assert_same_bits(u, v, "bessel")
    for (u1, u2), (v1, v2) in zip(a["time"], b["time"]):
        assert_same_bits(u1, v1, "row_time")
        assert_same_bits(u2, v2, "row_theta")
    h = sqrt_inputs()
    assert_same_bits(dev[0].sqrt4(h), dev[1].sqrt4(h), "sqrt4")


# ---- sqrt4 ----------------------------------------------------------------------------

def sqrt_inputs():
    e = np.arange(-1074, 1024)
    p2 = neighbours(np.ldexp(1.0, e), 2)
    hi = lambda w: np.array([w << 32], dtype=np.int64).view(np.float64)[0]
    edges = neighbours(np.array([hi(0x03500000), hi(0x7ff00000) - 0.0, np.finfo(float).max, 2.0 ** -970,
                                 np.finfo(float).tiny]), 3)
    edges = edges[np.isfinite(edges)]
    special = np.array([0.0, -0.0, -1.0, -1e-300, -np.inf, np.inf, np.nan, 5e-324, np.finfo(float).max])
    v = np.concatenate([p2, edges, special])
    return np.concatenate([v, np.ones((-v.size) % 4)])


@pytest.mark.gpu
def test_sqrt4_equals_sqrt(dev):
    """sqrt4 = sqrt() = the correctly rounded square root, bit for bit: binade edges, the edges of
    the range check (high word 0x03500000 ~ 2^-970, just below inf), subnormals, +-0, negatives,
    +-inf, NaN, DBL_MAX; a quad with one out-of-range value in each position; 2^24 random
    positive bit patterns"""
    rng = np.random.default_rng(22)
    fixed = sqrt_inputs()
    quads = []
    for odd in (0.0, 1e-300, 5e-324, -4.0, np.inf, np.nan, np.finfo(float).max):
        for pos in range(4):
            q = rng.uniform(0.5, 8.0, 4)
            q[pos] = odd
            quads.append(q)
    bits = rng.integers(0, 0x7ff0000000000000, 1 << 24, dtype=np.int64).view(np.float64)
    h = np.concatenate([fixed, np.concatenate(quads), bits])
    ref = np.sqrt(h)
    for d in dev:
        r4, r = d.sqrt4(h), d.sqrt(h)
        assert_same_bits(r, ref, "sqrt() vs numpy sqrt")
        assert_same_bits(r4, r, "sqrt4 vs sqrt()")


# ---- end to end: FC channels of extreme magnitude ---------------------------------------

FC_SCALES = [1.0, "zeros", 1e-310, 1e-150, 1e150, 1e300, 1e307, 1e-305]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["tensor", "dmma", "direct"])
def test_fc_magnitude_end_to_end(gp, ora, monkeypatch, mode):
    """Only the FC phase enters the model, so FC channels scaled to subnormal, tiny, huge and
    overflowing-square magnitudes, or with exact-zero and signed-zero rows, must fit like the
    oracle, group by group.  Runs with the tensor-core harmonic kernel (default), the DMMA one,
    and the direct evaluator."""
    tab = gp.synthetic.make_table(6000, k=3)
    t, z = gp.synthetic.to_complex(tab, gp.synthetic.stefan_centres())
    z = np.array(z)
    for g, s in enumerate(FC_SCALES):
        if s == "zeros":
            z[100:110, 32 + g] = 0.0
            z[200:204, 32 + g] = [complex(0.0, -0.0), complex(-0.0, 0.0), complex(-0.0, -0.0), 0j]
            z[3000:3005, 32 + g] = complex(-0.0, 0.0)
        else:
            z[:, 32 + g] *= s
    fcm = np.abs(z[:, 32:])
    assert (fcm[:, 2][fcm[:, 2] > 0] < 2.3e-308).all() and np.isinf(fcm[:, 6] ** 2).all()
    monkeypatch.setenv("GPPD_HARMONICS", "dmma" if mode == "dmma" else "tensor")
    out, par, like = gp.demodulateall(t, z, raw=True, method="direct" if mode == "direct" else "auto")
    oo, op, ol = ora.demodulateall(t, z, nthreads=8)
    assert np.isfinite(par).all() and np.isfinite(like).all(), \
        "non-finite fits in groups %s" % sorted(set(np.flatnonzero(~np.isfinite(par).all(1)) // 4))
    coincide, _ = compare_fits(par, like, op, ol)
    assert coincide.sum() >= MIN_COINCIDE, coincide
    err = np.abs(out[:, :32] - oo[:, :32]).max(axis=0) / np.abs(z[:, :32]).max(axis=0)
    assert err[coincide].max() <= 1e-9, err
