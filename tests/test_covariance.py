"""GPPD_COVARIANCE: the Gauss-Newton covariance of every fit's reported parameters
(definition in include/gppd.h, numpy reference in tests/covariance_ref.py)."""
import ctypes as C
import os
import re
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import covariance_ref as cref  # noqa: E402


# ---------------------------------------------------------------------------- CPU
def test_reference_jacobian_matches_finite_differences():
    rng = np.random.default_rng(1)
    n = 200
    t = 1e-3 * np.arange(n) + 0.37
    fc = np.exp(1j * rng.uniform(-np.pi, np.pi, n))
    power = rng.uniform(0.5, 2.0, n)
    for _ in range(5):
        p = np.array([*rng.normal(size=4), rng.uniform(0.3, 2.5), rng.uniform(-3, 3)])
        J = cref.jacobian(t, fc, p, power)
        for k in range(6):
            h = 1e-6 * max(1.0, abs(p[k]))
            pp, pm = p.copy(), p.copy()
            pp[k] += h
            pm[k] -= h
            fd = (cref.model(t, fc, pp, power) - cref.model(t, fc, pm, power)) / (2 * h)
            assert np.abs(fd - J[:, k]).max() <= 1e-7 * max(1.0, np.abs(J[:, k]).max()), k


def _mc_case(rng, faint, offsets, n=300):
    """Small synthetic arrays with known power and weight per row: bright (one level), or FAINT
    (two states of different power and noise, weights 1 / sigma^2)."""
    t = 1.7 + 1e-3 * np.arange(n)
    fc = np.exp(1j * np.cumsum(rng.normal(0, 0.05, n)))
    if faint:
        hi = (np.arange(n) // 50) % 2 == 0
        power = np.where(hi, 1.0, 0.4)
        sigma = np.where(hi, 0.05, 0.12)
    else:
        power, sigma = np.ones(n), np.full(n, 0.08)
    weight = 1.0 / sigma ** 2
    truth = np.array([0.05 if offsets else 0.0, -0.03 if offsets else 0.0, 0.8, 0.4, 1.3, 0.6])
    return t, fc, power, sigma, weight, truth


def _lsq_fit(t, d, fc, power, weight, x0, offsets):
    from scipy.optimize import least_squares
    k0 = 0 if offsets else 2
    sw = np.sqrt(weight)

    def res(x):
        p = np.zeros(6)
        p[k0:] = x
        r = (cref.model(t, fc, p, power) - d) * sw
        return np.concatenate([r.real, r.imag])

    sol = least_squares(res, x0[k0:], method="lm", xtol=1e-14, ftol=1e-14, gtol=1e-14)
    p = np.zeros(6)
    p[k0:] = sol.x
    return p


def _cov_given(t, d, fc, p, power, weight, offsets):
    """The reference's definition with the given power and weight (no states)."""
    k0 = 0 if offsets else 2
    k = 6 - k0
    J = cref.jacobian(t, fc, p, power)[:, k0:]
    H = np.real((J.conj() * weight[:, None]).T @ J)
    r = cref.model(t, fc, p, power) - d
    s2 = np.sum(weight * np.abs(r) ** 2) / (2 * t.size - k)
    out = np.zeros((6, 6))
    out[k0:, k0:] = s2 * np.linalg.inv(H)
    return out


def _zscore_bounds(z):
    z = np.asarray(z)
    mad = 1.4826 * np.median(np.abs(z - np.median(z)))
    return mad, np.mean(np.abs(z) < 5)


def test_definition_is_calibrated_by_monte_carlo():
    """Fits of K noise realisations: (theta_hat - theta_true) / sigma of b, phi, a.re, a.im has
    a robust standard deviation within [0.9, 1.1], and >= 99 % of |z| < 5."""
    rng = np.random.default_rng(7)
    zs = []
    for faint in (False, True):
        for offsets in (False, True):
            t, fc, power, sigma, weight, truth = _mc_case(rng, faint, offsets)
            m = cref.model(t, fc, truth, power)
            for _ in range(60):
                noise = sigma / np.sqrt(2) * (rng.normal(size=t.size) + 1j * rng.normal(size=t.size))
                d = m + noise
                p = _lsq_fit(t, d, fc, power, weight, truth, offsets)
                V = _cov_given(t, d, fc, p, power, weight, offsets)
                sd = np.sqrt(np.diag(V))[2:]
                assert sd[2] >= 1e-3
                zs.extend((p - truth)[2:] / sd)
    mad, frac = _zscore_bounds(zs)
    assert 0.9 <= mad <= 1.1, mad
    assert frac >= 0.99, frac


def test_reference_uses_states_and_nan_rules(ora):
    """The reference with states: FAINT powers / weights from compute_mean_var_power, TRANSIENT
    rows left out; NaN for too few rows and for a zero diode."""
    rng = np.random.default_rng(3)
    n = 400
    t = 2.0 + 1e-3 * np.arange(n)
    st = np.where((np.arange(n) // 40) % 2 == 0, 3, 1).astype(np.int8)
    st[::37] = -1
    fc = np.exp(1j * rng.uniform(-np.pi, np.pi, n))
    p = np.array([0.0, 0.0, 0.6, 0.2, 1.1, 0.3])
    m, w = ora.compute_mean_var_power(st, np.ones(n))
    d = cref.model(t, fc, p, np.where(st == 3, 1.0, 0.5)) + 0.05 * rng.normal(size=n)
    V = cref.covariance(t, d, fc, p, st)
    assert np.isfinite(V).all() and (V[:2] == 0).all() and (np.diag(V)[2:] > 0).all()
    Vh = cref.covariance(t, d, fc, p, st, onlyhigh=True)
    assert Vh[4, 4] > V[4, 4]                           # fewer rows, larger variance
    assert np.isnan(cref.covariance(t[:2], d[:2], fc[:2], p)).all()
    assert np.isnan(cref.covariance(t, np.zeros(n), fc, np.array([0, 0, 0, 0, 1.0, 0.3]))).all()


def test_flag_and_stride_agree_everywhere():
    from gppd_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "gppd.h")).read()
    jl = open(os.path.join(ROOT, "julia", "GPPDB200.jl")).read()
    flag = int(re.search(r"#define GPPD_COVARIANCE (0x[0-9a-fA-F]+)u", hdr).group(1), 16)
    stride = int(re.search(r"#define GPPD_COV_STRIDE (\d+)", hdr).group(1))
    assert flag == _lib.COVARIANCE == 256 and stride == _lib.COV_STRIDE == 36
    assert flag < (1 << 16)                              # bits 16..23 carry group_mask
    other = [int(v) for v in re.findall(r"#define GPPD_[A-Z0-9_]+ (\d+)u", hdr)]
    other += [int(v, 16) for v in re.findall(r"#define GPPD_[A-Z0-9_]+ (0x[0-9a-fA-F]+)u", hdr)]
    assert other.count(flag) == 1
    assert int(re.search(r"const GPPD_COVARIANCE\s*=\s*UInt32\((0x[0-9a-fA-F]+)\)", jl).group(1), 16) == flag
    assert int(re.search(r"const GPPD_COV_STRIDE\s*=\s*(\d+)", jl).group(1)) == stride
    assert "gppd_covariances" in jl and "int gppd_covariances(gppd_handle h, int slot, int64_t nfits, double *cov);" in hdr


def test_cli_accepts_uncertainty():
    from gppd_b200 import cli
    assert cli.build_parser().parse_args(["--uncertainty", "x"]).uncertainty
    assert not cli.build_parser().parse_args(["x"]).uncertainty


def test_delta_method_helpers_match_finite_differences():
    from gppd_b200.api import uncertainties, uncertainty_keys, window_uncertainty_columns
    rng = np.random.default_rng(5)
    P = rng.normal(size=(64, 6))
    A = rng.normal(size=(64, 6, 6)) * 1e-3
    V = A @ A.transpose(0, 2, 1)
    u = uncertainties(P, V)
    h = 1e-7
    for f, key in ((np.abs, "ABSA"), (np.angle, "ARGA")):
        for i in range(64):
            a = complex(P[i, 2], P[i, 3])
            g = np.array([(f(a + h) - f(a - h)) / (2 * h), (f(a + 1j * h) - f(a - 1j * h)) / (2 * h)])
            assert abs(u[key][i] - np.sqrt(g @ V[i, 2:4, 2:4] @ g)) <= 1e-6 * u[key][i]
    assert np.array_equal(u["B"], np.sqrt(V[:, 4, 4])) and np.array_equal(u["PHI"], np.sqrt(V[:, 5, 5]))
    assert np.array_equal(u["X0"], np.sqrt(V[:, 0, 0])) and np.array_equal(u["Y0"], np.sqrt(V[:, 1, 1]))
    k = uncertainty_keys(P[:32], V[:32], True)
    assert len(k) == 6 * 32 and k["DEMODULATION SIN PHASE ERR SC T2 D3"] == u["PHI"][16 + 2 + 4]
    assert len(uncertainty_keys(P[:32], V[:32], False)) == 4 * 32
    cols = window_uncertainty_columns(P, V, 250, 100, 2, False)
    assert set(cols) == {"ABSA_ERR", "ARGA_ERR", "B_ERR", "PHI_ERR"}
    assert cols["B_ERR"].shape == (250, 32) and cols["B_ERR"].dtype == np.float32
    assert np.array_equal(cols["B_ERR"][150], u["B"][32:].astype(np.float32))


# ---------------------------------------------------------------------------- GPU
def _near(dev, ref, tol=1e-9):
    """Entry by entry within tol * sqrt(V_ii V_jj) of the reference; NaN where it is NaN."""
    dev, ref = np.asarray(dev), np.asarray(ref)
    assert np.array_equal(np.isnan(dev), np.isnan(ref))
    ok = ~np.isnan(ref[:, 0, 0]) | ~np.isnan(ref[:, 2, 2])
    d = np.sqrt(np.abs(np.diagonal(ref, axis1=1, axis2=2)))
    scale = d[:, :, None] * d[:, None, :]
    err = np.abs(dev - ref)[ok] / np.maximum(scale[ok], 1e-300)
    err[(scale[ok] == 0) & (dev[ok] == ref[ok])] = 0.0
    assert err.max() <= tol, err.max()


def _table_arrays(gp, ora, tab, offsets):
    t = ora.make_times(tab["time_us"], tab["mjd"])
    v = tab["volt"].astype(np.float64)
    z = v[:, 0::2] + 1j * v[:, 1::2]
    if offsets is not None:
        z = z - np.asarray(offsets)[None, :]
    return t, z


@pytest.mark.gpu
@pytest.mark.parametrize("faint,fitoffsets,window,method,onlyhigh", [
    (False, False, None, "auto", False),
    (True, False, None, "auto", False),
    (False, True, None, "direct", False),
    (True, True, 1.0, "auto", False),
    (True, False, 1.0, "direct", True),
])
def test_table_path_matches_reference(gp, ora, faint, fitoffsets, window, method, onlyhigh):
    from conftest import make_case
    tab = make_case(gp.synthetic, 12000, k=11, faint=faint, ora=ora)
    off = None if fitoffsets else gp.synthetic.stefan_centres()
    wrows, nwin = gp.table_windows(tab["time_us"], tab["mjd"], window)
    cov = np.empty((nwin * 32, 6, 6))
    fs = tab["faintstates"]
    fsp = gp.FaintStates(fs.timer1, fs.timer2, 1.0, 2.0) if faint else None
    _, P, _, _, state = gp.process_table(tab["time_us"], tab["volt"], tab["mjd"], offsets=off, faintparam=fsp,
                                         window=window, method=method, onlyhigh=onlyhigh, cov_out=cov)
    t, z = _table_arrays(gp, ora, tab, off)
    ref = cref.covariances_table(t, z, P, state, onlyhigh, fitoffsets, wrows)
    _near(cov, ref)
    if not fitoffsets:                                  # no c in the model: rows / columns 0-1 are 0
        fin = np.isfinite(cov).all(axis=(1, 2))         # (onlyhigh windows without HIGH rows are NaN)
        assert fin.any()
        assert (cov[fin][:, :2, :] == 0).all() and (cov[fin][:, :, :2] == 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("faint,fitoffsets,nwindow,method", [
    (False, True, 0, "auto"), (True, False, 0, "direct"), (False, False, 3000, "auto"), (True, True, 4000, "auto"),
])
def test_array_path_matches_reference(gp, ora, faint, fitoffsets, nwindow, method):
    from conftest import make_case
    tab = make_case(gp.synthetic, 10000, k=12, faint=faint, ora=ora)
    t, z = gp.synthetic.to_complex(tab, gp.synthetic.stefan_centres())
    _, P, _, cov = gp.demodulateall(t, z, raw=True, faintparam=tab["state"], fitoffsets=fitoffsets,
                                    nwindow=nwindow, method=method, return_cov=True)
    _near(cov, cref.covariances_table(t, z, P, tab["state"], False, fitoffsets, nwindow))


@pytest.mark.gpu
def test_direct_fallback_fits_match_reference(gp, ora):
    """A start at |b| > 5 makes the harmonic evaluator give up: every fit is redone by the
    direct evaluator (info[:, 2] == 1), and its covariance is that of the reference."""
    from conftest import make_case
    tab = make_case(gp.synthetic, 6000, k=13)
    t, z = gp.synthetic.to_complex(tab, gp.synthetic.stefan_centres())
    _, P, _, info, cov = gp.demodulateall(t, z, raw=True, init=[6.0, 0.3], return_info=True, return_cov=True)
    assert (info[:, 2] == 1).all()
    _near(cov, cref.covariances_table(t, z, P))


@pytest.mark.gpu
def test_flag_changes_nothing_else(gp, ora):
    from conftest import make_case
    tab = make_case(gp.synthetic, 8000, k=14, faint=True, ora=ora)
    fs = gp.FaintStates(tab["faintstates"].timer1, tab["faintstates"].timer2, 1.0, 2.0)
    for off in (gp.synthetic.stefan_centres(), None, True, "ellipse"):
        for window in (None, 1.0):
            _, nwin = gp.table_windows(tab["time_us"], tab["mjd"], window)
            a = gp.process_table(tab["time_us"], tab["volt"], tab["mjd"], offsets=off, faintparam=fs, window=window)
            b = gp.process_table(tab["time_us"], tab["volt"], tab["mjd"], offsets=off, faintparam=fs, window=window,
                                 cov_out=np.empty((nwin * 32, 6, 6)))
            for x, y in zip(a, b):
                assert x.tobytes() == y.tobytes()
    t, z = gp.synthetic.to_complex(tab, gp.synthetic.stefan_centres())
    a = gp.demodulateall(t, z, raw=True, faintparam=tab["state"], fitoffsets=True, nwindow=3000, return_info=True)
    b = gp.demodulateall(t, z, raw=True, faintparam=tab["state"], fitoffsets=True, nwindow=3000, return_info=True,
                         return_cov=True)
    for x, y in zip(a, b[:4]):
        assert x.tobytes() == y.tobytes()


def _dev_batch(gp, tabs, faint_flags, cov_nfits, slot=1, offsets=None):
    """The tables as one gppd_process_tables_f32_dev batch with GPPD_COVARIANCE; returns
    (params per table, covariances of the batch)."""
    import torch
    from gppd_b200 import _lib
    h = gp.default_handle()
    T = len(tabs)
    keep = []

    def dev(a):
        x = torch.from_numpy(np.ascontiguousarray(a)).cuda()
        keep.append(x)
        return x.data_ptr()

    PP = C.c_void_p * T
    n = (C.c_int64 * T)(*[tb["time_us"].size for tb in tabs])
    mjd = (C.c_double * T)(*[tb["mjd"] for tb in tabs])
    tu = PP(*[dev(tb["time_us"]) for tb in tabs])
    vo = PP(*[dev(tb["volt"]) for tb in tabs])
    vout = PP(*[dev(np.zeros((tb["time_us"].size, 80), np.float32)) for tb in tabs])
    par = [torch.zeros((32, 6), dtype=torch.float64, device="cuda") for _ in tabs]
    chi = [torch.zeros(32, dtype=torch.float64, device="cuda") for _ in tabs]
    pars, chis = PP(*[p.data_ptr() for p in par]), PP(*[c.data_ptr() for c in chi])
    t1 = [tb["faintstates"].timer1 if f else None for tb, f in zip(tabs, faint_flags)]
    t2 = [tb["faintstates"].timer2 if f else None for tb, f in zip(tabs, faint_flags)]
    T1 = (_lib._dp * T)(*[_lib.ptr(x) for x in t1])
    T2 = (_lib._dp * T)(*[_lib.ptr(x) for x in t2])
    n1 = (C.c_int64 * T)(*[0 if x is None else x.size for x in t1])
    n2 = (C.c_int64 * T)(*[0 if x is None else x.size for x in t2])
    o = gp.api._options(covariance=True)
    doff = dev(np.ascontiguousarray(offsets).view(np.float64)) if offsets is not None else None
    _lib.check(_lib.lib().gppd_process_tables_f32_dev(h.raw, slot, None, T, n, None, tu, mjd, vo, doff, T1, n1, T2,
                                                      n2, C.byref(o), vout, pars, chis, None, None))
    cov = gp.api.covariances(h, slot, cov_nfits)
    return [p.cpu().numpy() for p in par], cov


@pytest.mark.gpu
def test_bitwise_across_runs_batches_and_entry_points(gp, ora, tmp_path):
    from conftest import make_case
    off = gp.synthetic.stefan_centres()
    tf = make_case(gp.synthetic, 9000, k=15, faint=True, ora=ora)
    tb = make_case(gp.synthetic, 7000, k=16)
    fs = gp.FaintStates(tf["faintstates"].timer1, tf["faintstates"].timer2, 1.0, 2.0)
    c1, c2 = np.empty((32, 6, 6)), np.empty((32, 6, 6))
    gp.process_table(tf["time_us"], tf["volt"], tf["mjd"], offsets=off, faintparam=fs, cov_out=c1)
    gp.process_table(tf["time_us"], tf["volt"], tf["mjd"], offsets=off, faintparam=fs, cov_out=c2)
    assert c1.tobytes() == c2.tobytes()
    # inside a mixed batch (FAINT + bright) of the device entry point
    _, cb = _dev_batch(gp, [tb, tf], [False, True], 64, offsets=off)
    assert cb[32:].tobytes() == c1.tobytes()
    cb1 = np.empty((32, 6, 6))
    gp.process_table(tb["time_us"], tb["volt"], tb["mjd"], offsets=off, cov_out=cb1)
    assert cb[:32].tobytes() == cb1.tobytes()
    # the record entry point (submit_fits_rows, through the CLI's scheduler) and the native file path
    from gppd_b200 import cli, fits
    p = gp.synthetic.make_fits(str(tmp_path / "f.fits"), tf, tf["header"])
    h = gp.default_handle()
    for native in (True, False):
        sched = cli.NightScheduler(h, off, False, uncertainty=True)
        args = cli.build_parser().parse_args((["--no-native"] if not native else []) + [str(tmp_path)])
        job = cli._plan_file(p, args, str(tmp_path / ("n" if native else "p")))
        sched.submit(2, job)
        jb, b = sched.busy[2]
        if native:
            gp._lib.check(gp._lib.lib().gppd_file_wait(h.raw, 2, gp._lib.ptr(np.empty((32, 6))), None, None, None))
        else:
            gp._lib.check(gp._lib.lib().gppd_wait(h.raw, 2))
        assert gp.api.covariances(h, 2, 32).tobytes() == c1.tobytes(), native
        if native:
            gp._lib.check(gp._lib.lib().gppd_file_drain(h.raw))
    # the array entry points on the same arrays agree with each other
    t, z = gp.synthetic.to_complex(tb, off)
    ca = gp.demodulateall(t, z, raw=True, return_cov=True)[-1]
    import torch
    dt, dz = torch.from_numpy(t).cuda(), torch.from_numpy(np.asfortranarray(z).T.reshape(-1).view(np.float64)).cuda()
    dout = torch.empty_like(dz)
    dp, dc = torch.empty(32 * 6, dtype=torch.float64, device="cuda"), torch.empty(32, dtype=torch.float64, device="cuda")
    o = gp.api._options(covariance=True)
    gp._lib.check(gp._lib.lib().gppd_demodulate_f64_dev(h.raw, 3, None, t.size, 0, dt.data_ptr(), dz.data_ptr(),
                                                         None, C.byref(o), dout.data_ptr(), dp.data_ptr(),
                                                         dc.data_ptr(), None))
    torch.cuda.synchronize()
    assert gp.api.covariances(h, 3, 32).tobytes() == ca.tobytes()


@pytest.mark.gpu
def test_degenerate_fits_are_nan_and_getter_errors(gp, ora):
    from conftest import make_case
    tab = make_case(gp.synthetic, 6002, k=17)
    t, z = gp.synthetic.to_complex(tab, gp.synthetic.stefan_centres())
    z[:, 5] = 0.0
    _, P, _, cov = gp.demodulateall(t, z, raw=True, nwindow=3000, return_cov=True)
    bad = np.isnan(cov).all(axis=(1, 2))
    # diode 5 of each window, and every fit of the 2-row last window (2 N_valid = 4 <= k = 4)
    assert set(np.nonzero(bad)[0]) == {5, 37} | set(range(64, 96))
    assert np.isfinite(cov[~bad]).all()
    _, P, _, cov = gp.demodulateall(t, z, raw=True, groups=0b00000110, return_cov=True)
    on = np.zeros(32, bool)
    on[4:12] = True
    on[5] = False
    assert np.array_equal(~np.isnan(cov).all(axis=(1, 2)), on)
    h = gp.default_handle()
    gp.demodulateall(t, z, raw=True)                    # without the flag
    with pytest.raises(gp.GppdError) as e:
        gp.api.covariances(h, 0, 32)
    assert e.value.status == 1
    gp.demodulateall(t, z, raw=True, return_cov=True)
    with pytest.raises(gp.GppdError) as e:
        gp.api.covariances(h, 0, 33)
    assert e.value.status == 1


@pytest.mark.gpu
def test_ellipse_mode_equals_array_path_on_corrected_channels(gp, ora):
    from conftest import make_case
    tab = make_case(gp.synthetic, 8000, k=18)
    ell = np.empty((40, 6))
    cov = np.empty((32, 6, 6))
    gp.process_table(tab["time_us"], tab["volt"], tab["mjd"], offsets="ellipse", ellipses_out=ell, cov_out=cov)
    t = ora.make_times(tab["time_us"], tab["mjd"])
    v = tab["volt"].astype(np.float64)
    x, y = v[:, 0::2] - ell[:, 0], v[:, 1::2] - ell[:, 1]
    yc = ell[:, 4] * x + ell[:, 5] * y                  # numpy: every operation rounded, no FMA
    z = x + 1j * yc
    ca = gp.demodulateall(t, z, raw=True, return_cov=True)[-1]
    assert ca.tobytes() == cov.tobytes()


@pytest.mark.gpu
def test_device_monte_carlo_is_calibrated(gp):
    """Device fits of noise realisations, NEWUOA run to rhoend = 1e-8: the z-scores of b, phi,
    a.re and a.im against the truth follow the device's covariances."""
    rng = np.random.default_rng(11)
    n, K = 2000, 12
    t = 1.5 + 1e-3 * np.arange(n)
    fc = np.exp(1j * np.cumsum(rng.normal(0, 0.05, n)))
    zs = []
    for _ in range(K):
        z = np.zeros((n, 40), complex)
        z[:, 32:] = fc[:, None]
        # (truths near the common start: every fit converges to the minimum the noise moved)
        truth = np.column_stack([np.zeros(32), np.zeros(32), rng.uniform(0.5, 1.0, 32), rng.uniform(-0.5, 0.5, 32),
                                 rng.uniform(1.1, 1.5, 32), rng.uniform(-0.4, 0.4, 32)])
        for ch in range(32):
            z[:, ch] = cref.model(t, fc, truth[ch], np.ones(n)) + 0.3 / np.sqrt(2) * (
                rng.normal(size=n) + 1j * rng.normal(size=n))
        _, P, _, cov = gp.demodulateall(t, z, raw=True, init=[1.3, 0.0], maxfun=400, rhoend=1e-8, return_cov=True)
        sd = np.sqrt(np.diagonal(cov, axis1=1, axis2=2))
        assert (sd[:, 4] >= 1e-3).all()
        dphi = np.remainder(P[:, 5] - truth[:, 5] + np.pi, 2 * np.pi) - np.pi
        zs.extend(((P[:, 2:5] - truth[:, 2:5]) / sd[:, 2:5]).ravel())
        zs.extend(dphi / sd[:, 5])
    mad, frac = _zscore_bounds(zs)
    assert 0.9 <= mad <= 1.1, mad
    assert frac >= 0.99, frac


@pytest.mark.gpu
@pytest.mark.parametrize("native", [True, False])
@pytest.mark.parametrize("window", [None, 2.0])
def test_cli_uncertainty_keys_and_columns(gp, ora, tmp_path, native, window):
    from conftest import make_case
    from gppd_b200 import cli, fits
    from gppd_b200.api import uncertainty_keys, window_uncertainty_columns
    d = tmp_path / "in"
    d.mkdir()
    tab = make_case(gp.synthetic, 5000, k=19, faint=True, ora=ora)
    gp.synthetic.make_fits(str(d / "f.fits"), tab, tab["header"])
    mode = [] if native else ["--no-native"]
    win = [] if window is None else ["-w", str(window)]
    assert cli.main(mode + win + ["-d", str(tmp_path / "a"), str(d / "f.fits")]) == 0
    assert cli.main(mode + win + ["--uncertainty", "-d", str(tmp_path / "b"), str(d / "f.fits")]) == 0
    fs = gp.FaintStates(tab["faintstates"].timer1, tab["faintstates"].timer2, 1.0, 2.0)
    wrows, nwin = gp.table_windows(tab["time_us"], tab["mjd"], window)
    cov = np.empty((nwin * 32, 6, 6))
    _, P, _, _, _ = gp.process_table(tab["time_us"], tab["volt"], tab["mjd"], offsets=gp.synthetic.stefan_centres(),
                                     faintparam=fs, window=window, cov_out=cov)
    a = fits.read_fits(str(tmp_path / "a" / "f.fits"))[3]
    b = fits.read_fits(str(tmp_path / "b" / "f.fits"))[3]
    rb, n, cols = fits.bintable_layout(b.header)
    rec = np.frombuffer(b.data, np.uint8, n * rb).reshape(n, rb)
    ra, _, cols_a = fits.bintable_layout(a.header)
    reca = np.frombuffer(a.data, np.uint8, n * ra).reshape(n, ra)
    for name, (o, _, *_r) in cols_a.items():           # every column of the plain output is unchanged
        w = fits.tform_bytes(cols_a[name][1])
        ob = cols[name][0]
        assert np.array_equal(rec[:, ob:ob + w], reca[:, o:o + w]), name
    if window is None:
        for k, v in uncertainty_keys(P, cov, False).items():
            assert b.header[k] == v, k
        assert not any("ERR" in k for k in a.header)
    else:
        for k, v in window_uncertainty_columns(P, cov, n, wrows, nwin, False).items():
            o = cols[k][0]
            assert np.array_equal(rec[:, o:o + 128].copy().view(">f4").astype(np.float32), v), k
        assert not any(k.endswith("_ERR") for k in cols_a)
