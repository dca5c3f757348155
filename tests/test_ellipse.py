"""`--center ellipse` (GPPD_CENTER_ELLIPSE): offset and ellipse (Heydemann) correction of
the 40 VOLT channels before the fit (include/gppd.h states the definition).

tests/ellipse_ref.py restates the definition with lstsq on top of the oracle (ellipse_fit /
compute_ellipses / apply_ellipses / processmetrology); the CPU tests pin it on ellipses with known parameters and show what the
correction buys on distorted synthetic tables; the GPU tests hold the device fit to the
oracle and the table path to "the correction + the existing array path", bit for bit."""
import ctypes as C
import hashlib
import os
import re

import numpy as np
import pytest

import ellipse_ref as er
from conftest import make_case

ELL_TOL = 1e-10   # centre / radius, r, alpha: device moments + Cholesky vs lstsq, well-conditioned channels


def _solve_tolerance(z, state):
    """Per-channel bound of |device - lstsq| (r, alpha; centre / radius).  The device solves the
    normal equations (condition kappa = cond(design)^2) formed from sums taken relative to the
    table's first sample and moved to the centroid analytically, which loses rho^4 (rho = that
    pivot's distance from the centroid in rms radii: large for the HIGH samples of a short FAINT
    table).  A NumPy restatement of that arithmetic against lstsq, on the distorted tables of
    this file at 700 / 5 000 / 20 011 rows, bright and FAINT: |delta| <= 1.4e-15 kappa rho^4, at
    most 5e-12 on bright tables and 1.0e-10 on 700-row FAINT ones.  Bound: 2e-14 kappa rho^4,
    and never below ELL_TOL."""
    sel = slice(None) if state is None else (np.asarray(state) == 3)
    tol = np.full(40, ELL_TOL)
    for ch in range(40):
        x, y = z[sel, ch].real, z[sel, ch].imag
        if x.size < 5:
            continue
        u, v = x - x.mean(), y - y.mean()
        s = np.sqrt(np.mean(u * u + v * v))
        if not s > 0:
            continue
        u, v = u / s, v / s
        kappa = np.linalg.cond(np.stack([u * u - v * v, u * v, u, v, np.ones_like(u)], axis=1)) ** 2
        rho = max(1.0, abs(z[0, ch] - complex(x.mean(), y.mean())) / s)
        tol[ch] = max(ELL_TOL, 2e-14 * kappa * rho ** 4)
    return tol


def _ellipse_points(x0, y0, r, alpha, R, th):
    """the Heydemann forward model around a circle of radius R"""
    u1, u2 = R * np.cos(th), R * np.sin(th)
    return x0 + u1, y0 + (u2 * np.cos(alpha) - u1 * np.sin(alpha)) / r


def _case(gp, ora, n, k, faint=False, quadrature=True):
    """make_case with imperfect quadrature detectors"""
    tab = make_case(gp.synthetic, n, k=k, faint=faint, ora=ora)
    return dict(tab, **{kk: v for kk, v in gp.synthetic.make_table(
        n, k=k, faint=faint, state=tab["state"], quadrature=quadrature).items() if kk in ("volt", "truth")})


def _cmplx(volt):
    v = np.asarray(volt).astype(np.float64)
    return v[:, 0::2] + 1j * v[:, 1::2]


# ---------------------------------------------------------------------------- CPU
def test_oracle_ellipse_known_parameters(ora):
    rng = np.random.default_rng(7)
    cases = [(0.3, -0.2, 1.3, 0.4, 0.5, 2 * np.pi),       # full ellipse
             (-1.0, 2.0, 0.7, -0.4, 0.2, 2.5),            # 2.5-rad arc
             (2000 * 0.1, -0.5, 1.3, -0.4, 0.1, 2 * np.pi),  # centre 2000 radii away
             (0.05, 0.01, 0.7, 0.4, 0.3, 3.0)]
    for x0, y0, r, al, R, arc in cases:
        th = rng.uniform(0.2, 0.2 + arc, size=500)
        x, y = _ellipse_points(x0, y0, r, al, R, th)
        gx, gy, gr, ga, st = er.ellipse_fit(x, y)
        assert st == 2
        assert abs(complex(gx - x0, gy - y0)) <= 1e-9 * R, (x0, y0, gx, gy)
        assert abs(gr - r) <= 1e-9 and abs(ga - al) <= 1e-9, (r, al, gr, ga)
        # the correction maps the points onto a circle of radius R
        ell, _ = er.compute_ellipses(np.repeat((x + 1j * y)[:, None], 40, axis=1))
        z = er.apply_ellipses(np.repeat((x + 1j * y)[:, None], 40, axis=1), ell)[:, 0]
        assert np.abs(np.abs(z) - R).max() <= 1e-9 * R
    # a true circle: r = 1, alpha = 0, the circle centre of --center empirical
    th = rng.uniform(0, 2 * np.pi, size=300)
    x, y = 3.0 + 0.4 * np.cos(th), -4.0 + 0.4 * np.sin(th)
    gx, gy, gr, ga, st = er.ellipse_fit(x, y)
    assert st == 2 and abs(gr - 1) <= 1e-9 and abs(ga) <= 1e-9
    assert abs(complex(gx, gy) - ora.circle_centre(x, y)) <= 1e-12 * 0.4 * 1e1


def test_oracle_ellipse_fallbacks(ora):
    # fewer than 5 points: the circle centre, identity shape
    x, y = np.array([1.0, 0.0, -1.0, 0.0]) + 2, np.array([0.0, 1.0, 0.0, -1.0]) - 1
    assert er.ellipse_fit(x, y) == (pytest.approx(2.0), pytest.approx(-1.0), 1.0, 0.0, 1)
    # a line: no conic, no circle either
    t = np.linspace(0, 1, 50)
    assert er.ellipse_fit(t, 2 * t + 1) == (0.0, 0.0, 1.0, 0.0, 0)
    # one point
    assert er.ellipse_fit(np.ones(10), np.ones(10)) == (0.0, 0.0, 1.0, 0.0, 0)
    # both branches of a hyperbola: no ellipse (A or C <= 0 or the axis ratio), circle centre
    s = np.linspace(-1.5, 1.5, 60)
    x = np.concatenate([np.cosh(s), -np.cosh(s)]) + 0.5
    y = np.concatenate([np.sinh(s), np.sinh(s)]) - 0.25
    gx, gy, gr, ga, st = er.ellipse_fit(x, y)
    c = ora.circle_centre(x, y)
    assert st == 1 and (gr, ga) == (1.0, 0.0) and complex(gx, gy) == c
    # a very flat ellipse (axis ratio 20 > 10): no ellipse
    th = np.linspace(0, 2 * np.pi, 200, endpoint=False)
    gx, gy, gr, ga, st = er.ellipse_fit(1 + np.cos(th), 2 + 0.05 * np.sin(th))
    assert st == 1 and (gr, ga) == (1.0, 0.0)


def test_oracle_ellipses_use_high_samples(ora):
    rng = np.random.default_rng(11)
    n = 3000
    state = rng.choice(np.array([ora.OFF, ora.LOW, ora.NORMAL, ora.HIGH, ora.TRANSIENT]), size=n)
    th = rng.uniform(0, 2 * np.pi, size=(n, 40))
    c_high = (np.arange(40) - 20) * (0.01 + 0.02j)
    xh, yh = _ellipse_points(c_high.real[None, :], c_high.imag[None, :], 1.2, 0.1, 0.3, th)
    xo, yo = _ellipse_points(5.0, -1.0, 0.8, -0.2, 0.1, th)
    hi = (state == ora.HIGH)[:, None]
    v = np.where(hi, xh + 1j * yh, xo + 1j * yo)          # other states: another ellipse
    ell, st = er.compute_ellipses(v, state)
    assert (st == 2).all()
    assert np.abs(ell[:, 0] + 1j * ell[:, 1] - c_high).max() < 1e-9
    assert np.abs(ell[:, 2] - 1.2).max() < 1e-9 and np.abs(ell[:, 3] - 0.1).max() < 1e-9
    assert np.abs(er.compute_ellipses(v, None)[0][:, 2] - 1.2).min() > 1e-3


def test_make_table_default_unchanged(gp):
    """the generator without `quadrature` returns the bytes it always has (the golden vectors
    rebuild their inputs from it)"""
    want = {(3000, 3, False): "3fbb2ff0ba2ccb3d44f06b02b8cf8ae61c34eb4b311f92ccf5d37b9359e3985b",
            (2000, 5, True): "6fbc64b836ea5b329d80c8758123d5546913e7348aec89b5e84aa8c0ba17f876"}
    for (n, k, faint), digest in want.items():
        t = gp.synthetic.make_table(n, k=k, faint=faint, jitter=faint)
        assert hashlib.sha256(t["time_us"].tobytes() + t["volt"].tobytes()).hexdigest() == digest
    q = gp.synthetic.make_table(3000, k=3, quadrature=True)
    assert not np.array_equal(q["volt"], gp.synthetic.make_table(3000, k=3)["volt"])
    assert (np.abs(q["truth"]["quad_r"] - 1) <= 0.15).all() and (np.abs(q["truth"]["quad_alpha"]) <= 0.15).all()


def test_ellipse_recovery_oracle(ora, gp):
    """20 000 rows, every channel distorted with r ~ U(0.85, 1.15), alpha ~ U(-0.15, 0.15):
    the circle model fits a distorted phase, the corrected channels do not.  (Measured here:
    median |b - b_true| 3.0e-4 undistorted / circle, 1.2e-2 distorted / circle, 4.0e-4
    distorted / ellipse.)"""
    import fitref
    n = 20000
    und = gp.synthetic.make_table(n, k=3)
    dis = gp.synthetic.make_table(n, k=3, quadrature=True)
    b_true = und["truth"]["b"]

    def fit(tab, mode):
        t = ora.make_times(tab["time_us"], tab["mjd"])
        z = _cmplx(tab["volt"])
        if mode == "circle":
            z = z - ora.compute_offsets(z)[None, :]
        else:
            z = er.apply_ellipses(z, er.compute_ellipses(z)[0])
        return ora.demodulateall(t, z, nthreads=8)[1]

    p_uc, p_dc, p_de, p_ue = fit(und, "circle"), fit(dis, "circle"), fit(dis, "ellipse"), fit(und, "ellipse")
    err = lambda p: np.median(np.abs(np.abs(p[:, 4]) - b_true))
    assert err(p_de) <= err(p_dc) / 10
    assert err(p_de) <= 3 * err(p_uc)
    # undistorted data: the ellipse mode moves the fits by the typical size of a NEWUOA fork
    # (its own r and alpha are estimated from noisy samples, hence no per-fit hard bound)
    db = np.abs(np.abs(p_ue[:, 4]) - np.abs(p_uc[:, 4]))
    assert np.median(db) <= fitref.FORK_TYPICAL and err(p_ue) <= 3 * err(p_uc)


def test_cli_parser_and_header_keys(gp, ora):
    from gppd_b200 import cli
    assert cli.build_parser().parse_args(["-c", "ellipse", "x.fits"]).center == "ellipse"
    ell = np.arange(240, dtype=np.float64).reshape(40, 6)
    keys = gp.ellipse_keys(ell)
    pat = re.compile(r"DEMODULATION ELLIPSE (X0|Y0|RATIO|ANGLE) (FT|SC) T[1-4] (D[1-4]|FC)$")
    assert len(keys) == 160 and all(pat.match(k) for k in keys)
    assert keys == er.ellipse_keys(ell)
    assert keys["DEMODULATION ELLIPSE RATIO SC T2 FC"] == ell[ora.idx(ora.SC, 2, ora.FC) - 1, 2]


def test_ellipse_flag_agrees_everywhere(gp):
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    hdr = open(os.path.join(root, "include", "gppd.h")).read()
    jl = open(os.path.join(root, "julia", "GPPDB200.jl")).read()
    assert int(re.search(r"#define GPPD_CENTER_ELLIPSE (0x[0-9a-f]+)u", hdr).group(1), 16) == 128
    assert int(re.search(r"#define GPPD_ELLIPSE_STRIDE (\d+)", hdr).group(1)) == 6
    assert gp._lib.CENTER_ELLIPSE == 128 and gp._lib.ELLIPSE_STRIDE == 6
    assert re.search(r"const GPPD_CENTER_ELLIPSE\s*=\s*UInt32\(128\)", jl)
    assert re.search(r"const GPPD_ELLIPSE_STRIDE\s*=\s*6", jl)


# ---------------------------------------------------------------------------- GPU
def _fs_gpu(gp, tab):
    fs = tab["faintstates"]
    return None if fs is None else gp.FaintStates(fs.timer1, fs.timer2, 1.0, 2.0)


def _run(gp, tab, **kw):
    ell, st = np.empty((40, 6)), np.empty(40, dtype=np.int32)
    res = gp.process_table(tab["time_us"], tab["volt"], tab["mjd"], offsets="ellipse",
                           faintparam=_fs_gpu(gp, tab), ellipses_out=ell, ellipse_status_out=st, **kw)
    return res, ell, st


@pytest.mark.gpu
@pytest.mark.parametrize("faint", [False, True])
@pytest.mark.parametrize("n", [700, 5000, 20011])
def test_ellipses_match_oracle(gp, ora, n, faint):
    tab = _case(gp, ora, n, k=51, faint=faint)
    _, ell, st = _run(gp, tab)
    z = _cmplx(tab["volt"])
    want, wst = er.compute_ellipses(z, tab["state"])
    assert np.array_equal(st, wst)
    tol = _solve_tolerance(z, tab["state"])
    scale = np.abs(z - (want[:, 0] + 1j * want[:, 1])[None, :]).max(axis=0)
    assert (np.abs((ell[:, 0] - want[:, 0]) + 1j * (ell[:, 1] - want[:, 1])) <= tol * scale).all()
    assert (np.abs(ell[:, 2:4] - want[:, 2:4]).max(axis=1) <= tol).all()
    if not faint:
        assert (tol == ELL_TOL).sum() >= 36          # bright tables: the plain bound almost everywhere
    assert np.abs(ell[:, 4] - np.tan(ell[:, 3])).max() <= 1e-15 and (st == 2).sum() >= 20


def _compose(gp, ora, tab, ell, state, window=None, keepraw=False):
    """the correction on the host with the returned maps, then the array path"""
    t = ora.make_times(tab["time_us"], tab["mjd"])
    zc = er.apply_ellipses(_cmplx(tab["volt"]), ell)
    wrows, _ = gp.table_windows(tab["time_us"], tab["mjd"], window)
    out, par, like = gp.demodulateall(t, zc, faintparam=state, nwindow=wrows if window else 0, raw=True)
    if keepraw:
        v = np.empty((t.size, 144), dtype=np.float32)
        v[:, :80] = tab["volt"]
        v[:, 80::2], v[:, 81::2] = out[:, :32].real, out[:, :32].imag
    else:
        v = np.empty((t.size, 80), dtype=np.float32)
        v[:, 0::2], v[:, 1::2] = out.real, out.imag
    return v, par, like


@pytest.mark.gpu
@pytest.mark.parametrize("faint,window,keepraw", [(False, None, False), (True, None, False),
                                                  (True, 1.0, False), (False, None, True), (True, 1.0, True)])
def test_ellipse_mode_is_correction_plus_array_path(gp, ora, faint, window, keepraw):
    tab = _case(gp, ora, 6000, k=52, faint=faint)
    (vout, par, chi2, _, state), ell, _ = _run(gp, tab, window=window, keepraw=keepraw)
    if faint:
        assert np.array_equal(state, tab["state"])
    v, p, c = _compose(gp, ora, tab, ell, state, window, keepraw)
    assert par.tobytes() == p.tobytes() and chi2.tobytes() == c.tobytes()
    assert vout.tobytes() == v.tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("faint", [False, True])
def test_ellipse_big_endian_table_bytes(gp, ora, faint):
    tab = _case(gp, ora, 3000, k=53, faint=faint)
    (v0, p0, c0, _, s0), ell0, _ = _run(gp, tab)
    L, h = gp._lib.lib(), gp.default_handle()
    tu_be, v_be = tab["time_us"].astype(">i4"), tab["volt"].astype(">f4")
    o = gp.api._options(ellipse=True)
    o.flags |= gp._lib.BIG_ENDIAN
    vout = np.empty((3000, 80), dtype=">f4")
    par, chi2, st = np.empty((32, 6)), np.empty(32), np.empty(3000, dtype=np.int8)
    fs = _fs_gpu(gp, tab)
    t1, t2 = (fs.timer1, fs.timer2) if fs else (None, None)
    gp._lib.check(L.gppd_process_table_f32(
        h.raw, 3000, tu_be.ctypes.data_as(gp._lib._i32p), tab["mjd"], v_be.ctypes.data_as(gp._lib._fp), None,
        gp._lib.ptr(t1), 0 if t1 is None else t1.size, gp._lib.ptr(t2), 0 if t2 is None else t2.size, 0.0,
        C.byref(o), vout.ctypes.data_as(gp._lib._fp), par.ctypes.data_as(gp._lib._dp),
        chi2.ctypes.data_as(gp._lib._dp), None, st.ctypes.data_as(gp._lib._i8p)))
    ell, _ = gp.ellipses()
    assert ell[0].tobytes() == ell0.tobytes()
    assert np.array_equal(vout.astype(np.float32), v0) and par.tobytes() == p0.tobytes()
    assert chi2.tobytes() == c0.tobytes()


@pytest.mark.gpu
def test_ellipse_processmetrology_vs_oracle(gp, ora):
    import fitref
    tab = _case(gp, ora, 5000, k=33, faint=True)
    fs_o = tab["faintstates"]
    tg, hg = gp.processmetrology({"TIME": tab["time_us"], "VOLT": tab["volt"]}, tab["mjd"],
                                 faintparam=_fs_gpu(gp, tab), offsets="ellipse")
    to, ho = er.processmetrology(tab["time_us"], tab["volt"], tab["mjd"], faintparam=fs_o, nthreads=8)
    assert set(hg) == set(ho) and sum("ELLIPSE" in k for k in hg) == 160
    for k in hg:
        if "ELLIPSE" in k:
            assert abs(hg[k] - ho[k]) <= 1e-9 * max(1.0, abs(ho[k])), k
    keys = [k for k in ho if "SIN AMPLITUDE" in k]
    close = sum(abs(hg[k] - ho[k]) <= 1e-6 * abs(ho[k]) for k in keys)
    # (the maps agree to 1e-10 only, hence 1e-6 rather than 1e-9; forks inside the envelope)
    assert close >= fitref.MIN_COINCIDE and all(abs(hg[k] - ho[k]) <= fitref.FORK_HARD for k in keys)
    assert np.abs(tg["VOLT"][:, 64:].astype(np.float64) - to["VOLT"][:, 64:]).max() <= 1e-6


@pytest.mark.gpu
def test_ellipse_degenerate_channels(gp, ora):
    tab = _case(gp, ora, 4096 + 17, k=54)
    _, ell_ref, st_ref = _run(gp, tab)
    volt = tab["volt"].copy()
    volt[:, 2 * 39], volt[:, 2 * 39 + 1] = 0.25, -0.5               # FC channel 40: one point
    x = np.linspace(-1, 1, volt.shape[0], dtype=np.float32)
    volt[:, 2 * 38], volt[:, 2 * 38 + 1] = x, 0.5 * x                # FC channel 39: a line
    th = np.linspace(0, 2 * np.pi, volt.shape[0], endpoint=False)
    volt[:, 2 * 37], volt[:, 2 * 37 + 1] = 0.3 * np.cos(th), 0.01 * np.sin(th) + 0.2   # axis ratio 30
    (vout, _, _, _, _), ell, st = _run(gp, dict(tab, volt=volt))
    want, wst = er.compute_ellipses(_cmplx(volt), None)
    assert np.array_equal(st, wst) and list(st[37:]) == [1, 0, 0]
    assert (ell[38:, :2] == 0).all() and (ell[37:, 2:] == [1, 0, 0, 1]).all()
    assert abs(complex(*ell[37, :2]) - complex(*want[37, :2])) <= 1e-9
    # the FC channels without a circle pass through unchanged; the other channels are unaffected
    assert np.array_equal(vout[:, 76:80], volt[:, 76:80])
    assert ell[:37].tobytes() == ell_ref[:37].tobytes() and np.array_equal(st[:37], st_ref[:37])


@pytest.mark.gpu
def test_ellipse_batch_independent(gp, ora):
    import torch
    L, h = gp._lib.lib(), gp.default_handle()
    tabs = [_case(gp, ora, n, k=60 + i, faint=i == 1) for i, n in enumerate((4096 * 2 + 5, 3001, 9999))]
    alone = []
    for tb in tabs:
        (v, p, c, _, _), e, s = _run(gp, tb, window=1.0)
        alone.append((v, p, c, e, s))
    dev = torch.device("cuda", h.device)
    F = len(tabs)
    wr = [gp.table_windows(tb["time_us"], tb["mjd"], 1.0) for tb in tabs]
    tt = [torch.from_numpy(tb["time_us"]).to(dev) for tb in tabs]
    vv = [torch.from_numpy(tb["volt"]).to(dev) for tb in tabs]
    oo = [torch.empty((tb["volt"].shape[0], 80), dtype=torch.float32, device=dev) for tb in tabs]
    pp = [torch.empty((w[1] * 32, 6), dtype=torch.float64, device=dev) for w in wr]
    cc = [torch.empty(w[1] * 32, dtype=torch.float64, device=dev) for w in wr]
    fss = [_fs_gpu(gp, tb) for tb in tabs]
    vp = lambda ts: (C.c_void_p * F)(*[t.data_ptr() for t in ts])
    i64 = lambda v: (C.c_int64 * F)(*v)
    dpp = lambda arrs: (gp._lib._dp * F)(*[C.cast(None, gp._lib._dp) if a is None else a.ctypes.data_as(gp._lib._dp)
                                          for a in arrs])
    o = gp.api._options(ellipse=True)
    torch.cuda.synchronize()
    gp._lib.check(L.gppd_process_tables_f32_dev(
        h.raw, 0, None, F, i64([tb["volt"].shape[0] for tb in tabs]), i64([w[0] for w in wr]), vp(tt),
        (C.c_double * F)(*[tb["mjd"] for tb in tabs]), vp(vv), None,
        dpp([f.timer1 if f else None for f in fss]), i64([f.timer1.size if f else 0 for f in fss]),
        dpp([f.timer2 if f else None for f in fss]), i64([f.timer2.size if f else 0 for f in fss]),
        C.byref(o), vp(oo), vp(pp), vp(cc), None, None))
    gp._lib.check(L.gppd_wait(h.raw, 0))
    ell, st = gp.ellipses(h, 0, F)
    for i, (v, p, c, e, s) in enumerate(alone):
        assert ell[i].tobytes() == e.tobytes() and np.array_equal(st[i], s)
        assert oo[i].cpu().numpy().tobytes() == v.tobytes()
        assert pp[i].cpu().numpy().tobytes() == p.tobytes() and cc[i].cpu().numpy().tobytes() == c.tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["whole", "window"])
@pytest.mark.parametrize("native", [True, False])
def test_cli_ellipse_files(gp, ora, tmp_path, mode, native, monkeypatch):
    from gppd_b200 import cli, fits
    d, out = str(tmp_path / "night"), str(tmp_path / "out")
    os.makedirs(os.path.join(d, "sub"))
    tabs = {"bright": _case(gp, ora, 3000, k=41), "faint": _case(gp, ora, 3000, k=42, faint=True)}
    gp.synthetic.make_fits(os.path.join(d, "bright.fits"), tabs["bright"])
    gp.synthetic.make_fits(os.path.join(d, "sub", "faint.fits"), tabs["faint"], tabs["faint"]["header"])
    argv = ["-r", "-d", out, "-s", "_demod", "-c", "ellipse"] + (["-w", "2.0"] if mode == "window" else [])
    argv += [] if native else ["--no-native"]
    assert cli.main(argv + [d]) == 0
    for name, sub in (("bright", ""), ("faint", "sub")):
        tab = tabs[name]
        src = fits.read_fits(os.path.join(d, sub, name + ".fits"))
        dst = fits.read_fits(os.path.join(out, name + "_demod.fits"))
        for a, b in zip(src[:3], dst[:3]):                      # every other HDU: byte-exact copy
            assert a.cards == b.cards and a.data == b.data
        ell = np.empty((40, 6))
        vg = gp.process_table(tab["time_us"], tab["volt"], tab["mjd"], offsets="ellipse",
                              faintparam=_fs_gpu(gp, tab), window=2.0 if mode == "window" else None,
                              ellipses_out=ell)[0]
        rb, n, cols = fits.bintable_layout(dst[3].header)
        rec = np.frombuffer(dst[3].data, np.uint8, n * rb).reshape(n, rb)
        assert np.array_equal(rec[:, 4:324].copy().view(">f4").astype(np.float32), vg)
        srec = np.frombuffer(src[3].data, np.uint8, n * 332).reshape(n, 332)
        assert np.array_equal(rec[:, :4], srec[:, :4])
        po = cols["POWER_LASER"][0]
        assert np.array_equal(rec[:, po:po + 8], srec[:, 324:332])
        for k, v in gp.ellipse_keys(ell).items():
            assert dst[3].header[k] == v, k


@pytest.mark.gpu
def test_ellipse_errors(gp, ora):
    L, h = gp._lib.lib(), gp.default_handle()
    tab = _case(gp, ora, 1000, k=55)
    vout, par, chi2 = np.empty((1000, 80), dtype=np.float32), np.empty((32, 6)), np.empty(32)

    def table(flags, mask=0):
        o = gp.api._options(ellipse=True)
        o.flags |= flags
        o.group_mask = mask
        return L.gppd_process_table_f32(
            h.raw, 1000, tab["time_us"].ctypes.data_as(gp._lib._i32p), tab["mjd"],
            tab["volt"].ctypes.data_as(gp._lib._fp), None, None, 0, None, 0, 0.0, C.byref(o),
            vout.ctypes.data_as(gp._lib._fp), par.ctypes.data_as(gp._lib._dp), chi2.ctypes.data_as(gp._lib._dp),
            None, None)

    assert table(gp._lib.CENTER_EMPIRICAL) == 1 and table(gp._lib.FITOFFSETS) == 1   # GPPD_ERR_ARG
    assert table(0, mask=0x0f) == 5                                                  # GPPD_ERR_UNSUPPORTED
    assert table(0) == 0
    t = ora.make_times(tab["time_us"], tab["mjd"])
    z = np.asfortranarray(_cmplx(tab["volt"]))
    o = gp.api._options(ellipse=True)
    out = np.empty((1000, 40), dtype=np.complex128, order="F")
    rc = L.gppd_demodulate_f64(h.raw, 1000, 0, t.ctypes.data_as(gp._lib._dp),
                               z.T.reshape(-1).view(np.float64).ctypes.data_as(gp._lib._dp), None, C.byref(o),
                               out.T.reshape(-1).view(np.float64).ctypes.data_as(gp._lib._dp),
                               par.ctypes.data_as(gp._lib._dp), chi2.ctypes.data_as(gp._lib._dp), None, None)
    assert rc == 5
