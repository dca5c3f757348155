"""Host-side mirror of the reference's Julia interface for the demodulateall
path (same names, argument meaning and error behaviour), on top of the C ABI.

Reference: ``demodulateall`` src/Modulation.jl:344-435, ``buildstates``
src/Faint.jl:21-73, ``FaintStates`` src/Faint.jl:3-19, ``idx`` src/Modulation.jl:17-22,
``processmetrology`` src/GPPupilDemodulation.jl:128-255,
``buildfaintparameters`` :64-81, ``read_stefan_file`` :84-104.
All numerics run in libgppd.so on the GPU; nothing here computes a fit.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from enum import IntEnum

import numpy as np

from . import _lib
from ._lib import Options, check, lib, ptr
from .synthetic import stefan_centres

M_2PI = 6.283185           # src/Modulation.jl:11
MJD_1970_1_1 = 40587.0     # src/GPPupilDemodulation.jl:15
DAY_TO_SEC = 24 * 60 * 60  # src/GPPupilDemodulation.jl:16


class MetState(IntEnum):   # src/Faint.jl:1
    OFF = 0
    LOW = 1
    NORMAL = 2
    HIGH = 3
    TRANSIENT = -1


class Side(IntEnum):       # src/Modulation.jl:9
    FT = 0
    SC = 16


class Diode(IntEnum):      # src/Modulation.jl:10
    D1 = 1
    D2 = 2
    D3 = 3
    D4 = 4
    FC = 5


FT, SC = Side.FT, Side.SC
D1, D2, D3, D4, FC = Diode.D1, Diode.D2, Diode.D3, Diode.D4, Diode.FC
OFF, LOW, NORMAL, HIGH, TRANSIENT = (MetState.OFF, MetState.LOW, MetState.NORMAL,
                                     MetState.HIGH, MetState.TRANSIENT)


def idx(side, telescope: int, diode) -> int:
    """1-based channel number (src/Modulation.jl:17-22)."""
    r = lib().gppd_idx(int(side), int(telescope), int(diode))
    if r < 0:
        raise ValueError("idx: bad (side, telescope, diode)")
    return r


@dataclass
class ModulationWithOffsets:   # src/Modulation.jl:26-32
    c: complex
    a: complex
    b: float
    ϕ: float
    ω: float = M_2PI


@dataclass
class ModulationNoOffsets:     # src/Modulation.jl:34-39
    a: complex
    b: float
    ϕ: float
    ω: float = M_2PI


class FaintStates:
    """src/Faint.jl:3-19; the constructor swap guarantees timer1 = HIGH series."""

    def __init__(self, timer1, timer2, voltage1, voltage2):
        timer1 = np.ascontiguousarray(timer1, dtype=np.float64)
        timer2 = np.ascontiguousarray(timer2, dtype=np.float64)
        if voltage1 > voltage2:
            timer1, timer2, voltage1, voltage2 = timer2, timer1, voltage2, voltage1
        self.timer1, self.timer2 = timer1, timer2
        self.voltage1, self.voltage2 = float(voltage1), float(voltage2)
        self.state1, self.state2 = MetState.HIGH, MetState.LOW


def buildfaintparameters(hdr) -> FaintStates:
    """src/GPPupilDemodulation.jl:64-81 (hdr: mapping of FITS keywords)."""
    start1 = hdr["ESO INS ANLO3 TIMER1"] + MJD_1970_1_1 * DAY_TO_SEC
    start2 = hdr["ESO INS ANLO3 TIMER2"] + MJD_1970_1_1 * DAY_TO_SEC

    def timer(start, rate, repeat):  # start .+ rate .* (0:(repeat-1)), rounded once
        k = np.arange(int(repeat), dtype=np.longdouble)
        return (np.longdouble(start) + np.longdouble(rate) * k).astype(np.float64)

    return FaintStates(timer(start1, hdr["ESO INS ANLO3 RATE1"], hdr["ESO INS ANLO3 REPEAT1"]),
                       timer(start2, hdr["ESO INS ANLO3 RATE2"], hdr["ESO INS ANLO3 REPEAT2"]),
                       hdr["ESO INS ANLO3 VOLTAGE1"], hdr["ESO INS ANLO3 VOLTAGE2"])


def read_stefan_file(filename=None) -> np.ndarray:
    """The 40 centres of ``--center stefan`` (src/GPPupilDemodulation.jl:84-104)."""
    if filename is None:
        return stefan_centres()
    off = np.zeros(40, dtype=np.complex128)
    with open(filename) as fh:
        for line in fh:
            if line.startswith("avg"):
                v = line.split()
                name = v[1]
                side = Side.FT if name[:2] == "FT" else Side.SC
                dio = Diode.FC if name[4:6] == "FC" else Diode(int(name[5]))
                off[idx(side, int(name[3]), dio) - 1] = 1e-3 * (float(v[2]) + 1j * float(v[4]))
    return off


def buildstates(faintstates: FaintStates, timestamp, lag: int = 0, preswitchdelay=0,
                postwitchdelay=0, handle=None) -> np.ndarray:
    """src/Faint.jl:21-73 -> int8 array of MetState values."""
    h = handle or _lib.default_handle()
    t = np.ascontiguousarray(timestamp, dtype=np.float64)
    out = np.empty(t.size, dtype=np.int8)
    check(lib().gppd_buildstates(h.raw, t.size, ptr(t), ptr(faintstates.timer1),
                                 faintstates.timer1.size, ptr(faintstates.timer2),
                                 faintstates.timer2.size, int(lag), float(preswitchdelay),
                                 float(postwitchdelay), ptr(out, _lib._i8p)))
    return out


def _options(onlyhigh=False, fitoffsets=False, recenter=True, keepraw=False, init="auto",
             method="auto", maxfun=0, empirical=False, groups=0, fp32=False, ellipse=False,
             covariance=False) -> Options:
    o = Options()
    o.group_mask = int(groups) & 0xff
    o.flags = ((_lib.ONLYHIGH if onlyhigh else 0) | (_lib.FITOFFSETS if fitoffsets else 0) |
               (0 if recenter else _lib.NO_RECENTER) | (_lib.KEEPRAW if keepraw else 0) |
               (_lib.CENTER_EMPIRICAL if empirical else 0) | (_lib.FP32 if fp32 else 0) |
               (_lib.CENTER_ELLIPSE if ellipse else 0) | (_lib.COVARIANCE if covariance else 0))
    o.method = {"auto": _lib.METHOD_AUTO, "direct": _lib.METHOD_DIRECT,
                "harmonic": _lib.METHOD_HARMONIC}[method]
    o.maxfun = int(maxfun)
    if isinstance(init, str):
        if init != "auto":
            raise ValueError("init must be 'auto' or a 2-vector")  # init::Union{Symbol,Vector}
        o.has_xinit = 0
    else:
        x = np.asarray(init, dtype=np.float64)
        if x.shape != (2,):
            raise ValueError("init must be 'auto' or a 2-vector")
        o.has_xinit = 1
        o.xinit[0], o.xinit[1] = float(x[0]), float(x[1])
    return o


def _params_to_structs(params, fitoffsets):
    out = []
    for p in params:
        if fitoffsets:
            out.append(ModulationWithOffsets(complex(p[0], p[1]), complex(p[2], p[3]),
                                             float(p[4]), float(p[5])))
        else:
            out.append(ModulationNoOffsets(complex(p[2], p[3]), float(p[4]), float(p[5])))
    return out


def demodulateall(timestamp, data, init="auto", recenter=True, faintparam=None,
                  onlyhigh=False, fitoffsets=False, preswitchdelay=0.01, postwitchdelay=0.3,
                  *, raw=False, nwindow=0, method="auto", maxfun=0, return_info=False,
                  return_trace=False, handle=None, groups=0, return_cov=False, rhoend=0.0):
    """demodulateall(timestamp, data; init, recenter, faintparam, onlyhigh,
    fitoffsets, preswitchdelay, postwitchdelay) -> (output, param, likelihood)
    (src/Modulation.jl:344-435).

    data: (N, 40) complex128.  faintparam: None | FaintStates | vector of MetState.
    Keyword-only extras (not in the reference): ``raw`` returns param as a
    (nwin*32, 6) array (c.re, c.im, a.re, a.im, b, phi); ``nwindow`` runs the
    per-window loop of src/GPPupilDemodulation.jl:204-225 in one call; ``groups`` is
    ``gppd_options.group_mask`` (bit g = (telescope, side) group g of
    src/Modulation.jl:387; 0 = all): only those groups' columns, params and chi2 entries
    are computed, the rest of the returned arrays is unspecified -- see
    ``sharding.gather_groups``.  ``return_cov`` (GPPD_COVARIANCE) appends the
    (nwin*32, 6, 6) parameter covariances (``covariances``); ``rhoend`` is NEWUOA's final
    trust-region radius (0: the reference's 1e-3).
    """
    h = handle or _lib.default_handle()
    t = np.ascontiguousarray(timestamp, dtype=np.float64)
    dat = np.asfortranarray(data, dtype=np.complex128)
    n = t.size
    if dat.shape != (n, 40):
        raise ValueError("voltage and time must have the same number of lines")  # :258
    state = None
    if isinstance(faintparam, FaintStates):          # :366-367
        state = buildstates(faintparam, t, preswitchdelay=preswitchdelay,
                            postwitchdelay=postwitchdelay, handle=h)
    elif faintparam is not None:                     # :368-369
        state = np.ascontiguousarray(np.asarray(faintparam).astype(np.int8))
        if state.shape != (n,):
            raise ValueError("state and time must have the same number of lines")
    o = _options(onlyhigh=onlyhigh, fitoffsets=fitoffsets, recenter=recenter, init=init,
                 method=method, maxfun=maxfun, groups=groups, covariance=return_cov)
    o.rhoend = float(rhoend)
    nwin = int(lib().gppd_num_windows(n, int(nwindow)))
    out = np.empty((n, 40), dtype=np.complex128, order="F")
    params = np.empty((nwin * 32, 6))
    like = np.empty(nwin * 32)
    info = np.zeros((nwin * 32, _lib.INFO_STRIDE), dtype=np.int32)
    trace = np.zeros((nwin * 32, _lib.TRACE_MAX, 3)) if return_trace else None
    check(lib().gppd_demodulate_f64(
        h.raw, n, int(nwindow), ptr(t), ptr(dat.T.reshape(-1).view(np.float64)),
        ptr(state, _lib._i8p), C.byref(o), ptr(out.T.reshape(-1).view(np.float64)),
        ptr(params), ptr(like), ptr(info, _lib._i32p), ptr(trace)))
    res = [out, params if raw else _params_to_structs(params, fitoffsets), like]
    if return_info:
        res.append(info)
    if return_trace:
        res.append(trace)
    if return_cov:
        res.append(covariances(h, 0, nwin * 32))
    return tuple(res)


def covariances(handle=None, slot=0, nfits=32):
    """The (nfits, 6, 6) parameter covariances of the last GPPD_COVARIANCE call on pipeline
    slot ``slot`` (``gppd_covariances``), in params order (c.re, c.im, a.re, a.im, b, phi)."""
    h = handle or _lib.default_handle()
    cov = np.empty((int(nfits), 6, 6))
    check(lib().gppd_covariances(h.raw, int(slot), int(nfits), ptr(cov)))
    return cov


def table_windows(time_us, mjd, window):
    """(rows per window, number of windows) for ``--window`` seconds
    (src/GPPupilDemodulation.jl:192)."""
    tu = np.ascontiguousarray(time_us, dtype=np.int32)
    w, k = C.c_int64(0), C.c_int64(0)
    check(lib().gppd_table_windows(tu.size, ptr(tu, _lib._i32p), float(mjd),
                                   float(window or 0.0), C.byref(w), C.byref(k)))
    return w.value, k.value


def process_table(time_us, volt, mjd, offsets=None, faintparam: FaintStates | None = None,
                  window=None, keepraw=False, onlyhigh=False, method="auto", maxfun=0,
                  handle=None, centres_out=None, fp32=False, ellipses_out=None,
                  ellipse_status_out=None, cov_out=None):
    """Array-level fast path (C ABI ``gppd_process_table_f32``): returns
    (volt_out float32 (N, 80|144), params (nwin*32, 6), chi2, info, state|None).
    ``offsets``: (40,) complex128 centres, ``None`` (fit the centres) or ``True``
    (empirical circle centres, fitted on the device; ``centres_out``, a (40,)
    complex128 array, then receives them).  ``fp32=True`` (GPPD_FP32): the optional
    reduced-precision harmonic sums; parameters within 1e-5 of the FP64 path.
    ``offsets="ellipse"`` (GPPD_CENTER_ELLIPSE): one least-squares ellipse per channel,
    fitted on the device, maps every channel onto a circle before the fit (include/gppd.h);
    ``ellipses_out`` ((40, 6) float64: x0, y0, r, alpha, m21, m22) and
    ``ellipse_status_out`` ((40,) int32: 2 ellipse, 1 circle only, 0 neither) then receive
    the maps.  ``cov_out``, a (nwin*32, 6, 6) float64 array, turns on GPPD_COVARIANCE and
    receives the parameter covariances."""
    h = handle or _lib.default_handle()
    tu = np.ascontiguousarray(time_us, dtype=np.int32)
    v = np.ascontiguousarray(volt, dtype=np.float32)
    n = tu.size
    if v.shape != (n, 80):
        raise ValueError("VOLT must be (N, 80) float32")
    empirical = offsets is True
    ellipse = isinstance(offsets, str) and offsets == "ellipse"
    if isinstance(offsets, str) and not ellipse:
        raise ValueError("offsets: (40,) centres, None, True or 'ellipse'")
    off = (None if (offsets is None or empirical or ellipse)
           else np.ascontiguousarray(offsets, dtype=np.complex128))
    _, nwin = table_windows(tu, mjd, window)
    o = _options(onlyhigh=onlyhigh, keepraw=keepraw, method=method, maxfun=maxfun,
                 empirical=empirical, fp32=fp32, ellipse=ellipse, covariance=cov_out is not None)
    vout = np.empty((n, 144 if keepraw else 80), dtype=np.float32)
    params = np.empty((nwin * 32, 6))
    chi2 = np.empty(nwin * 32)
    info = np.zeros((nwin * 32, _lib.INFO_STRIDE), dtype=np.int32)
    state = np.empty(n, dtype=np.int8) if faintparam is not None else None
    t1 = faintparam.timer1 if faintparam is not None else None
    t2 = faintparam.timer2 if faintparam is not None else None
    check(lib().gppd_process_table_f32(
        h.raw, n, ptr(tu, _lib._i32p), float(mjd), ptr(v, _lib._fp),
        ptr(None if off is None else off.view(np.float64)), ptr(t1),
        0 if t1 is None else t1.size, ptr(t2), 0 if t2 is None else t2.size,
        float(window or 0.0), C.byref(o), ptr(vout, _lib._fp), ptr(params), ptr(chi2),
        ptr(info, _lib._i32p), ptr(state, _lib._i8p)))
    if empirical and centres_out is not None:
        c = np.empty(40, dtype=np.complex128)
        check(lib().gppd_centres(h.raw, 0, 1, ptr(c.view(np.float64))))
        centres_out[:] = c
    if ellipse and (ellipses_out is not None or ellipse_status_out is not None):
        e, st = ellipses(h, 0, 1)
        if ellipses_out is not None:
            ellipses_out[:] = e[0]
        if ellipse_status_out is not None:
            ellipse_status_out[:] = st[0]
    if cov_out is not None:
        cov_out[...] = covariances(h, 0, nwin * 32).reshape(cov_out.shape)
    return vout, params, chi2, info, state


def ellipses(handle=None, slot=0, ntables=1):
    """The maps of the last ``offsets="ellipse"`` call on pipeline slot ``slot``
    (``gppd_ellipses``): (ell (ntables, 40, 6) = x0, y0, r, alpha, m21, m22,
    status (ntables, 40) int32)."""
    h = handle or _lib.default_handle()
    e = np.empty((ntables, 40, _lib.ELLIPSE_STRIDE))
    st = np.empty((ntables, 40), dtype=np.int32)
    check(lib().gppd_ellipses(h.raw, int(slot), int(ntables), ptr(e), ptr(st, _lib._i32p)))
    return e, st


def ellipse_keys(ell) -> dict:
    """Header keywords of ``--center ellipse``, the transform applied to VOLT:
    DEMODULATION ELLIPSE {X0|Y0|RATIO|ANGLE} {FT|SC} T{1-4} {D1-D4|FC} (160 values) from
    the (40, 6) maps of ``ellipses``."""
    ell = np.asarray(ell, dtype=np.float64).reshape(40, 6)
    hdr = {}
    for s in (Side.FT, Side.SC):
        for j in range(1, 5):
            for d in (Diode.D1, Diode.D2, Diode.D3, Diode.D4, Diode.FC):
                # idx() of src/Modulation.jl:17-22, 0-based (no library call: a header helper)
                ch = 32 + s // 4 + (j - 1) if d == Diode.FC else s + (d - 1) + (j - 1) * 4
                for q, k in (("X0", 0), ("Y0", 1), ("RATIO", 2), ("ANGLE", 3)):
                    hdr[f"DEMODULATION ELLIPSE {q} {s.name} T{j} {d.name}"] = float(ell[ch, k])
    return hdr


def _rem2pi_nearest(x):
    return float(np.remainder(x + np.pi, 2 * np.pi) - np.pi)


def demodulation_keys(params, fitoffsets: bool) -> dict:
    """The whole-file header keywords of src/GPPupilDemodulation.jl:174-189 from the
    (32, 6) parameter array (c.re, c.im, a.re, a.im, b, phi)."""
    hdr = {}
    for s in (Side.FT, Side.SC):
        for j in range(1, 5):
            for d in (Diode.D1, Diode.D2, Diode.D3, Diode.D4):
                p = params[idx(s, j, d) - 1]
                b, phi = p[4], p[5]
                if b < 0:
                    b, phi = -b, _rem2pi_nearest(phi + np.pi)
                a = complex(p[2], p[3])
                suffix = f"{s.name} T{j} {d.name}"
                if fitoffsets:
                    hdr[f"DEMODULATION CENTER X0 {suffix}"] = float(p[0])
                    hdr[f"DEMODULATION CENTER Y0 {suffix}"] = float(p[1])
                hdr[f"DEMODULATION AMPLITUDE ABS {suffix}"] = abs(a)
                hdr[f"DEMODULATION AMPLITUDE ARG {suffix}"] = float(np.angle(a))
                hdr[f"DEMODULATION SIN AMPLITUDE {suffix}"] = float(b)
                hdr[f"DEMODULATION SIN PHASE {suffix}"] = float(phi)
    return hdr


def uncertainties(params, cov) -> dict:
    """One-sigma uncertainties of the reported quantities from the (nfits, 6) parameters and
    their (nfits, 6, 6) covariances: |a| and arg a by the delta method on the a block
    (d|a| = (a.re, a.im) / |a|, d arg a = (-a.im, a.re) / |a|^2), b, phi, x0 = c.re and
    y0 = c.im from the diagonal.  (nfits,) arrays keyed ABSA, ARGA, B, PHI, X0, Y0."""
    P = np.asarray(params, dtype=np.float64).reshape(-1, 6)
    V = np.asarray(cov, dtype=np.float64).reshape(-1, 6, 6)
    ar, ai = P[:, 2], P[:, 3]
    r2 = ar * ar + ai * ai
    vrr, vri, vii = V[:, 2, 2], V[:, 2, 3], V[:, 3, 3]
    with np.errstate(invalid="ignore", divide="ignore"):
        var_abs = (ar * ar * vrr + 2 * ar * ai * vri + ai * ai * vii) / r2
        var_arg = (ai * ai * vrr - 2 * ar * ai * vri + ar * ar * vii) / (r2 * r2)
        diag = np.sqrt(np.diagonal(V, axis1=1, axis2=2))
    return {"ABSA": np.sqrt(var_abs), "ARGA": np.sqrt(var_arg), "B": diag[:, 4], "PHI": diag[:, 5],
            "X0": diag[:, 0], "Y0": diag[:, 1]}


def uncertainty_keys(params, cov, fitoffsets: bool) -> dict:
    """The whole-file header keywords of ``--uncertainty``, next to those of
    ``demodulation_keys``: DEMODULATION {AMPLITUDE ABS|AMPLITUDE ARG|SIN AMPLITUDE|SIN PHASE}
    ERR {FT|SC} T{1-4} D{1-4}, and CENTER {X0|Y0} ERR where the CENTER keys are written."""
    u = uncertainties(params, cov)
    hdr = {}
    for s in (Side.FT, Side.SC):
        for j in range(1, 5):
            for d in (Diode.D1, Diode.D2, Diode.D3, Diode.D4):
                ch = s + (d - 1) + (j - 1) * 4      # idx() - 1, src/Modulation.jl:17-22
                suffix = f"{s.name} T{j} {d.name}"
                if fitoffsets:
                    hdr[f"DEMODULATION CENTER X0 ERR {suffix}"] = float(u["X0"][ch])
                    hdr[f"DEMODULATION CENTER Y0 ERR {suffix}"] = float(u["Y0"][ch])
                hdr[f"DEMODULATION AMPLITUDE ABS ERR {suffix}"] = float(u["ABSA"][ch])
                hdr[f"DEMODULATION AMPLITUDE ARG ERR {suffix}"] = float(u["ARGA"][ch])
                hdr[f"DEMODULATION SIN AMPLITUDE ERR {suffix}"] = float(u["B"][ch])
                hdr[f"DEMODULATION SIN PHASE ERR {suffix}"] = float(u["PHI"][ch])
    return hdr


def window_uncertainty_columns(params, cov, n: int, wrows: int, nwin: int, fitoffsets: bool) -> dict:
    """The per-row columns of ``--uncertainty`` in window mode, next to those of
    ``window_columns``: ABSA_ERR, ARGA_ERR, B_ERR, PHI_ERR (and X0_ERR, Y0_ERR), each
    window's values broadcast over its rows, Float32 (n, 32)."""
    u = uncertainties(params, cov)
    rows = np.minimum(np.arange(n) // wrows, nwin - 1)
    names = (("X0", "Y0") if fitoffsets else ()) + ("ABSA", "ARGA", "B", "PHI")
    return {k + "_ERR": u[k].reshape(nwin, 32)[rows].astype(np.float32) for k in names}


def window_columns(params, n: int, wrows: int, nwin: int, fitoffsets: bool) -> dict:
    """The per-row parameter tables of window mode (src/GPPupilDemodulation.jl:209-247):
    each window's values broadcast over its rows, Float32 (n, 32)."""
    P = np.asarray(params).reshape(nwin, 32, 6)
    b, phi = P[:, :, 4].copy(), P[:, :, 5].copy()
    neg = b < 0
    phi[neg] = np.remainder(phi[neg] + np.pi + np.pi, 2 * np.pi) - np.pi
    b[neg] = -b[neg]
    a = P[:, :, 2] + 1j * P[:, :, 3]
    rows = np.minimum(np.arange(n) // wrows, nwin - 1)

    def col(x):
        return x[rows].astype(np.float32)

    out = {}
    if fitoffsets:
        out["X0"], out["Y0"] = col(P[:, :, 0]), col(P[:, :, 1])
    out["ABSA"], out["ARGA"] = col(np.abs(a)), col(np.angle(a))
    out["B"], out["PHI"] = col(b), col(phi)
    return out


def processmetrology(table, mjd, window=None, faintparam: FaintStates | None = None,
                     keepraw=False, verb=False, onlyhigh=False, offsets=True, handle=None,
                     method="auto", uncertainty=False):
    """processmetrology(metrologyhdu, mjd; window, faintparam, keepraw, verb,
    onlyhigh, offsets) -> (table, hdr)   (src/GPPupilDemodulation.jl:128-255).

    ``table``: mapping with the METROLOGY columns ``TIME`` (N,) int32 and ``VOLT``
    (N, 80) float32 (other columns are passed through).  ``offsets``: (40,)
    complex128 centres, ``False`` (fit the centres) or ``True`` (the default:
    empirical centres, ``compute_offsets`` :105-125 -- one least-squares circle per
    channel over the HIGH samples of a FAINT table, all samples otherwise.  The
    reference throws here because its ``Circle`` is undefined; this is the algebraic
    circle fit that call stands for) or ``"ellipse"`` (one ellipse per channel, see
    ``process_table``; the header then records the maps, ``ellipse_keys``).
    ``uncertainty`` adds the one-sigma uncertainties (``uncertainty_keys``,
    ``window_uncertainty_columns``)."""
    out = dict(table)
    hdr = {}
    ell = np.empty((40, 6)) if isinstance(offsets, str) and offsets == "ellipse" else None
    if ell is not None:
        off = "ellipse"
    elif offsets is True:
        off = True
    else:
        off = None if offsets is False else np.asarray(offsets, dtype=np.complex128)
    fitoffsets = off is None
    wrows, nwin = table_windows(table["TIME"], mjd, window)
    cov = np.empty((nwin * 32, 6, 6)) if uncertainty else None
    vout, params, chi2, info, state = process_table(
        table["TIME"], table["VOLT"], mjd, offsets=off, faintparam=faintparam, window=window,
        keepraw=keepraw, onlyhigh=onlyhigh, handle=handle, method=method, ellipses_out=ell,
        cov_out=cov)
    n = vout.shape[0]
    if window is None:
        hdr.update(demodulation_keys(params, fitoffsets))
        if uncertainty:
            hdr.update(uncertainty_keys(params, cov, fitoffsets))
    else:
        out.update(window_columns(params, n, wrows, nwin, fitoffsets))
        if uncertainty:
            out.update(window_uncertainty_columns(params, cov, n, wrows, nwin, fitoffsets))
        if state is not None:
            out["STATE"] = state.astype(np.int8)   # :248
    if ell is not None:
        hdr.update(ellipse_keys(ell))
    hdr["PROCSOFT"] = "GPPupilDemodulation.jl"     # :252
    out["VOLT"] = vout                             # :253
    return out, hdr
