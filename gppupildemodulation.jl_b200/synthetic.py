"""Deterministic synthetic GRAVITY+-shaped METROLOGY tables (SURVEY.md §8d).

Rows at 500 Hz, ``TIME`` int32 microseconds, 80 float32 ``VOLT`` columns =
40 complex channels (channel c = VOLT[2c-1] + j VOLT[2c], 1-based;
reference src/GPPupilDemodulation.jl:148).  The 32 diode channels follow the
reference's fitted model (src/Modulation.jl:137-141, tex note "Faint model,
guess 2"):  d = c + a * P_state * exp(j Phi_FC) * exp(j b sin(w t + phi)) + e
with w = 6.283185 on ABSOLUTE times (src/Modulation.jl:11,
src/GPPupilDemodulation.jl:139); the 8 FC channels are c_FC + 0.3 exp(j Phi_FC).
NumPy only: no GPU, no oracle.
"""
from __future__ import annotations

import os

import numpy as np

M_2PI = 6.283185
DAY_TO_SEC = 24 * 60 * 60
MJD_1970_1_1 = 40587.0
_HERE = os.path.dirname(os.path.abspath(__file__))


def stefan_centres() -> np.ndarray:
    """The 40 complex centres (volts) of ``--center stefan``
    (reference src/GPPupilDemodulation.jl:84-104: 1e-3*(VX + j VY))."""
    off = np.zeros(40, dtype=np.complex128)
    with open(os.path.join(_HERE, "data", "stefan_centres.txt")) as fh:
        for line in fh:
            if line.startswith("#") or not line.strip():
                continue
            name, vx, vy = line.split()
            side = 0 if name[:2] == "FT" else 16
            tel = int(name[3])
            dio = name[4:6]
            if dio == "FC":
                ch = 32 + side // 4 + (tel - 1) + 1
            else:
                ch = side + (int(dio[1]) - 1) + (tel - 1) * 4 + 1
            off[ch - 1] = 1e-3 * (float(vx) + 1j * float(vy))
    return off


def faint_header(mjd: float, t_first: float = 10.0, rate: float = 3.0,
                 gap: float = 0.5, repeat: int = 60) -> dict:
    """ANLO3 keywords of a FAINT file (reference src/GPPupilDemodulation.jl:64-81).
    TIMERk are unix seconds; VOLTAGE1 < VOLTAGE2 so timer1 is the HIGH series."""
    t0_unix = DAY_TO_SEC * float(mjd) - MJD_1970_1_1 * DAY_TO_SEC
    return {
        "MJD-OBS": float(mjd),
        "ESO INS MET MODE": "FAINT",
        "ESO INS PMC1 MODULATE": True,
        "ESO INS ANLO3 RATE1": rate, "ESO INS ANLO3 RATE2": rate,
        "ESO INS ANLO3 REPEAT1": repeat, "ESO INS ANLO3 REPEAT2": repeat,
        "ESO INS ANLO3 TIMER1": t0_unix + t_first,
        "ESO INS ANLO3 TIMER2": t0_unix + t_first + gap,
        "ESO INS ANLO3 VOLTAGE1": 1.0, "ESO INS ANLO3 VOLTAGE2": 5.0,
    }


def make_table(nrows: int = 100_000, k: int = 0, faint: bool = False,
               jitter: bool = False, noise: float = 0.02, centred: bool = False,
               state=None, seed: int | None = None, quadrature=None):
    """One synthetic file.  Returns a dict with
    ``time_us`` (N,) int32, ``volt`` (N,80) float32, ``mjd``, ``truth``
    (dict of the generating a, b, phi, c per diode), ``header`` (keywords).
    ``state``: optional int8 MetState vector used for the power scale in FAINT
    files (NORMAL 1.0 / HIGH 3.0 / LOW 0.2 / others 1.0); callers obtain it
    from ``buildstates`` so that generator and segmentation agree.
    ``quadrature``: imperfect quadrature detectors (``--center ellipse``), ``(r[40],
    alpha[40])`` or ``True`` for r ~ U(0.85, 1.15), alpha ~ U(-0.15, 0.15) rad drawn from
    a generator of their own (the other draws, hence the default output, do not change).
    Each channel is distorted about its generating centre c with the Heydemann forward
    model x = c.re + U1, y = c.im + (U2 cos alpha - U1 sin alpha) / r; ``truth`` then holds
    ``quad_r``, ``quad_alpha`` and the 40 generating centres ``centres``."""
    mjd = 59949.0 + k / 100.0
    rng = np.random.Generator(np.random.PCG64(20230105 + k if seed is None else seed))
    time_us = (2000 * np.arange(nrows, dtype=np.int64))
    if jitter:
        time_us = time_us + rng.integers(-1, 2, size=nrows)
        time_us[0] = 0
    time_us = time_us.astype(np.int32)
    t = time_us.astype(np.float64) * 1e-6 + DAY_TO_SEC * mjd
    centres = stefan_centres()
    volt = np.empty((nrows, 80), dtype=np.float32)
    truth = dict(a=np.zeros(32, complex), b=np.zeros(32), phi=np.zeros(32),
                 c=np.zeros(32, complex))
    pscale = np.ones(nrows)
    if faint and state is not None:
        st = np.asarray(state)
        pscale = np.where(st == 3, 3.0, np.where(st == 1, 0.2, 1.0))
    wt = M_2PI * t
    quad = None
    if quadrature is True:
        qrng = np.random.Generator(np.random.PCG64(77_000_000 + (k if seed is None else seed)))
        quad = (qrng.uniform(0.85, 1.15, size=40), qrng.uniform(-0.15, 0.15, size=40))
    elif quadrature is not None:
        quad = (np.asarray(quadrature[0], dtype=np.float64).reshape(40),
                np.asarray(quadrature[1], dtype=np.float64).reshape(40))
    gen_c = np.zeros(40, dtype=np.complex128) if centred else centres

    def distort(z, ch):
        if quad is None:
            return z
        r, al = quad[0][ch], quad[1][ch]
        u = z - gen_c[ch]
        return gen_c[ch] + (u.real + 1j * ((u.imag * np.cos(al) - u.real * np.sin(al)) / r))

    for side in (0, 16):
        for tel in range(1, 5):
            fc_ch = 32 + side // 4 + (tel - 1)
            phi_fc = np.cumsum(rng.normal(0.0, 0.02, size=nrows)) + rng.uniform(-np.pi, np.pi)
            fc = (0.0 if centred else centres[fc_ch]) + 0.3 * np.exp(1j * phi_fc)
            fc = distort(fc + 0.002 * (rng.normal(size=nrows) + 1j * rng.normal(size=nrows)), fc_ch)
            volt[:, 2 * fc_ch] = fc.real
            volt[:, 2 * fc_ch + 1] = fc.imag
            for dio in range(4):
                ch = side + dio + (tel - 1) * 4
                amp = rng.uniform(0.05, 0.5)
                a = amp * np.exp(1j * rng.uniform(-np.pi, np.pi))
                b = rng.uniform(0.3, 2.5)
                phi = rng.uniform(-np.pi, np.pi)
                c = 0.0 if centred else centres[ch]
                e = noise * amp * (rng.normal(size=nrows) + 1j * rng.normal(size=nrows))
                d = distort(c + a * pscale * np.exp(1j * phi_fc) * np.exp(1j * b * np.sin(wt + phi)) + e, ch)
                volt[:, 2 * ch] = d.real
                volt[:, 2 * ch + 1] = d.imag
                truth["a"][ch], truth["b"][ch], truth["phi"][ch], truth["c"][ch] = a, b, phi, c
    if quad is not None:
        truth["quad_r"], truth["quad_alpha"], truth["centres"] = quad[0], quad[1], gen_c.copy()
    header = faint_header(mjd) if faint else {
        "MJD-OBS": mjd, "ESO INS MET MODE": "ON", "ESO INS PMC1 MODULATE": True}
    return dict(time_us=time_us, volt=volt, mjd=mjd, truth=truth, header=header)


def to_complex(table, offsets=None):
    """(times, cmplxV) at the demodulateall boundary
    (reference src/GPPupilDemodulation.jl:139,147-152)."""
    t = table["time_us"].astype(np.float64) * 1e-6 + DAY_TO_SEC * table["mjd"]
    v = table["volt"].astype(np.float64)
    z = v[:, 0::2] + 1j * v[:, 1::2]
    if offsets is not None:
        z = z - np.asarray(offsets).reshape(1, 40)
    return t, z


def make_fits(path, table, header=None, modulate=True, met_mode=None):
    """Write ``table`` (make_table) as a GRAVITY-shaped FITS file: primary header with
    the keywords ``main`` looks at (src/GPPupilDemodulation.jl:362-389), a dummy image
    extension and a dummy table before, and the ``METROLOGY`` BINTABLE with columns
    TIME (1J), VOLT (80E), POWER_LASER (1E), LAMBDA_LASER (1E) -- 332-byte records,
    big-endian, as in tex/GPPupilDemodulation.tex:40-52."""
    from . import fits
    n = table["time_us"].size
    keys = [("MJD-OBS", float(table["mjd"])), ("ESO INS PMC1 MODULATE", bool(modulate))]
    hdr = dict(header or {})
    mode = met_mode or hdr.get("ESO INS MET MODE", "ON")
    keys.append(("ESO INS MET MODE", mode))
    for k, v in hdr.items():
        if k not in ("MJD-OBS", "ESO INS PMC1 MODULATE", "ESO INS MET MODE"):
            keys.append((k, v))
    rng = np.random.default_rng(int(n) + 17)
    cols = [("TIME", "1J", "usec", table["time_us"].astype(">i4")),
            ("VOLT", "80E", "V", table["volt"].astype(">f4")),
            ("POWER_LASER", "1E", "mW", rng.normal(1.0, 0.01, n).astype(">f4")),
            ("LAMBDA_LASER", "1E", "nm", np.full(n, 1908.0, dtype=">f4"))]
    img = fits.HDU([fits.format_card("XTENSION", "IMAGE"), fits.format_card("BITPIX", 16),
                    fits.format_card("NAXIS", 2), fits.format_card("NAXIS1", 7),
                    fits.format_card("NAXIS2", 5), fits.format_card("PCOUNT", 0),
                    fits.format_card("GCOUNT", 1), fits.format_card("EXTNAME", "IMAGING_DATA_ACQ")],
                   rng.integers(0, 255, 70, dtype=np.uint8).tobytes(), {})
    for c in img.cards:
        k, v = fits.parse_card(c)
        if k:
            img.header.setdefault(k, v)
    other = fits.make_bintable("OPDC", [("TIME", "1J", "usec", np.arange(11, dtype=">i4")),
                                        ("STATE", "1J", None, rng.integers(0, 9, 11).astype(">i4"))])
    hdus = [fits.make_primary(keys), img, other, fits.make_bintable("METROLOGY", cols)]
    fits.write_fits(path, hdus)
    return path
