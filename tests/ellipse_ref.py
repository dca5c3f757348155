"""CPU restatement of `--center ellipse` (GPPD_CENTER_ELLIPSE, definition in include/gppd.h)
on top of the oracle -- TEST INFRASTRUCTURE ONLY, like ``oracle``: the ellipse fit by lstsq,
the correction in float64 NumPy (no FMA) and processmetrology(offsets = "ellipse") on arrays.
"""
import numpy as np

import oracle

ELLIPSE_MIN_DET = 4 * 0.01 / 1.01 ** 2     # 4AC - B^2 at an axis ratio of 10 (with A + C = 1)


def _kasa(x, y):
    """(centre, True) of the algebraic circle, or (0, False) when there is none."""
    if x.size < 3:
        return 0j, False
    xm, ym = x.mean(), y.mean()
    u, v = x - xm, y - ym
    A = np.stack([2 * u, 2 * v, np.ones_like(u)], axis=1)
    sol, _, rank, _ = np.linalg.lstsq(A, u * u + v * v, rcond=1e-9)
    if rank < 3:
        return 0j, False
    return complex(xm + sol[0], ym + sol[1]), True


def ellipse_fit(x, y):
    """`--center ellipse` for one channel: (x0, y0, r, alpha, status).

    The algebraic least-squares conic A u^2 + B uv + C v^2 + D u + E v + F = 0 under
    A + C = 1, i.e. the linear problem A (u^2 - v^2) + B uv + D u + E v + F = -v^2, solved
    by lstsq on the samples shifted to their centroid and scaled to unit rms radius.
    Centre: [2A B; B 2C] (x0, y0) = -(D, E); gain ratio r = sqrt(C/A); quadrature error
    alpha = asin(B / (2 sqrt(AC))).  status 2 = ellipse; 1 = no ellipse (fewer than 5
    points, rank-deficient design, A <= 0 or C <= 0, axis ratio above 10): the circle
    centre of `oracle.circle_centre` with r = 1, alpha = 0; 0 = no circle either: centre 0."""
    x = np.asarray(x, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    c, ok = _kasa(x, y)
    fallback = (c.real, c.imag, 1.0, 0.0, 1 if ok else 0)
    if x.size < 5:
        return fallback
    xm, ym = x.mean(), y.mean()
    u, v = x - xm, y - ym
    s = np.sqrt(np.mean(u * u + v * v))
    if not s > 0:
        return fallback
    u, v = u / s, v / s
    M = np.stack([u * u - v * v, u * v, u, v, np.ones_like(u)], axis=1)
    sol, _, rank, _ = np.linalg.lstsq(M, -v * v, rcond=1e-6)
    if rank < 5:
        return fallback
    A, B, D, E = sol[0], sol[1], sol[2], sol[3]
    C = 1.0 - A
    det = 4 * A * C - B * B
    if not (A > 0 and C > 0 and det > ELLIPSE_MIN_DET):
        return fallback
    xs = (B * E - 2 * C * D) / det
    ys = (B * D - 2 * A * E) / det
    return (float(xm + xs * s), float(ym + ys * s), float(np.sqrt(C / A)),
            float(np.arcsin(B / (2 * np.sqrt(A * C)))), 2)


def compute_ellipses(cmplxV, state=None):
    """`ellipse_fit` of each of the 40 channels over the samples `oracle.compute_offsets` uses
    (the HIGH samples when there are states).  Returns (ell (40, 6) = x0, y0, r, alpha,
    m21 = tan alpha, m22 = r / cos alpha; status (40,) int32)."""
    cmplxV = np.asarray(cmplxV)
    sel = slice(None) if state is None else (np.asarray(state) == oracle.HIGH)
    ell = np.empty((40, 6))
    status = np.empty(40, dtype=np.int32)
    for ch in range(40):
        x0, y0, r, al, st = ellipse_fit(cmplxV[sel, ch].real, cmplxV[sel, ch].imag)
        ell[ch] = (x0, y0, r, al, np.tan(al), r / np.cos(al))
        status[ch] = st
    return ell, status


def apply_ellipses(cmplxV, ell):
    """The correction of every row: x' = x - x0, y' = m21 x' + m22 (y - y0) in float64,
    every operation rounded (NumPy has no FMA); ell as returned by `compute_ellipses`."""
    z = np.asarray(cmplxV, dtype=np.complex128)
    ell = np.asarray(ell, dtype=np.float64).reshape(40, 6)
    xp = z.real - ell[:, 0]
    yp = ell[:, 4] * xp + ell[:, 5] * (z.imag - ell[:, 1])
    out = np.empty(z.shape, dtype=np.complex128)
    out.real = xp
    out.imag = yp
    return out


def ellipse_keys(ell) -> dict:
    """Header keywords of `--center ellipse`: DEMODULATION ELLIPSE {X0|Y0|RATIO|ANGLE}
    {FT|SC} T{1-4} {D1-D4|FC} (160 values) from the (40, 6) maps."""
    ell = np.asarray(ell, dtype=np.float64).reshape(40, 6)
    hdr = {}
    for s, sn in ((oracle.FT, "FT"), (oracle.SC, "SC")):
        for j in range(1, 5):
            for d, dn in ((oracle.D1, "D1"), (oracle.D2, "D2"), (oracle.D3, "D3"), (oracle.D4, "D4"), (oracle.FC, "FC")):
                ch = oracle.idx(s, j, d) - 1
                for q, k in (("X0", 0), ("Y0", 1), ("RATIO", 2), ("ANGLE", 3)):
                    hdr[f"DEMODULATION ELLIPSE {q} {sn} T{j} {dn}"] = float(ell[ch, k])
    return hdr


def processmetrology(time_us, volt, mjd, faintparam=None, keepraw=False, onlyhigh=False, nthreads=1,
                     maxfun=60):
    """oracle.processmetrology with offsets = "ellipse", whole-file mode: the ellipses of the
    channels (the HIGH samples of a FAINT table), the correction of every row, demodulateall
    in the NoOffsets model; the header holds the whole-file keys and `ellipse_keys`.
    Returns (table dict, hdr dict)."""
    volt32 = np.asarray(volt, dtype=np.float32)
    times = oracle.make_times(time_us, mjd)
    state = None if faintparam is None else oracle.buildstates(faintparam, times)
    v = volt32.astype(np.float64)
    ell, _ = compute_ellipses(v[:, 0::2] + 1j * v[:, 1::2], state)
    cmplx = apply_ellipses(v[:, 0::2] + 1j * v[:, 1::2], ell)
    out, param, _ = oracle.demodulateall(times, cmplx, faintparam=state, onlyhigh=onlyhigh,
                                         nthreads=nthreads, maxfun=maxfun)
    hdr = {}
    for s, sn in ((oracle.FT, "FT"), (oracle.SC, "SC")):
        for j in range(1, 5):
            for d in range(1, 5):
                ch = oracle.idx(s, j, d) - 1
                b, phi = param[ch, 4], param[ch, 5]
                if b < 0:
                    b, phi = -b, float(np.remainder(phi + np.pi + np.pi, 2 * np.pi) - np.pi)
                a = complex(param[ch, 2], param[ch, 3])
                suffix = f"{sn} T{j} D{d}"
                hdr[f"DEMODULATION AMPLITUDE ABS {suffix}"] = abs(a)
                hdr[f"DEMODULATION AMPLITUDE ARG {suffix}"] = float(np.angle(a))
                hdr[f"DEMODULATION SIN AMPLITUDE {suffix}"] = b
                hdr[f"DEMODULATION SIN PHASE {suffix}"] = phi
    hdr.update(ellipse_keys(ell))
    if keepraw:
        s = np.empty((v.shape[0], 144))
        s[:, :80] = v
        s[:, 80::2], s[:, 81::2] = out[:, :32].real, out[:, :32].imag
        v = s
    else:
        v = v.copy()
        v[:, 0::2], v[:, 1::2] = out.real, out.imag
    hdr["PROCSOFT"] = "GPPupilDemodulation.jl"
    return {"VOLT": v.astype(np.float32)}, hdr
