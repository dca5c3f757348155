"""numpy float64 reference of the parameter covariance of one fit (GPPD_COVARIANCE,
definition in include/gppd.h): the Gauss-Newton covariance s^2 H^-1 of the reported
parameters (c.re, c.im, a.re, a.im, b, phi) at the reported values."""
import numpy as np

OMEGA = 6.283185            # src/Modulation.jl:11
ST_HIGH, ST_NORMAL, ST_TRANSIENT = 3, 2, -1


def valid_rows(state, n, onlyhigh=False):
    """The rows the fit uses (src/Modulation.jl:373-385)."""
    if state is None:
        return np.ones(n, dtype=bool)
    s = np.asarray(state)
    if onlyhigh:
        return (s == ST_HIGH) | (s == ST_NORMAL)
    return s != ST_TRANSIENT


def power_weight(state, d):
    """Per-sample (power, weight): compute_mean_var_power (src/Faint.jl:89-100) in FAINT mode,
    ones in bright mode."""
    if state is None:
        return np.ones(d.size), np.ones(d.size)
    import oracle
    return oracle.compute_mean_var_power(state, d)


def _phase(t, phi):
    """sin and cos of the rounded argument fl(fl(omega t) + phi)."""
    arg = (OMEGA * np.asarray(t, dtype=np.float64)) + phi
    return np.sin(arg), np.cos(arg)


def model(t, fc, params, power):
    """m_n = c + a p_n exp(j b s_n), p_n = power_n FCphasor_n."""
    c, a, b, phi = complex(params[0], params[1]), complex(params[2], params[3]), params[4], params[5]
    s, _ = _phase(t, phi)
    p = power * np.exp(1j * np.angle(fc))
    return c + a * p * np.exp(1j * b * s)


def jacobian(t, fc, params, power):
    """(N, 6) complex dm/dtheta, theta = (c.re, c.im, a.re, a.im, b, phi)."""
    a, b, phi = complex(params[2], params[3]), params[4], params[5]
    s, cs = _phase(t, phi)
    g = power * np.exp(1j * np.angle(fc)) * np.exp(1j * b * s)
    one = np.ones_like(g)
    return np.stack([one, 1j * one, g, 1j * g, 1j * a * s * g, 1j * a * b * cs * g], axis=1)


def covariance(t, d, fc, params, state=None, onlyhigh=False, fitoffsets=False):
    """(6, 6) covariance of one fit: t (N,) seconds, d (N,) complex diode samples (as the fit
    sees them), fc (N,) complex FC samples of the diode's group, params the six reported
    values.  FAINT weights and powers from the oracle's compute_mean_var_power on the
    given rows."""
    t = np.asarray(t, dtype=np.float64)
    d = np.asarray(d, dtype=np.complex128)
    fc = np.asarray(fc, dtype=np.complex128)
    params = np.asarray(params, dtype=np.float64)
    power, weight = power_weight(state, d)
    v = valid_rows(state, t.size, onlyhigh)
    k0 = 0 if fitoffsets else 2
    k = 6 - k0
    nan = np.full((6, 6), np.nan)
    nv = int(v.sum())
    if 2 * nv <= k or np.isnan(params).any():
        return nan
    J = jacobian(t[v], fc[v], params, power[v])[:, k0:]
    w = weight[v]
    H = np.real((J.conj() * w[:, None]).T @ J)
    r = model(t[v], fc[v], params, power[v]) - d[v]
    s2 = float(np.sum(w * np.abs(r) ** 2)) / (2 * nv - k)
    dg = np.diag(H)
    if not (dg > 0).all():
        return nan
    D = 1.0 / np.sqrt(dg)
    Hs = H * D[:, None] * D[None, :]
    # Cholesky with the pivot test of the device pass
    L = np.zeros_like(Hs)
    for j in range(k):
        piv = Hs[j, j] - np.dot(L[j, :j], L[j, :j])
        if not piv > 1e-12:
            return nan
        L[j, j] = np.sqrt(piv)
        L[j + 1:, j] = (Hs[j + 1:, j] - L[j + 1:, :j] @ L[j, :j]) / L[j, j]
    Li = np.linalg.inv(L)
    C = s2 * (Li.T @ Li) * D[:, None] * D[None, :]
    out = np.zeros((6, 6))
    out[k0:, k0:] = C
    return out


def covariances_table(t, z, params, state=None, onlyhigh=False, fitoffsets=False, wrows=None):
    """(nwin*32, 6, 6) for a (N, 40) complex array z, windows of `wrows` rows (None: whole)."""
    n = t.size
    wrows = n if not wrows or wrows >= n else int(wrows)
    nwin = (n + wrows - 1) // wrows
    P = np.asarray(params).reshape(nwin * 32, 6)
    out = np.empty((nwin * 32, 6, 6))
    for w in range(nwin):
        sl = slice(w * wrows, min(n, (w + 1) * wrows))
        st = None if state is None else np.asarray(state)[sl]
        for ch in range(32):
            out[w * 32 + ch] = covariance(t[sl], z[sl, ch], z[sl, 32 + ch // 4], P[w * 32 + ch], st,
                                          onlyhigh, fitoffsets)
    return out
