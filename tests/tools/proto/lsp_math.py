"""Generalised Lomb–Scargle periodogram with a floating mean (Zechmeister & Kürster 2009), the definition K9
(csrc/lsp.cuh, pioran_lombscargle) computes: LombScargle.jl's default, `fit_mean = true`, `center_data = true`, normalisation
`:standard`, weights 1/σ² when errors are given.  For one row y on the times t, with w_n = (1/σ²_n) / Σ 1/σ² (or 1/N) and
x_n = 2 f (t_n − t_1):

    Ȳ  = Σ w y          ỹ = y − Ȳ          YY = Σ w ỹ²
    YC = Σ w ỹ cos πx    YS = Σ w ỹ sin πx
    C  = Σ w cos πx      S  = Σ w sin πx
    CC = Σ w cos² πx − C²   SS = Σ w sin² πx − S²   CS = Σ w cos πx sin πx − C·S
    p(f) = (SS·YC² + CC·YS² − 2·CS·YC·YS) / (YY · (CC·SS − CS²))

The phase goes through an exact range reduction (sincospi below), so that sin πx is exactly 0 at integer x, as CUDA's
sincospi gives it.  `dtype=np.longdouble` evaluates the same formulas in 80-bit arithmetic (x86) for triage."""
import numpy as np


def sincospi(x):
    """(sin πx, cos πx) with x reduced exactly: q = rint(2x), r = x − q/2 ∈ [−1/4, 1/4], then the quadrant of q."""
    x = np.asarray(x)
    pi = np.arccos(x.dtype.type(-1))
    q = np.rint(2 * x)
    r = x - q / 2
    s, c = np.sin(pi * r), np.cos(pi * r)
    k = q.astype(np.int64) & 3
    sn = np.where(k == 0, s, np.where(k == 1, c, np.where(k == 2, -s, -c)))
    cs = np.where(k == 0, c, np.where(k == 1, -s, np.where(k == 2, -c, s)))
    return sn, cs


def weights(s2, n, weighted=True, dtype=np.float64):
    if not weighted:
        return np.full(n, dtype(1) / n, dtype=dtype)
    iv = 1 / np.asarray(s2, dtype=dtype)
    return iv / np.sum(iv)


def _basis(t, freq, w, dtype):
    x = (2 * np.asarray(freq, dtype=dtype))[:, None] * (t - t[0])[None, :]   # [F × N]
    sn, cs = sincospi(x)
    C, S = cs @ w, sn @ w
    return sn, cs, (cs * cs) @ w - C * C, (sn * sn) @ w - S * S, (cs * sn) @ w - C * S


def condition(t, freq, s2=None):
    """|CC·SS| / |CC·SS − CS²| per frequency, in 80-bit arithmetic: how much rounding in the normalisers is amplified in p.
    A relative error of ε in CC, SS or CS moves p by up to about ε times this; it is infinite where the basis is degenerate
    (p = 0/0) and about 1e16 where the denominator vanishes to rounding only, as for three points at f = 1/T (the first and
    the last phase coincide and leave two distinct phases for three parameters)."""
    t = np.asarray(t, dtype=np.longdouble)
    _, _, CC, SS, CS = _basis(t, freq, weights(s2, t.shape[0], s2 is not None, np.longdouble), np.longdouble)
    with np.errstate(invalid="ignore", divide="ignore"):
        return (np.abs(CC * SS) / np.abs(CC * SS - CS * CS)).astype(np.float64)


def lombscargle(t, Y, freq, s2=None, dtype=np.float64):
    """Power [B × F] (or [F] for a one-dimensional Y) of the rows of Y on the times t at the frequencies freq (inverse unit
    of t); weights 1/s2 when s2 is given, equal weights otherwise.  0/0 gives NaN, as on the device."""
    t = np.asarray(t, dtype=dtype)
    Y = np.asarray(Y, dtype=dtype)
    one = Y.ndim == 1
    Y = np.atleast_2d(Y)
    w = weights(s2, t.shape[0], s2 is not None, dtype)
    sn, cs, CC, SS, CS = _basis(t, freq, w, dtype)
    yt = Y - (Y @ w)[:, None]
    YY = (yt * yt) @ w
    yw = yt * w[None, :]
    YC, YS = yw @ cs.T, yw @ sn.T                             # [B × F]
    with np.errstate(invalid="ignore", divide="ignore"):
        p = (SS * YC * YC + CC * YS * YS - 2 * CS * YC * YS) / (YY[:, None] * (CC * SS - CS * CS))
    return p[0] if one else p


def frequency_grid(t, F):
    """F log-spaced frequencies from 1/T to 1/(2·min Δt), the grid of the posterior predictive check."""
    t = np.asarray(t, dtype=np.float64)
    if F == 1:
        return np.array([1.0 / (t[-1] - t[0])])
    return np.geomspace(1.0 / (t[-1] - t[0]), 0.5 / np.min(np.diff(t)), F)
