"""ctypes binding of tests/tools/oracle_jvp.c (+ its 80-bit twin oracle_jvp_ld.c): the forward-mode oracle of the K5g kernel and
of the gradient with PSD features.  TEST INFRASTRUCTURE ONLY.

The library is compiled on first use with the flags of oracle/Makefile, together with oracle/pioran_oracle.c (spectral grid and
matrix), into a per-user temporary directory keyed by the sources' hash: the repository tree is never written."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(os.path.dirname(_HERE))
_SRCS = [os.path.join(_ROOT, "oracle", "pioran_oracle.c"), os.path.join(_HERE, "oracle_jvp.c"), os.path.join(_HERE, "oracle_jvp_ld.c")]
_CFLAGS = ["-O3", "-march=native", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-fPIC", "-std=gnu11"]
_dp = C.POINTER(C.c_double)
_lib = None

PSD_MODELS = {"SingleBendingPowerLaw": 0, "DoubleBendingPowerLaw": 1, "SBPL": 0, "DBPL": 1}
BASES = {"SHO": 0, "DRWCelerite": 1}
N_PSD_PAR = {0: 3, 1: 5}


def lib():
    global _lib
    if _lib is not None:
        return _lib
    h = hashlib.sha256()
    for s in _SRCS:
        with open(s, "rb") as f:
            h.update(f.read())
    d = os.path.join(tempfile.gettempdir(), f"pioran_oracle_jvp_{os.getuid()}_{h.hexdigest()[:16]}")
    so = os.path.join(d, "liboracle_jvp.so")
    if not os.path.exists(so):
        os.makedirs(d, exist_ok=True)
        tmp = so + f".{os.getpid()}"
        subprocess.check_call(["gcc"] + _CFLAGS + ["-shared", "-I", _HERE, "-o", tmp] + _SRCS + ["-lm"])
        os.replace(tmp, so)
    L = C.CDLL(so)
    for name in ("orc_celerite_logl_jvp_batch", "orc_celerite_logl_jvp_batch_ld"):
        fn = getattr(L, name)
        fn.restype = None
        fn.argtypes = [C.c_int, C.c_int, C.c_int] + [_dp] * 6 + [C.c_int64] + [_dp] * 15
    for name in ("orc_approx_features_logl_grad_batch", "orc_approx_features_logl_grad_batch_ld"):
        fn = getattr(L, name)
        fn.restype = None
        fn.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, _dp, C.c_double, C.c_double, C.c_int, C.c_double, C.c_double,
                       C.c_int, C.c_int, C.c_int64, _dp, _dp, _dp, _dp, _dp]
    _lib = L
    return L


def _a(x, shape=None):
    if x is None:
        return None
    a = np.ascontiguousarray(x, dtype=np.float64)
    if shape is not None and a.shape != shape:
        raise ValueError(f"expected shape {shape}, got {a.shape}")
    return a


def _p(a):
    return a.ctypes.data_as(_dp) if a is not None else None


def celerite_logl_jvp_batch(a, b, c, d, t, y, s2, *, mu=None, nu=None, y_batch=None, s2_batch=None, da=None, db=None, dc=None,
                            dd=None, dmu=None, dnu=None, dy=None, ds2=None, long_double=False):
    """Same shapes as Context.celerite_logl_jvp → (logL [B], dlogL [B × P])."""
    a, b, c, d = (np.atleast_2d(_a(x)) for x in (a, b, c, d))
    B, Jt = a.shape
    t, y, s2 = _a(t), _a(y), _a(s2)
    N = t.shape[0]
    given = [x for x in (da, db, dc, dd, dmu, dnu, dy, ds2) if x is not None]
    P = np.shape(given[0])[1]
    tj, tp, tn = (B, P, Jt), (B, P), (B, P, N)
    args = [_a(da, tj), _a(db, tj), _a(dc, tj), _a(dd, tj), _a(dmu, tp), _a(dnu, tp), _a(dy, tn), _a(ds2, tn)]
    L, G = np.empty(B), np.empty((B, P))
    fn = lib().orc_celerite_logl_jvp_batch_ld if long_double else lib().orc_celerite_logl_jvp_batch
    fn(B, Jt, P, _p(a), _p(b), _p(c), _p(d), _p(_a(mu, (B,))), _p(_a(nu, (B,))), N, _p(t), _p(y), _p(s2),
       _p(_a(y_batch, (B, N))), _p(_a(s2_batch, (B, N))), *[_p(x) for x in args], _p(L), _p(G))
    return L, G


def approx_features_logl_grad_batch(model, theta, n_features, f_min, f_max, J, t, y, s2, basis="SHO", S_low=20.0, S_high=20.0,
                                    is_integrated_power=True, long_double=False):
    """θ rows [psd parameters…, norm, ν, μ, (S₀, f₀, Q)…] → (logL [B], ∂logL/∂θ [B × ncol]), one dual sweep per column."""
    m = PSD_MODELS[model]
    theta = np.atleast_2d(_a(theta))
    B, ncol = theta.shape
    assert ncol == N_PSD_PAR[m] + 3 + 3 * n_features
    t, y, s2 = _a(t), _a(y), _a(s2)
    L, G = np.empty(B), np.empty((B, ncol))
    fn = lib().orc_approx_features_logl_grad_batch_ld if long_double else lib().orc_approx_features_logl_grad_batch
    fn(m, N_PSD_PAR[m], int(n_features), B, _p(theta), f_min, f_max, J, S_low, S_high, int(bool(is_integrated_power)),
       BASES[basis], t.shape[0], _p(t), _p(y), _p(s2), _p(L), _p(G))
    return L, G
