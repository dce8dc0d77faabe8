"""ctypes binding of tests/tools/oracle_sine.c (+ its 80-bit twin oracle_sine_ld.c): the forward-mode oracle of the likelihood with
a sinusoidal mean (pioran_approx_logl_sine_grad).  TEST INFRASTRUCTURE ONLY.

The library is compiled on first use with the flags of oracle/Makefile, together with oracle/pioran_oracle.c (spectral grid and
matrix) and, through an include, oracle/pioran_oracle_grad.c (the dual-number sweep), into a per-user temporary directory keyed
by the sources' hash: the repository tree is never written."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(os.path.dirname(_HERE))
_ORACLE = os.path.join(_ROOT, "oracle")
_SRCS = [os.path.join(_ORACLE, "pioran_oracle.c"), os.path.join(_HERE, "oracle_sine.c"), os.path.join(_HERE, "oracle_sine_ld.c")]
_DEPS = _SRCS + [os.path.join(_ORACLE, "pioran_oracle_grad.c")]
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
    for s in _DEPS:
        with open(s, "rb") as f:
            h.update(f.read())
    d = os.path.join(tempfile.gettempdir(), f"pioran_oracle_sine_{os.getuid()}_{h.hexdigest()[:16]}")
    so = os.path.join(d, "liboracle_sine.so")
    if not os.path.exists(so):
        os.makedirs(d, exist_ok=True)
        tmp = so + f".{os.getpid()}"
        subprocess.check_call(["gcc"] + _CFLAGS + ["-shared", "-I", _HERE, "-I", _ORACLE, "-o", tmp] + _SRCS + ["-lm"])
        os.replace(tmp, so)
    L = C.CDLL(so)
    for name in ("orc_approx_logl_sine_grad_batch", "orc_approx_logl_sine_grad_batch_ld"):
        fn = getattr(L, name)
        fn.restype = None
        fn.argtypes = [C.c_int, C.c_int, C.c_int, _dp, C.c_double, C.c_double, C.c_int, C.c_double, C.c_double, C.c_int,
                       C.c_int, C.c_int64, _dp, _dp, _dp, _dp, _dp, C.c_int]
    _lib = L
    return L


def approx_logl_sine_grad_batch(model, theta, f_min, f_max, J, t, y, s2, basis="SHO", S_low=20.0, S_high=20.0,
                                is_integrated_power=True, nthreads=0, long_double=False):
    """Sinusoidal mean μ + A·sin(2πt/T₀ + ϕ): theta rows = [psd params…, norm, ν, μ, A, ϕ, T₀]; y, s2 the series.
    Returns (logL [B], ∂logL/∂θ [B × (npar + 6)]); long_double: the same code in 80-bit arithmetic, rounded to FP64."""
    m = PSD_MODELS[model]
    theta = np.ascontiguousarray(np.atleast_2d(theta), dtype=np.float64)
    npar = N_PSD_PAR[m]
    if theta.shape[1] != npar + 6:
        raise ValueError(f"theta must have {npar + 6} columns")
    t, y, s2 = (np.ascontiguousarray(x, dtype=np.float64) for x in (t, y, s2))
    out = np.empty(theta.shape[0])
    grad = np.empty(theta.shape)
    fn = lib().orc_approx_logl_sine_grad_batch_ld if long_double else lib().orc_approx_logl_sine_grad_batch
    p = lambda a: a.ctypes.data_as(_dp)
    fn(m, npar, theta.shape[0], p(theta), f_min, f_max, J, S_low, S_high, int(is_integrated_power), BASES[basis], len(t),
       p(t), p(y), p(s2), p(out), p(grad), nthreads)
    return out, grad
