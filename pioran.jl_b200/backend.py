"""Thin Python handle on a libpioran_b200 context (one CUDA device).  numpy in, numpy out; every call runs
the sm_100a kernels through the C ABI of include/pioran_b200.h."""
import collections
import ctypes as C
import os

import numpy as np

from . import _lib
from ._lib import ApproxSpec, PriorSpec, check

PSD_MODELS = {"SingleBendingPowerLaw": 0, "DoubleBendingPowerLaw": 1}
N_PSD_PAR = {0: 3, 1: 5}
BASES = {"SHO": 0, "DRWCelerite": 1}

_dp = C.POINTER(C.c_double)


def _f64(x, shape=None):
    a = np.ascontiguousarray(x, dtype=np.float64)
    if shape is not None and a.shape != shape:
        raise ValueError(f"expected shape {shape}, got {a.shape}")
    return a


def _p(a):
    return a.ctypes.data_as(_dp) if a is not None else None


def make_spec(psd_model, f_min, f_max, n_components=20, S_low=20.0, S_high=20.0, is_integrated_power=True,
              basis_function="SHO"):
    if basis_function not in BASES:
        # same failure mode as src/psd.jl:285
        raise ValueError(f"Basis function {basis_function} not implemented")
    model = PSD_MODELS[psd_model] if isinstance(psd_model, str) else int(psd_model)
    return ApproxSpec(model, int(n_components), BASES[basis_function], int(bool(is_integrated_power)), float(f_min),
                      float(f_max), float(S_low), float(S_high))


class Series:
    def __init__(self, ctx, sid, N):
        self.ctx, self.id, self.N = ctx, sid, N

    def free(self):
        if self.id is not None:
            check(self.ctx.lib.pioran_series_free(self.ctx.h, self.id))
            self.id = None


ScanCheck = collections.namedtuple("ScanCheck", "estimate fallback refined")


class Context:
    """pioran_ctx bound to one device."""

    def __init__(self, device=None):
        """device: an int (one GPU), or a sequence of ints — a device group (pioran_ctx_create_multi): one process, the batched
        host entries split their parameter vectors over the devices."""
        self.lib = _lib.load()
        if device is None:
            device = int(os.environ.get("LOCAL_RANK", "0"))
        h = C.c_void_p()
        if isinstance(device, (list, tuple)):
            devs = (C.c_int * len(device))(*[int(d) for d in device])
            check(self.lib.pioran_ctx_create_multi(devs, len(device), C.byref(h)))
            self.device = int(device[0])
        else:
            check(self.lib.pioran_ctx_create(int(device), C.byref(h)))
            self.device = int(device)
        self.h = h

    @property
    def device_count(self):
        return int(self.lib.pioran_ctx_device_count(self.h))

    def close(self):
        if getattr(self, "h", None):
            self.lib.pioran_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- plumbing
    def set_stream(self, cuda_stream_ptr):
        check(self.lib.pioran_ctx_set_stream(self.h, C.c_void_p(cuda_stream_ptr or 0)))

    def synchronize(self):
        check(self.lib.pioran_ctx_synchronize(self.h))

    @property
    def launch_count(self):
        return int(self.lib.pioran_ctx_launch_count(self.h))

    def last_kernel_ms(self):
        """Device time of the most recent K2/K3/K4 launch (CUDA events inside the library)."""
        ms = C.c_double(0.0)
        check(self.lib.pioran_ctx_last_kernel_ms(self.h, C.byref(ms)))
        return ms.value

    def last_kernel_name(self):
        """Kernel of that launch with its template integers, e.g. "blocked<5,5,true,16>" ("" before the first launch)."""
        buf = C.create_string_buffer(64)
        check(self.lib.pioran_ctx_last_kernel_name(self.h, buf, len(buf)))
        return buf.value.decode()

    def upload_series(self, t, y, s2):
        t, y, s2 = _f64(t), _f64(y), _f64(s2)
        if not (t.ndim == 1 and t.shape == y.shape == s2.shape):
            raise ValueError("t, y, s2 must be 1-D arrays of equal length")
        sid = C.c_int(-1)
        check(self.lib.pioran_series_upload(self.h, t.shape[0], _p(t), _p(y), _p(s2), C.byref(sid)))
        return Series(self, sid.value, t.shape[0])

    # -- K1
    def approx_coeffs(self, spec, theta):
        """theta [B × (n_psd_par+1)] → (a, b, c, d) each [B × Jt]  (src/psd.jl:214-289)."""
        theta = np.atleast_2d(_f64(theta))
        npar = N_PSD_PAR[spec.psd_model]
        if theta.shape[1] != npar + 1:
            raise ValueError(f"theta must have {npar + 1} columns (psd parameters, norm)")
        B = theta.shape[0]
        Jt = spec.n_components * (1 if spec.basis == 0 else 2)
        out = [np.empty((B, Jt)) for _ in range(4)]
        check(self.lib.pioran_approx_coeffs(self.h, C.byref(spec), B, _p(theta), *[_p(o) for o in out]))
        return tuple(out)

    def approx_coeffs_features(self, spec, n_features, theta):
        """theta [B × (n_psd_par + 1 + 3·n_features)] = psd parameters…, norm, (S₀, f₀, Q)… → (a, b, c, d) each
        [B × (Jt + n_features)]  (src/psd.jl:214-289 with separate_psd features)."""
        theta = np.atleast_2d(_f64(theta))
        npar = N_PSD_PAR[spec.psd_model]
        if theta.shape[1] != npar + 1 + 3 * n_features:
            raise ValueError(f"theta must have {npar + 1 + 3 * n_features} columns")
        B = theta.shape[0]
        Jt = spec.n_components * (1 if spec.basis == 0 else 2) + n_features
        out = [np.empty((B, Jt)) for _ in range(4)]
        check(self.lib.pioran_approx_coeffs_features(self.h, C.byref(spec), int(n_features), B, _p(theta), *[_p(o) for o in out]))
        return tuple(out)

    def approx_features_logl(self, series, spec, n_features, theta):
        """theta rows = [psd parameters…, norm, ν, μ, (S₀, f₀, Q)…] → logL [B]."""
        theta = np.atleast_2d(_f64(theta))
        npar = N_PSD_PAR[spec.psd_model]
        if theta.shape[1] != npar + 3 + 3 * n_features:
            raise ValueError(f"theta must have {npar + 3 + 3 * n_features} columns")
        out = np.empty(theta.shape[0])
        check(self.lib.pioran_approx_features_logl(self.h, series.id, C.byref(spec), int(n_features), theta.shape[0], _p(theta), _p(out)))
        return out

    # -- K2 generic
    def celerite_logl(self, series, a, b, c, d, mu=None, nu=None, y_batch=None, s2_batch=None):
        """Batched logl(a,b,c,d,τ,y,σ2) (src/celerite_solver.jl:312-334); coefficient arrays [B × Jt]."""
        a, b, c, d = (np.atleast_2d(_f64(x)) for x in (a, b, c, d))
        B, Jt = a.shape
        for x in (b, c, d):
            if x.shape != (B, Jt):
                raise ValueError("a, b, c, d must have the same shape")
        mu = _f64(mu, (B,)) if mu is not None else None
        nu = _f64(nu, (B,)) if nu is not None else None
        yb = _f64(y_batch, (B, series.N)) if y_batch is not None else None
        sb = _f64(s2_batch, (B, series.N)) if s2_batch is not None else None
        out = np.empty(B)
        check(self.lib.pioran_celerite_logl(self.h, series.id, B, Jt, _p(a), _p(b), _p(c), _p(d), _p(mu), _p(nu),
                                            _p(yb), _p(sb), _p(out)))
        return out

    # -- fused approx + logpdf
    def approx_logl(self, series_list, specs, theta, theta_per_series=False):
        """theta rows = [psd parameters…, norm, ν, μ].  Returns logL [S × B]."""
        if isinstance(series_list, Series):
            series_list, specs = [series_list], [specs]
        S = len(series_list)
        npar = N_PSD_PAR[specs[0].psd_model]
        theta = _f64(theta)
        if theta_per_series:
            if theta.ndim != 3 or theta.shape[0] != S or theta.shape[2] != npar + 3:
                raise ValueError(f"theta must be [S, B, {npar + 3}]")
            B = theta.shape[1]
        else:
            theta = np.atleast_2d(theta)
            if theta.shape[1] != npar + 3:
                raise ValueError(f"theta must have {npar + 3} columns (psd parameters, norm, ν, μ)")
            B = theta.shape[0]
        ids = (C.c_int * S)(*[s.id for s in series_list])
        sp = (ApproxSpec * S)(*specs)
        out = np.empty((S, B))
        check(self.lib.pioran_approx_logl(self.h, S, ids, sp, B, _p(theta), int(theta_per_series), _p(out)))
        return out

    # -- device-side prior transform (SURVEY §8f #4)
    @staticmethod
    def _prior_array(priors):
        """priors: sequence of (kind, ref_col, p0, p1) tuples (sampler.PriorTransform.device_spec())."""
        arr = (PriorSpec * len(priors))()
        for k, (kind, ref, p0, p1) in enumerate(priors):
            arr[k] = PriorSpec(int(kind), int(ref), float(p0), float(p1))
        return arr

    def prior_transform(self, priors, cube):
        """Unit-cube points [B × ncol] → parameter vectors [B × ncol] on the device (pioran_prior_transform)."""
        cube = np.atleast_2d(_f64(cube))
        B, ncol = cube.shape
        out = np.empty((B, ncol))
        check(self.lib.pioran_prior_transform(self.h, ncol, self._prior_array(priors), B, _p(cube), _p(out)))
        return out

    def prior_transform_logl(self, series, spec, priors, cube, return_theta=False):
        """Prior transform + fused likelihood in one call; the parameter vectors stay on the device unless return_theta."""
        cube = np.atleast_2d(_f64(cube))
        B, ncol = cube.shape
        out = np.empty(B)
        theta = np.empty((B, ncol)) if return_theta else None
        check(self.lib.pioran_prior_transform_logl(self.h, series.id, C.byref(spec), ncol, self._prior_array(priors), B, _p(cube),
                                                   _p(theta), _p(out)))
        return (out, theta) if return_theta else out

    def approx_logl_logshift(self, series, spec, theta):
        """Log-normal series (docs/src/timeseries.md:16-21): theta rows = [psd parameters…, norm, ν, μ, c];
        yn = log(y − c), σ² = ν σ²/(y − c)², transformed on the device.  Returns logL [B]."""
        npar = N_PSD_PAR[spec.psd_model]
        theta = np.atleast_2d(_f64(theta))
        if theta.shape[1] != npar + 4:
            raise ValueError(f"theta must have {npar + 4} columns (psd parameters, norm, ν, μ, c)")
        out = np.empty(theta.shape[0])
        check(self.lib.pioran_approx_logl_logshift(self.h, series.id, C.byref(spec), theta.shape[0], _p(theta), _p(out)))
        return out

    def approx_logl_dev(self, series_list, specs, B, theta_ptr, out_ptr, theta_per_series=False):
        """Device-resident variant: raw device pointers (ints), asynchronous on the context's stream."""
        S = len(series_list)
        ids = (C.c_int * S)(*[s.id for s in series_list])
        sp = (ApproxSpec * S)(*specs)
        check(self.lib.pioran_approx_logl_dev(self.h, S, ids, sp, int(B), C.c_void_p(theta_ptr), int(theta_per_series),
                                              C.c_void_p(out_ptr)))

    # -- K5: gradient of the fused path
    def approx_logl_grad(self, series, spec, theta):
        """theta rows = [psd parameters…, norm, ν, μ].  Returns (logL [B], ∂logL/∂θ [B × (npar+3)])."""
        npar = N_PSD_PAR[spec.psd_model]
        theta = np.atleast_2d(_f64(theta))
        if theta.shape[1] != npar + 3:
            raise ValueError(f"theta must have {npar + 3} columns (psd parameters, norm, ν, μ)")
        B = theta.shape[0]
        out, grad = np.empty(B), np.empty((B, npar + 3))
        check(self.lib.pioran_approx_logl_grad(self.h, series.id, C.byref(spec), B, _p(theta), _p(out), _p(grad)))
        return out, grad

    def approx_logl_logshift_grad(self, series, spec, theta):
        """Log-normal series: theta rows = [psd parameters…, norm, ν, μ, c] → (logL [B], ∂logL/∂θ [B × (n_psd_par + 4)])."""
        npar = N_PSD_PAR[spec.psd_model]
        theta = np.atleast_2d(_f64(theta))
        if theta.shape[1] != npar + 4:
            raise ValueError(f"theta must have {npar + 4} columns (psd parameters, norm, ν, μ, c)")
        B = theta.shape[0]
        out, grad = np.empty(B), np.empty((B, npar + 4))
        check(self.lib.pioran_approx_logl_logshift_grad(self.h, series.id, C.byref(spec), B, _p(theta), _p(out), _p(grad)))
        return out, grad

    # -- K5g: forward-mode derivatives of the explicit-coefficient likelihood
    def celerite_logl_jvp(self, series, a, b, c, d, *, da=None, db=None, dc=None, dd=None, mu=None, nu=None, dmu=None,
                          dnu=None, y_batch=None, s2_batch=None, dy=None, ds2=None):
        """d/dε of celerite_logl along P directions per coefficient set (ForwardDiff's chunk mode over logl).
        a, b, c, d [B × Jt]; tangents da, db, dc, dd [B × P × Jt], dmu, dnu [B × P], dy, ds2 [B × P × N]; a tangent left out is
        zero, and at least one must be given (P is read from their shapes).  Returns (logL [B], dlogL [B × P])."""
        a, b, c, d = (np.atleast_2d(_f64(x)) for x in (a, b, c, d))
        B, Jt = a.shape
        for x in (b, c, d):
            if x.shape != (B, Jt):
                raise ValueError("a, b, c, d must have the same shape")
        N = series.N
        tangents = {"da": (da, Jt), "db": (db, Jt), "dc": (dc, Jt), "dd": (dd, Jt), "dmu": (dmu, None), "dnu": (dnu, None),
                    "dy": (dy, N), "ds2": (ds2, N)}
        Ps = {name: np.shape(x)[1] for name, (x, _) in tangents.items() if x is not None and np.ndim(x) >= 2}
        if not any(x is not None for x, _ in tangents.values()):
            raise ValueError("at least one tangent (da, db, dc, dd, dmu, dnu, dy, ds2) must be given")
        if len(set(Ps.values())) != 1:
            raise ValueError(f"the tangents disagree on the number of directions P: {Ps}")
        P = next(iter(Ps.values()))
        conv = {name: (_f64(x, (B, P) if inner is None else (B, P, inner)) if x is not None else None)
                for name, (x, inner) in tangents.items()}
        mu = _f64(mu, (B,)) if mu is not None else None
        nu = _f64(nu, (B,)) if nu is not None else None
        yb = _f64(y_batch, (B, N)) if y_batch is not None else None
        sb = _f64(s2_batch, (B, N)) if s2_batch is not None else None
        out, grad = np.empty(B), np.empty((B, P))
        check(self.lib.pioran_celerite_logl_jvp(self.h, series.id, B, Jt, P, _p(a), _p(b), _p(c), _p(d), _p(mu), _p(nu), _p(yb),
                                                _p(sb), *[_p(conv[n]) for n in ("da", "db", "dc", "dd", "dmu", "dnu", "dy", "ds2")],
                                                _p(out), _p(grad)))
        return out, grad

    def approx_features_logl_grad(self, series, spec, n_features, theta):
        """theta rows = [psd parameters…, norm, ν, μ, (S₀, f₀, Q)…] → (logL [B], ∂logL/∂θ [B × n_col]) in the column order of theta."""
        theta = np.atleast_2d(_f64(theta))
        ncol = N_PSD_PAR[spec.psd_model] + 3 + 3 * int(n_features)
        if theta.shape[1] != ncol:
            raise ValueError(f"theta must have {ncol} columns")
        B = theta.shape[0]
        out, grad = np.empty(B), np.empty((B, ncol))
        check(self.lib.pioran_approx_features_logl_grad(self.h, series.id, C.byref(spec), int(n_features), B, _p(theta), _p(out),
                                                        _p(grad)))
        return out, grad

    # -- K5r: reverse-mode gradient of the explicit-coefficient likelihood
    def celerite_logl_vjp(self, series, a, b, c, d, *, mu=None, nu=None, y_batch=None, s2_batch=None, data_grad=False):
        """logL and its gradient with respect to every input of celerite_logl, from one backward sweep per coefficient set.
        a, b, c, d [B × Jt].  Returns (logL [B], {"a", "b", "c", "d" [B × Jt], "mu", "nu" [B]}); with data_grad also "y" and
        "s2" [B × N], the gradient with respect to the data row as it enters (ỹ = y − μ, σ̃² = ν·s2)."""
        a, b, c, d = (np.atleast_2d(_f64(x)) for x in (a, b, c, d))
        B, Jt = a.shape
        for x in (b, c, d):
            if x.shape != (B, Jt):
                raise ValueError("a, b, c, d must have the same shape")
        N = series.N
        mu = _f64(mu, (B,)) if mu is not None else None
        nu = _f64(nu, (B,)) if nu is not None else None
        yb = _f64(y_batch, (B, N)) if y_batch is not None else None
        sb = _f64(s2_batch, (B, N)) if s2_batch is not None else None
        out = np.empty(B)
        g = {k: np.empty((B, Jt)) for k in ("a", "b", "c", "d")}
        g["mu"], g["nu"] = np.empty(B), np.empty(B)
        if data_grad:
            g["y"], g["s2"] = np.empty((B, N)), np.empty((B, N))
        check(self.lib.pioran_celerite_logl_vjp(self.h, series.id, B, Jt, _p(a), _p(b), _p(c), _p(d), _p(mu), _p(nu), _p(yb), _p(sb),
                                                _p(out), *[_p(g[k]) for k in ("a", "b", "c", "d", "mu", "nu")],
                                                _p(g.get("y")), _p(g.get("s2"))))
        return out, g

    def approx_features_logl_grad_reverse(self, series, spec, n_features, theta):
        """approx_features_logl_grad computed in reverse mode (one K5r sweep instead of one forward direction per column)."""
        theta = np.atleast_2d(_f64(theta))
        ncol = N_PSD_PAR[spec.psd_model] + 3 + 3 * int(n_features)
        if theta.shape[1] != ncol:
            raise ValueError(f"theta must have {ncol} columns")
        B = theta.shape[0]
        out, grad = np.empty(B), np.empty((B, ncol))
        check(self.lib.pioran_approx_features_logl_grad_reverse(self.h, series.id, C.byref(spec), int(n_features), B, _p(theta),
                                                                _p(out), _p(grad)))
        return out, grad

    def set_vjp_workspace(self, nbytes):
        """Cap in bytes of the reverse-mode workspace of one θ-chunk (0 = 1 GiB, the default)."""
        check(self.lib.pioran_ctx_set_vjp_workspace(self.h, int(nbytes)))

    def approx_logl_grad_dev(self, series, spec, B, theta_ptr, logl_ptr, grad_ptr):
        """Device-resident variant: raw device pointers (ints); logl_ptr may be 0."""
        check(self.lib.pioran_approx_logl_grad_dev(self.h, series.id, C.byref(spec), int(B), C.c_void_p(theta_ptr),
                                                   C.c_void_p(logl_ptr or 0), C.c_void_p(grad_ptr)))

    def set_sweep_kernel(self, which="auto"):
        """Kernel of the fused path at ranks ≤ 63: "auto" (tensor-pipe, csrc/blocked.cuh) or "scalar" (csrc/celerite.cuh)."""
        check(self.lib.pioran_ctx_set_sweep_kernel(self.h, {"auto": 0, "scalar": 1}[which]))

    # -- K3
    def set_auto_scan(self, enabled=True):
        """Whether celerite_logl / approx_logl route ≤ 4 evaluations of a series of ≥ 4 096 steps to the scan path."""
        check(self.lib.pioran_ctx_set_auto_scan(self.h, int(bool(enabled))))

    def set_scan_chunks(self, chunks):
        """Chunks of the time axis per parameter vector in celerite_logl_scan (0 = automatic)."""
        check(self.lib.pioran_ctx_set_scan_chunks(self.h, int(chunks)))

    def set_scan_tolerance(self, tol):
        """Self-check of the scan path: parameter vectors whose deviation estimate exceeds tol·max(1, |log L|) are refined by
        Newton steps on the chunk states, then (if that fails) evaluated by the sequential sweep (default 1e-10; ≤ 0: never)."""
        check(self.lib.pioran_ctx_set_scan_tolerance(self.h, float(tol)))

    def last_scan_check(self):
        """ScanCheck(estimate, fallback, refined) of the last scan call: largest relative deviation estimate among its results,
        parameter vectors sent to the sequential sweep, parameter vectors accepted after a refinement pass."""
        est, nfb, nrf = C.c_double(0.0), C.c_int(0), C.c_int(0)
        check(self.lib.pioran_ctx_last_scan_check(self.h, C.byref(est), C.byref(nfb), C.byref(nrf)))
        return ScanCheck(est.value, nfb.value, nrf.value)

    def set_scan_floor_cap(self, cap):
        """Largest stalled estimate of a converged Newton iteration accepted as the rounding floor (default 1e-7; ≤ 0: never)."""
        check(self.lib.pioran_ctx_set_scan_floor_cap(self.h, float(cap)))

    def last_scan_history(self, index=0, max_passes=8):
        """(estimates, values) of parameter vector `index` of the last scan call after every pass it went through."""
        est, val, n = np.zeros(max_passes), np.zeros(max_passes), C.c_int(0)
        check(self.lib.pioran_ctx_last_scan_history(self.h, int(index), int(max_passes), _p(est), _p(val), C.byref(n)))
        k = min(n.value, max_passes)
        return est[:k], val[:k]

    def celerite_logl_scan(self, series, a, b, c, d, mu=None, nu=None):
        a, b, c, d = (np.atleast_2d(_f64(x)) for x in (a, b, c, d))
        B, Jt = a.shape
        mu = _f64(mu, (B,)) if mu is not None else None
        nu = _f64(nu, (B,)) if nu is not None else None
        out = np.empty(B)
        check(self.lib.pioran_celerite_logl_scan(self.h, series.id, B, Jt, _p(a), _p(b), _p(c), _p(d), _p(mu), _p(nu),
                                                 _p(out)))
        return out

    # -- K3 with the time axis split across ranks (see parallel.scan_logl_sharded)
    def scan_range_begin(self, series, a, b, c, d, n_lo, n_hi, mu=None, nu=None, max_prev=8):
        """Folds steps [n_lo, n_hi) of the series; returns the range's composite scan element (1-D array)."""
        a, b, c, d = (_f64(x).ravel() for x in (a, b, c, d))
        mu = _f64([mu]) if mu is not None else None
        nu = _f64([nu]) if nu is not None else None
        out = np.empty(self.lib.pioran_scan_composite_doubles())
        check(self.lib.pioran_celerite_scan_range_begin(self.h, series.id, a.shape[0], _p(a), _p(b), _p(c), _p(d), _p(mu), _p(nu),
                                                        int(n_lo), int(n_hi), int(max_prev), _p(out)))
        return out

    def scan_range_end(self, composites_prev):
        """composites_prev: [nprev × composite] of the ranges before this one, in time order → (Σ log|D|, Σ z²/D)."""
        prev = _f64(composites_prev) if composites_prev is not None and len(composites_prev) else None
        nprev = 0 if prev is None else int(np.atleast_2d(prev).shape[0])
        out = np.empty(2)
        check(self.lib.pioran_celerite_scan_range_end(self.h, nprev, _p(prev), _p(out)))
        return out

    def scan_range_check(self):
        """Self-check data of the range scan_range_end just finished (include/pioran_b200.h: pioran_celerite_scan_range_check)."""
        out = np.empty(8)
        check(self.lib.pioran_celerite_scan_range_check(self.h, _p(out)))
        return out

    # -- K4
    def direct_logl(self, series, a, b, c, d, mu=None, nu=None):
        """Batched log_likelihood_direct (src/direct_solver.jl:6-21): returns (+NLL [B], info [B])."""
        a, b, c, d = (np.atleast_2d(_f64(x)) for x in (a, b, c, d))
        B, Jt = a.shape
        mu = _f64(mu, (B,)) if mu is not None else None
        nu = _f64(nu, (B,)) if nu is not None else None
        out = np.empty(B)
        info = np.zeros(B, dtype=np.int32)
        check(self.lib.pioran_direct_logl(self.h, series.id, B, Jt, _p(a), _p(b), _p(c), _p(d), _p(mu), _p(nu),
                                          _p(out), info.ctypes.data_as(C.POINTER(C.c_int))))
        return out, info


    # -- widening rows: posterior mean and draws
    def celerite_predict(self, series, a, b, c, d, tau, mu=None, nu=None):
        """Batched pred(a,b,c,d,τ,t,y,σ²) (src/celerite_solver.jl:376-483): posterior mean [B × M] at ascending τ."""
        a, b, c, d = (np.atleast_2d(_f64(x)) for x in (a, b, c, d))
        B, Jt = a.shape
        tau = _f64(tau)
        mu = _f64(mu, (B,)) if mu is not None else None
        nu = _f64(nu, (B,)) if nu is not None else None
        out = np.empty((B, tau.shape[0]))
        check(self.lib.pioran_celerite_predict(self.h, series.id, B, Jt, _p(a), _p(b), _p(c), _p(d), _p(mu), _p(nu),
                                               tau.shape[0], _p(tau), _p(out)))
        return out

    def celerite_predict_var(self, series, a, b, c, d, tau, mu=None, nu=None, return_mean=True):
        """Posterior predictive variance of the latent f at ascending τ (the diagonal of predict_cov,
        src/direct_solver.jl:28-119), [B × M], by the O((N + M)·R²) sweep K6.  With return_mean, (mean, var), where mean is
        celerite_predict's result bit for bit.  A set whose covariance is not positive definite gets a NaN row."""
        a, b, c, d = (np.atleast_2d(_f64(x)) for x in (a, b, c, d))
        B, Jt = a.shape
        tau = _f64(tau)
        mu = _f64(mu, (B,)) if mu is not None else None
        nu = _f64(nu, (B,)) if nu is not None else None
        var = np.empty((B, tau.shape[0]))
        mean = np.empty((B, tau.shape[0])) if return_mean else None
        check(self.lib.pioran_celerite_predict_var(self.h, series.id, B, Jt, _p(a), _p(b), _p(c), _p(d), _p(mu), _p(nu),
                                                   tau.shape[0], _p(tau), _p(mean), _p(var)))
        return (mean, var) if return_mean else var

    def celerite_simulate(self, series, a, b, c, d, q, nu=None):
        """Batched sim(rng,a,b,c,d,t,σ²) (src/celerite_solver.jl:515-549) with the normal draws q [B × N] supplied."""
        a, b, c, d = (np.atleast_2d(_f64(x)) for x in (a, b, c, d))
        B, Jt = a.shape
        q = _f64(q, (B, series.N))
        nu = _f64(nu, (B,)) if nu is not None else None
        out = np.empty((B, series.N))
        check(self.lib.pioran_celerite_simulate(self.h, series.id, B, Jt, _p(a), _p(b), _p(c), _p(d), _p(nu), _p(q),
                                                _p(out)))
        return out


_default = {}


def get_context(device=None):
    """Process-wide context per device (created on first use)."""
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0"))
    if device not in _default:
        _default[device] = Context(device)
    return _default[device]
