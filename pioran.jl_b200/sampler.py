"""Vectorised sampler bridge (SURVEY §8f #4): the two callbacks a nested sampler needs, over whole batches of points.

The reference runs ultranest with `vectorized = false` (examples/ultranest/single_pl.jl:118): one `prior_transform(cube)` and
one `logl(pars)` per point.  With the GPU backend the natural mode is `vectorized = True`: ultranest hands over all proposed
points of an iteration at once — `transform(cubes [B × P]) → Θ [B × P]`, `loglike(Θ [B × P]) → logL [B]` — and ONE fused call
evaluates them (0.6–0.8 ms for 400 live points at N = 1 000, J = 20).

The prior transform runs on the host by default: it is P scalar quantiles per point (≈ 40 µs for 400 × 6 with numpy/scipy),
an order of magnitude under the call's own launch + copy overhead.  `PriorTransform.device_spec()` describes the same columns
for the device-side transform (`pioran_prior_transform`, `pioran_prior_transform_logl`: cube in, logℒ out, θ never leaves the
GPU) — `vectorized_callbacks(..., device_prior=True)`.  Quantiles follow Distributions.jl's definitions (`quantile(d, u)`),
which the reference calls.
"""
import numpy as np


class Uniform:
    def __init__(self, a, b):
        self.a, self.b = a, b

    def quantile(self, u, prev):
        return self.a + u * (self.b - self.a)

    def device(self):
        return (0, 0, self.a, self.b)


class UniformFrom:
    """Uniform(θ[col], b): the lower edge is an earlier column of the same point (α₂ ~ U(α₁, 4), single_pl.jl:99)."""

    def __init__(self, col, b):
        self.col, self.b = col, b

    def quantile(self, u, prev):
        lo = prev[:, self.col]
        return lo + u * (self.b - lo)

    def device(self):
        return (1, self.col, 0.0, self.b)


class LogUniform:
    def __init__(self, a, b):
        self.la, self.lb = np.log(a), np.log(b)

    def quantile(self, u, prev):
        return np.exp(self.la + u * (self.lb - self.la))

    def device(self):
        return (2, 0, float(np.exp(self.la)), float(np.exp(self.lb)))


class Normal:
    def __init__(self, mu, sigma):
        self.mu, self.sigma = mu, sigma

    def quantile(self, u, prev):
        from scipy.special import ndtri
        return self.mu + self.sigma * ndtri(u)

    def device(self):
        return (3, 0, self.mu, self.sigma)


class LogNormal(Normal):
    def quantile(self, u, prev):
        return np.exp(super().quantile(u, prev))

    def device(self):
        return (4, 0, self.mu, self.sigma)


class Gamma:
    """Gamma(shape k, scale θ) — Distributions.jl's parametrisation (single_pl.jl:101: Gamma(2, 0.5))."""

    def __init__(self, k, theta):
        self.k, self.theta = k, theta

    def quantile(self, u, prev):
        from scipy.special import gammaincinv
        return self.theta * gammaincinv(self.k, u)

    def device(self):
        return (5, 0, self.k, self.theta)


class PriorTransform:
    """Column-wise prior transform of unit-cube points; columns are evaluated left to right, so a prior may depend on earlier
    columns of the same point (UniformFrom)."""

    def __init__(self, priors):
        self.priors = list(priors)

    def __call__(self, cubes):
        cubes = np.asarray(cubes, dtype=np.float64)
        single = cubes.ndim == 1
        u = np.atleast_2d(cubes)
        out = np.empty_like(u)
        for k, p in enumerate(self.priors):
            out[:, k] = p.quantile(u[:, k], out)
        return out[0] if single else out

    def device_spec(self):
        """(kind, ref_col, p0, p1) per column — struct pioran_prior_spec of include/pioran_b200.h."""
        return [p.device() for p in self.priors]


def single_bending_power_law_prior(f_min, f_max, xbar, va, mu_v=-1.5, sigma_v=1.0, alpha2_max=4.0, log_data=False):
    """The prior of examples/ultranest/single_pl.jl:49-56,96-104 for Θ = (α₁, f₁, α₂, variance, ν, μ)."""
    f0, fM = f_min / 20.0, f_max * 20.0
    mu_n, sigma_n = 2 * mu_v, np.sqrt(2 * sigma_v ** 2)
    return PriorTransform([Uniform(0.0, 1.5), LogUniform(f0 * 4.0, fM / 4.0), UniformFrom(0, alpha2_max),
                           LogNormal(mu_n, sigma_n), Gamma(2, 0.5), Normal(xbar, 5 * np.sqrt(va))])


def log_normal_prior(f_min, f_max, y, mu_v=-1.5, sigma_v=1.0, alpha1_max=1.25, alpha2_max=4.0):
    """The prior of docs/src/ultranest.md:165-190,220-229 for Θ = (α₁, f₁, α₂, variance, ν, μ, c) — the log-normal model with
    an offset c ~ LogUniform(1e-6, 0.99·min y); x̄ and va are the mean and variance of log(y), f₁ ~ LogUniform(f0·4, fM/4)."""
    y = np.asarray(y, dtype=np.float64)
    f0, fM = f_min / 20.0, f_max * 20.0
    mu_n, sigma_n = 2 * mu_v, np.sqrt(2 * sigma_v ** 2)
    xbar, va = float(np.mean(np.log(y))), float(np.var(np.log(y), ddof=1))
    return PriorTransform([Uniform(0.0, alpha1_max), LogUniform(f0 * 4.0, fM / 4.0), UniformFrom(0, alpha2_max),
                           LogNormal(mu_n, sigma_n), Gamma(2, 0.5), Normal(xbar, 5 * np.sqrt(va)),
                           LogUniform(1e-6, float(np.min(y)) * 0.99)])


def vectorized_callbacks_log_normal(t, y, yerr, psd_model="SingleBendingPowerLaw", n_components=20, basis_function="SHO",
                                    prior=None, ctx=None, **approx_kw):
    """Same as vectorized_callbacks for the seven-parameter log-normal likelihood of docs/src/ultranest.md:197-217: the offset c
    is sampled, so the transform yn = log(y − c), σ² = ν σ²/(y − c)² is per point and runs on the device
    (pioran_approx_logl_logshift)."""
    from .api import BatchedLikelihood
    t, y, yerr = (np.asarray(x, dtype=np.float64) for x in (t, y, yerr))
    like = BatchedLikelihood(t, y, yerr ** 2, psd_model, n_components, basis_function, ctx=ctx, log_shift=True, **approx_kw)
    if prior is None:
        f_min, f_max = 1.0 / (t[-1] - t[0]), 1.0 / np.min(np.diff(t)) / 2.0
        prior = log_normal_prior(f_min, f_max, y, alpha2_max=4.0 if basis_function == "SHO" else 6.0)

    def loglike(theta):
        out = like(np.atleast_2d(theta))
        out[~np.isfinite(out)] = -1e300
        return out

    return loglike, prior, like.close


def vectorized_callbacks(t, y, yerr, psd_model="SingleBendingPowerLaw", n_components=20, basis_function="SHO",
                         log_transform=True, prior=None, ctx=None, device_prior=False, periodic_mean=False, **approx_kw):
    """(loglike, transform, close) for `ultranest.ReactiveNestedSampler(paramnames, loglike, transform=transform,
    vectorized=True)`.  log_transform follows single_pl.jl:70-73 (σ² = ν σ²/y², yn = log y); the series is uploaded once.
    periodic_mean: Θ rows end with (A, ϕ, T₀) and the mean is μ + A·sin(2πt/T₀ + ϕ) (single_pl_periodicity.jl, which
    samples with log_transform=False); its prior must be given, as the reference run's priors of A, ϕ and T₀ are not known here."""
    from .api import BatchedLikelihood
    if periodic_mean and prior is None:
        raise ValueError("periodic_mean=True needs an explicit prior (transform over psd parameters…, variance, ν, μ, A, ϕ, T₀)")
    if periodic_mean and device_prior:
        raise ValueError("the fused prior-transform entry takes no periodic mean; use device_prior=False")
    t, y, yerr = (np.asarray(x, dtype=np.float64) for x in (t, y, yerr))
    if log_transform:
        yn, s2 = np.log(y), yerr ** 2 / y ** 2
    else:
        yn, s2 = y, yerr ** 2
    like = BatchedLikelihood(t, yn, s2, psd_model, n_components, basis_function, ctx=ctx, periodic_mean=periodic_mean, **approx_kw)
    if prior is None:
        f_min, f_max = 1.0 / (t[-1] - t[0]), 1.0 / np.min(np.diff(t)) / 2.0
        prior = single_bending_power_law_prior(f_min, f_max, float(np.mean(yn)), float(np.var(yn, ddof=1)),
                                               alpha2_max=4.0 if basis_function == "SHO" else 6.0)

    def loglike(theta):
        out = like(np.atleast_2d(theta))
        out[~np.isfinite(out)] = -1e300        # ultranest needs finite values; the reference's scripts never hit non-PD priors
        return out

    if device_prior:
        # the transform callback on the device (same columns, pioran_prior_transform); loglike_from_cube fuses both callbacks
        spec = prior.device_spec()

        def transform(cubes):
            cubes = np.asarray(cubes, dtype=np.float64)
            out = like.ctx.prior_transform(spec, np.atleast_2d(cubes))
            return out[0] if cubes.ndim == 1 else out

        def loglike_from_cube(cubes):
            out = like.ctx.prior_transform_logl(like.series, like.spec, spec, np.atleast_2d(cubes))
            out[~np.isfinite(out)] = -1e300
            return out

        loglike.from_cube = loglike_from_cube
        return loglike, transform, like.close
    return loglike, prior, like.close
