"""Host-side mirror of the Pioran.jl interface for the likelihood path — same names, argument meaning and error
behaviour as the reference, with the arithmetic done by libpioran_b200's CUDA kernels.

    𝓟  = SingleBendingPowerLaw(α₁, f₁, α₂)
    𝓡  = approx(𝓟, f_min, f_max, 20, variance, basis_function="SHO")     # src/psd.jl:214
    f  = ScalableGP(μ, 𝓡)                                                 # src/scalable_GP.jl:36
    ℓ  = logpdf(f(t, σ²), y)                                              # src/scalable_GP.jl:162-166

Batched entry for samplers that evaluate many parameter vectors at once (ultranest `vectorized=True`):
    like = BatchedLikelihood(t, y, σ², psd_model="SingleBendingPowerLaw", n_components=20, basis_function="SHO")
    ℓ    = like(Θ)        # Θ rows = [psd parameters…, variance, ν, μ]  (examples/ultranest/single_pl.jl:67)
"""
import collections

import numpy as np

from . import backend
from .backend import get_context, make_spec


# ----------------------------------------------------------------------------------------------- PSD models
class PowerSpectralDensity:
    """Tonari.jl's abstract type (src/Pioran.jl:15,20)."""
    model_name = None

    def params(self):
        raise NotImplementedError


class SingleBendingPowerLaw(PowerSpectralDensity):
    """𝓟(f) = (f/f₁)^(−α₁) / (1 + (f/f₁)^(α₂−α₁))   (test/test_psd.jl:6)"""
    model_name = "SingleBendingPowerLaw"

    def __init__(self, α1, f1, α2):
        self.α1, self.f1, self.α2 = float(α1), float(f1), float(α2)

    def params(self):
        return [self.α1, self.f1, self.α2]


class DoubleBendingPowerLaw(PowerSpectralDensity):
    """𝓟(f) = (f/f₁)^(−α₁) / (1 + (f/f₁)^(α₂−α₁)) / (1 + (f/f₂)^(α₃−α₂))   (test/test_psd.jl:12)"""
    model_name = "DoubleBendingPowerLaw"

    def __init__(self, α1, f1, α2, f2, α3):
        self.α1, self.f1, self.α2, self.f2, self.α3 = map(float, (α1, f1, α2, f2, α3))

    def params(self):
        return [self.α1, self.f1, self.α2, self.f2, self.α3]


class QPO(PowerSpectralDensity):
    """QPO(S₀, f₀, Q): Tonari.jl's Lorentzian feature (fields read by convert_feature, src/psd.jl:15-28; docs/src/adding_features.md)."""
    model_name = "QPO"

    def __init__(self, S0, f0, Q):
        self.S0, self.f0, self.Q = float(S0), float(f0), float(Q)

    def params(self):
        return [self.S0, self.f0, self.Q]


class SumOfPowerSpectralDensity(PowerSpectralDensity):
    """𝓟₁ + 𝓟₂ + … (Tonari.jl): approx() splits it into ONE continuum and the narrow features (separate_psd, src/psd.jl:221)."""
    model_name = "Sum"

    def __init__(self, components):
        self.components = list(components)

    def params(self):
        return [v for comp in self.components for v in comp.params()]


def _psd_add(self, other):
    if not isinstance(other, PowerSpectralDensity):
        return NotImplemented
    left = self.components if isinstance(self, SumOfPowerSpectralDensity) else [self]
    right = other.components if isinstance(other, SumOfPowerSpectralDensity) else [other]
    return SumOfPowerSpectralDensity(left + right)


PowerSpectralDensity.__add__ = _psd_add


def separate_psd(psd_model):
    """(continuum, features) of a PSD model — features is None, or a list of QPO (src/psd.jl:221 uses Tonari's separate_psd)."""
    comps = psd_model.components if isinstance(psd_model, SumOfPowerSpectralDensity) else [psd_model]
    cont = [comp for comp in comps if not isinstance(comp, QPO)]
    feats = [comp for comp in comps if isinstance(comp, QPO)]
    if len(cont) > 1:
        raise ValueError("only one continuum component can be approximated")
    return (cont[0] if cont else None), (feats or None)


def convert_feature(psd_feature):
    """[a, b, c, d] of a PSD feature (src/psd.jl:15-28); only QPO is implemented, like the reference."""
    if not isinstance(psd_feature, QPO):
        raise ValueError(f"Feature {type(psd_feature).__name__} not implemented")
    Δ = np.sqrt(4.0 * psd_feature.Q ** 2 - 1.0)
    ω0 = 2.0 * np.pi * psd_feature.f0
    a = psd_feature.S0 * ω0 * psd_feature.Q / 4.0
    c = ω0 / psd_feature.Q / 2.0
    return np.array([a, a / Δ, c, c * Δ])


def get_covariance_from_psd(psd_features):
    """4 × n matrix of the features' celerite coefficients (src/psd.jl:35-44)."""
    feats = psd_features if isinstance(psd_features, (list, tuple)) else [psd_features]
    return np.column_stack([convert_feature(f) for f in feats])


# ----------------------------------------------------------------------------------------------- ACVF types
class SemiSeparable:
    """src/acvf.jl: abstract semi-separable covariance."""


class Celerite(SemiSeparable):
    """Celerite(a, b, c, d): k(τ) = exp(−cτ)(a cos dτ + b sin dτ)   (src/Celerite.jl:20-44)"""

    def __init__(self, a, b, c, d):
        self.a, self.b, self.c, self.d = float(a), float(b), float(c), float(d)


class SHO(Celerite):
    """SHO(A, ω₀, Q=1/√2)  → (A, A, ω₀/√2, ω₀/√2)   (src/SHO.jl)"""

    def __init__(self, A, ω0):
        super().__init__(A, A, ω0 / np.sqrt(2.0), ω0 / np.sqrt(2.0))


class Exp(Celerite):
    """Exp(A, α): k(τ) = A/2·exp(−ατ) → (A/2, 0, α, 0)   (src/Exp.jl:22-34; test/test_covariancefunctions.jl:44-47)"""

    def __init__(self, A, α):
        super().__init__(A / 2.0, 0.0, α, 0.0)


class SumOfCelerite(SemiSeparable):
    """Container of the coefficient vectors (src/acvf.jl:35-53).  `+` of terms concatenates."""

    def __init__(self, a, b, c, d, _fused=None):
        self.a, self.b, self.c, self.d = (np.asarray(x, dtype=np.float64).ravel().copy() for x in (a, b, c, d))
        if not (self.a.shape == self.b.shape == self.c.shape == self.d.shape):
            raise ValueError("a, b, c, d must have the same length")
        self._fused = _fused  # (spec, psd parameters, norm) when produced by approx(): enables the fused kernel

    def __call__(self, t1, t2):
        """Kernel value (src/acvf.jl:138-140); host arithmetic on J numbers, used by tests like `𝓡(0,0) ≈ va`."""
        τ = abs(t1 - t2)
        return float(np.sum(np.exp(-self.c * τ) * (self.a * np.cos(self.d * τ) + self.b * np.sin(self.d * τ))))

    def __add__(self, other):
        o = celerite_coefs(other)
        return SumOfCelerite(*(np.concatenate([x, y]) for x, y in zip(celerite_coefs(self), o)))


# ----------------------------------------------------------------------------------------------- CARMA front end
# SURVEY §8f #4: covariances whose decay rates and frequencies depend on the sampled parameters reach the GPU through the
# generic coefficient entry.  CARMA (src/CARMA.jl) is the reference's own example: host arithmetic on p roots, then (a, b, c, d).
def quad2roots(quad):
    """Roots of the product of quadratic factors x² + quad[k+1] x + quad[k] (k = 0, 2, …) and, for an odd count, the linear
    factor x + quad[-1]  (src/CARMA.jl:201-223; test/test_carma.jl:3-17)."""
    quad = np.asarray(quad, dtype=np.float64)
    n = quad.shape[0]
    r = np.zeros(n, dtype=np.complex128)
    if n % 2 == 1:
        r[-1] = -quad[-1]
    for k in range(0, n - n % 2, 2):
        lin, const = quad[k + 1], quad[k]
        disc = lin * lin - 4.0 * const
        if disc < 0:
            r[k] = (-lin + 1j * np.sqrt(-disc)) / 2.0
            r[k + 1] = np.conj(r[k])
        else:
            r[k], r[k + 1] = (-lin + np.sqrt(disc)) / 2.0, (-lin - np.sqrt(disc)) / 2.0
    return r


def roots2coeffs(r):
    """Coefficients, constant term first, of the monic polynomial with roots r (src/CARMA.jl:185-188)."""
    return np.poly(np.asarray(r, dtype=np.complex128))[::-1]


def _carma_residue(rk, roots, beta):
    """β(r_k) β(−r_k) / (−2 Re r_k ∏_{j: r_j ≠ r_k} (r_j − r_k)(conj r_j + r_k)): the weight of exp(r_k |τ|) in the CARMA
    autocovariance (src/CARMA.jl:230-247)."""
    powers = np.arange(beta.shape[0])
    num = np.sum(beta * rk ** powers) * np.sum(beta * (-rk) ** powers)
    den = -2.0 * rk.real
    for rj in roots:
        if rj != rk:
            den = den * ((rj - rk) * (np.conj(rj) + rk))
    return num / den


class CARMA(SemiSeparable):
    """CARMA(p, q, rα, β, norm=1, is_integrated_power=True)  (src/CARMA.jl:1-43): rα the p roots of the autoregressive polynomial
    (conjugate pairs next to each other, a real root last when p is odd), β the q + 1 moving-average coefficients."""

    def __init__(self, p, q, rα, β, norm=1.0, is_integrated_power=True):
        p, q = int(p), int(q)
        rα = np.asarray(rα, dtype=np.complex128).ravel()
        β = np.asarray(β, dtype=np.float64).ravel()
        if p < 1 or q < 0:
            raise ValueError("The order of the autoregressive and moving average polynomials must be positive")
        if q > p:
            raise ValueError("The order of the moving average polynomial must be less than or equal to the order of the "
                             "autoregressive polynomial")
        if rα.shape[0] != p:
            raise ValueError("The length of the roots of the autoregressive polynomial must be equal to the order of the "
                             "autoregressive polynomial")
        if β.shape[0] != q + 1:
            raise ValueError("The length of the moving average coefficients must be equal to q + 1")
        self.p, self.q, self.rα, self.β = p, q, rα, β
        self.norm, self.is_integrated_power = float(norm), bool(is_integrated_power)

    def covariance(self, τ):
        """CARMA_covariance(τ, cov) (src/CARMA.jl:230-275): Σ_k residue_k exp(r_k |τ|), normalised like celerite_coefs."""
        τ = np.abs(np.asarray(τ, dtype=np.float64))
        res = np.array([_carma_residue(rk, self.rα, self.β) for rk in self.rα])
        acv = np.real(np.sum(res[:, None] * np.exp(self.rα[:, None] * τ.ravel()[None, :]), axis=0)).reshape(τ.shape)
        # src/CARMA.jl:269-273: Cov = Re(R)·norm, divided by 2·Re(variance) when integrated, and 2·Cov is returned
        scale = self.norm / np.real(np.sum(res)) if self.is_integrated_power else 2.0 * self.norm
        return acv * scale


def carma_celerite_coefs(p, rα, β, norm=1.0, is_integrated_power=True):
    """CARMA_celerite_coefs (src/CARMA.jl:98-143): one celerite term per conjugate pair (a + i b = 2 × the pair's residue,
    c = −Re r, d = −Im r) and a real term (b = d = 0) for the unpaired last root of an odd p; with is_integrated_power the
    amplitudes are rescaled so that Σa = norm.  Pinned by test/test_carma.jl:53-70."""
    rα = np.asarray(rα, dtype=np.complex128).ravel()
    β = np.asarray(β, dtype=np.float64).ravel()
    J = (p + 1) // 2
    a, b, c, d = (np.empty(J) for _ in range(4))
    for k in range(J):
        rk = rα[2 * k]
        frac = 2.0 * _carma_residue(rk, rα, β)        # −β(r)β(−r)/Re r / ∏ …
        if k != J - 1 or p % 2 == 0:
            a[k], b[k], c[k], d[k] = 2.0 * frac.real, 2.0 * frac.imag, -rk.real, -rk.imag
        else:
            a[k], b[k], c[k], d[k] = frac.real, 0.0, -rk.real, 0.0
    scale = norm / np.sum(a) if is_integrated_power else norm
    return a * scale, b * scale, c, d


def carma_celerite_coefs_jacobian(p, q, qa, qb, variance):
    """carma_celerite_coefs ∘ (quad2roots, roots2coeffs) for one Θ row of BatchedCARMALikelihood (is_integrated_power) and its
    Jacobian, in forward mode on complex numbers along the p + q + 1 unit directions of (qa…, qb…, variance).
    Returns ((a, b, c, d) [J] each, (∂a, ∂b, ∂c, ∂d) [J × (p + q + 1)] each)."""
    qa, qb = np.asarray(qa, dtype=np.float64), np.asarray(qb, dtype=np.float64)
    P = p + q + 1
    eye = np.eye(P)

    def roots(quad, off):   # quad2roots with tangents [n × P]
        n = quad.shape[0]
        r, dr = np.zeros(n, dtype=np.complex128), np.zeros((n, P), dtype=np.complex128)
        dq = eye[off:off + n]
        if n % 2 == 1:
            r[-1], dr[-1] = -quad[-1], -dq[-1]
        for k in range(0, n - n % 2, 2):
            lin, const, dlin, dconst = quad[k + 1], quad[k], dq[k + 1], dq[k]
            disc, ddisc = lin * lin - 4.0 * const, 2.0 * lin * dlin - 4.0 * dconst
            if disc < 0:
                sq = np.sqrt(-disc)
                r[k], dr[k] = (-lin + 1j * sq) / 2.0, (-dlin - 1j * ddisc / (2.0 * sq)) / 2.0
                r[k + 1], dr[k + 1] = np.conj(r[k]), np.conj(dr[k])
            else:
                sq = np.sqrt(disc)
                dsq = ddisc / (2.0 * sq)
                r[k], dr[k] = (-lin + sq) / 2.0, (-dlin + dsq) / 2.0
                r[k + 1], dr[k + 1] = (-lin - sq) / 2.0, (-dlin - dsq) / 2.0
        return r, dr

    rα, drα = roots(qa, 0)
    if q > 0:
        rβ, drβ = roots(qb, p)
        co, dco = np.ones(1, dtype=np.complex128), np.zeros((1, P), dtype=np.complex128)   # constant term first
        for rj, drj in zip(rβ, drβ):
            nco, ndco = np.zeros(co.shape[0] + 1, dtype=np.complex128), np.zeros((co.shape[0] + 1, P), dtype=np.complex128)
            nco[1:], ndco[1:] = co, dco
            nco[:-1] -= rj * co
            ndco[:-1] -= rj * dco + co[:, None] * drj[None, :]
            co, dco = nco, ndco
        β, dβ = co.real, dco.real
    else:
        β, dβ = np.ones(1), np.zeros((1, P))
    J = (p + 1) // 2
    a, b, c, d = (np.empty(J) for _ in range(4))
    da, db, dc, dd = (np.zeros((J, P)) for _ in range(4))
    pw = np.arange(β.shape[0])
    for k in range(J):
        rk, drk = rα[2 * k], drα[2 * k]
        # the residue of _carma_residue and its tangent
        A = np.sum(β * rk ** pw)
        dA = dβ.T @ (rk ** pw) + np.sum(β[1:] * pw[1:] * rk ** (pw[1:] - 1)) * drk
        Bv = np.sum(β * (-rk) ** pw)
        dB = dβ.T @ ((-rk) ** pw) - np.sum(β[1:] * pw[1:] * (-rk) ** (pw[1:] - 1)) * drk
        den, dden = -2.0 * rk.real + 0j, -2.0 * drk.real + 0j
        for rj, drj in zip(rα, drα):
            if rj != rk:
                f = (rj - rk) * (np.conj(rj) + rk)
                df = (drj - drk) * (np.conj(rj) + rk) + (rj - rk) * (np.conj(drj) + drk)
                den, dden = den * f, dden * f + den * df
        num, dnum = A * Bv, dA * Bv + A * dB
        frac, dfrac = 2.0 * num / den, 2.0 * (dnum * den - num * dden) / den ** 2
        if k != J - 1 or p % 2 == 0:
            a[k], b[k], c[k], d[k] = 2.0 * frac.real, 2.0 * frac.imag, -rk.real, -rk.imag
            da[k], db[k], dc[k], dd[k] = 2.0 * dfrac.real, 2.0 * dfrac.imag, -drk.real, -drk.imag
        else:
            a[k], b[k], c[k], d[k] = frac.real, 0.0, -rk.real, 0.0
            da[k], dc[k] = dfrac.real, -drk.real
    sa, dsa = np.sum(a), np.sum(da, axis=0)
    dvar = eye[p + q]
    scale, dscale = variance / sa, dvar / sa - variance * dsa / sa ** 2
    return ((a * scale, b * scale, c, d),
            (da * scale + a[:, None] * dscale[None, :], db * scale + b[:, None] * dscale[None, :], dc, dd))


def celerite_repr(cov):
    """celerite_repr(cov::CARMA) (src/CARMA.jl:55-70) → SumOfCelerite."""
    return SumOfCelerite(*celerite_coefs(cov))


def celerite_coefs(cov):
    """(a, b, c, d) vectors of a covariance (src/acvf.jl:119-127, src/Celerite.jl:33-39, src/CARMA.jl:73-75)."""
    if isinstance(cov, SumOfCelerite):
        return cov.a, cov.b, cov.c, cov.d
    if isinstance(cov, CARMA):
        return carma_celerite_coefs(cov.p, cov.rα, cov.β, cov.norm, cov.is_integrated_power)
    if isinstance(cov, Celerite):
        return (np.array([cov.a]), np.array([cov.b]), np.array([cov.c]), np.array([cov.d]))
    raise TypeError(f"no celerite coefficients for {type(cov).__name__}")


# ----------------------------------------------------------------------------------------------- approx
def approx(psd_model, f_min, f_max, n_components=20, norm=1.0, S_low=20.0, S_high=20.0, *, is_integrated_power=True,
           basis_function="SHO", ctx=None):
    """approx(psd_model, f_min, f_max, n_components, norm, S_low, S_high; is_integrated_power, basis_function)
    (src/psd.jl:214-289) → SumOfCelerite.  Runs the K1 kernel."""
    if not isinstance(psd_model, PowerSpectralDensity):
        raise TypeError("psd_model must be a PowerSpectralDensity")
    ctx = ctx or get_context()
    continuum, features = separate_psd(psd_model)
    if continuum is None:      # src/psd.jl:223
        raise ValueError("The PSD model should contain at least one ContinuumPowerSpectrum component to be approximated")
    if features is not None:
        # continuum + QPO features (src/psd.jl:229-243, 254-259, 277-282): K1 appends one celerite term per feature
        spec = make_spec(continuum.model_name, f_min, f_max, n_components, S_low, S_high, is_integrated_power, basis_function)
        theta = np.array([continuum.params() + [float(norm)] + [v for f in features for v in f.params()]])
        a, b, c, d = ctx.approx_coeffs_features(spec, len(features), theta)
        return SumOfCelerite(a[0], b[0], c[0], d[0])
    psd_model = continuum
    spec = make_spec(psd_model.model_name, f_min, f_max, n_components, S_low, S_high, is_integrated_power, basis_function)
    theta = np.array([psd_model.params() + [float(norm)]])
    a, b, c, d = ctx.approx_coeffs(spec, theta)
    return SumOfCelerite(a[0], b[0], c[0], d[0], _fused=(spec, psd_model.params(), float(norm)))


# ----------------------------------------------------------------------------------------------- GP API
class CustomMean:
    """AbstractGPs.CustomMean: a callable evaluated on the time vector (test/test_mean.jl)."""

    def __init__(self, f):
        self.f = f

    def __call__(self, t):
        return np.asarray(self.f(np.asarray(t, dtype=np.float64)), dtype=np.float64)


_SOLVERS = ("celerite", "celerite_gpu", "direct")


class ScalableGP:
    """ScalableGP(μ, 𝓡[, solver])  (src/scalable_GP.jl:24-40).  μ: number or CustomMean."""

    def __init__(self, *args, solver="celerite"):
        if len(args) == 1:
            mean, kernel = 0.0, args[0]
        elif len(args) == 2:
            mean, kernel = args
        elif len(args) == 3:
            mean, kernel, solver = args
        else:
            raise TypeError("ScalableGP(kernel) | ScalableGP(μ, kernel) | ScalableGP(μ, kernel, solver)")
        if not isinstance(kernel, SemiSeparable):
            raise TypeError("kernel must be a SemiSeparable covariance")
        self.mean, self.kernel, self.solver = mean, kernel, str(solver).lstrip(":")

    def __call__(self, t, σ2):
        """f(t, σ²) → finite-dimensional projection (AbstractGPs.FiniteGP with Diagonal(σ²))."""
        t = np.asarray(t, dtype=np.float64)
        σ2 = np.broadcast_to(np.asarray(σ2, dtype=np.float64), t.shape).copy()
        return FiniteScalableGP(self, t, σ2)


class FiniteScalableGP:
    def __init__(self, f, x, σ2):
        self.f, self.x, self.σ2 = f, x, σ2

    def mean_vector(self):
        m = self.f.mean
        return m(self.x) if callable(m) else np.full(self.x.shape, float(m))


def log_likelihood(cov, τ, y, σ2, *, solver="celerite", ctx=None):
    """log_likelihood(cov, τ, y, σ2; solver)  (src/celerite_solver.jl:262-294).
    `celerite`, `celerite_matrix` (the reference's second solver name, :266-270) and `celerite_gpu` all run the B200 kernel
    (there is no CPU path in this package)."""
    solver = str(solver).lstrip(":")
    if solver not in ("celerite", "celerite_matrix", "celerite_gpu"):
        raise ValueError(f"solver {solver} not recognised, use either :celerite or :celerite_matrix")
    ctx = ctx or get_context()
    a, b, c, d = celerite_coefs(cov)
    τ = np.ascontiguousarray(τ, dtype=np.float64)
    if τ.shape[0] >= _RESIDENT_MAX_N:
        # long series: (t, y, σ²) go up together so that the library may route the call to its parallel-in-time path
        ser = ctx.upload_series(τ, y, σ2)
        try:
            return float(ctx.celerite_logl(ser, a, b, c, d)[0])
        finally:
            ser.free()
    ser = _resident_series(ctx, τ)
    y = np.ascontiguousarray(y, dtype=np.float64).reshape(1, -1)
    σ2 = np.ascontiguousarray(σ2, dtype=np.float64).reshape(1, -1)
    return float(ctx.celerite_logl(ser, a, b, c, d, y_batch=y, s2_batch=σ2)[0])


# The time vector of a `:celerite_gpu` call stays on the device between calls (julia/b200_solver.jl: b200_resident_series): a
# sampler passes the same t ~1e5 times while Y − mean and ν·σ² are fresh arrays, which travel with the call (16 N bytes).
_RESIDENT_MAX_N = 2048
_RESIDENT_CAP = 8
_resident = collections.OrderedDict()


def _resident_series(ctx, τ):
    key = (id(ctx), τ.shape[0], float(τ[0]), float(τ[-1]), float(τ.sum()))
    ser = _resident.get(key)
    if ser is not None and ser.id is not None:
        _resident.move_to_end(key)
        return ser
    ser = ctx.upload_series(τ, np.zeros_like(τ), np.ones_like(τ))
    _resident[key] = ser
    while len(_resident) > _RESIDENT_CAP:
        _, old = _resident.popitem(last=False)
        try:
            old.free()
        except Exception:
            pass
    return ser


def release_resident_series():
    """Frees the time vectors kept on the device by log_likelihood (b200_release!() of the Julia shim)."""
    while _resident:
        _, ser = _resident.popitem()
        try:
            ser.free()
        except Exception:
            pass


def log_likelihood_direct(cov, t, y, σ2, *, ctx=None):
    """log_likelihood_direct(cov, t, y, σ²)  (src/direct_solver.jl:6-21): returns +NLL; raises like the
    reference's PosDefException when the covariance is not positive definite."""
    ctx = ctx or get_context()
    a, b, c, d = celerite_coefs(cov)
    ser = ctx.upload_series(t, y, σ2)
    try:
        nll, info = ctx.direct_logl(ser, a, b, c, d)
    finally:
        ser.free()
    if info[0] != 0:
        raise np.linalg.LinAlgError(f"PosDefException: matrix is not positive definite; leading minor {int(info[0])}")
    return float(nll[0])


def logpdf(fx, Y, *, ctx=None):
    """logpdf(f(t, σ²), Y)  (src/scalable_GP.jl:162-166)."""
    if not isinstance(fx, FiniteScalableGP):
        raise TypeError("logpdf expects ScalableGP(...)(t, σ²)")
    y = np.asarray(Y, dtype=np.float64) - fx.mean_vector()
    if fx.f.solver == "direct":
        return -log_likelihood_direct(fx.f.kernel, fx.x, y, fx.σ2, ctx=ctx)
    return log_likelihood(fx.f.kernel, fx.x, y, fx.σ2, solver=fx.f.solver, ctx=ctx)


# ----------------------------------------------------------------------------------------------- posterior, draws
class PosteriorGP:
    """posterior(f(t, σ²), y)  (src/scalable_GP.jl:44-54): holds the finite GP and the data; mean(fp, τ) runs the batched
    `pred` kernel (src/celerite_solver.jl:376-483), var / std / mean_and_var(fp, τ) the posterior-variance sweep K6,
    cov / mean_and_cov(fp, τ) the posterior-covariance walk K8."""

    def __init__(self, fx, y):
        if not isinstance(fx, FiniteScalableGP):
            raise TypeError("posterior expects ScalableGP(...)(t, σ²)")
        self.f, self.y = fx, np.asarray(y, dtype=np.float64)

    def __call__(self, τ, σ2=1e-18):
        """fp(τ, σ²): the posterior at ascending τ plus independent noise of variance σ² (AbstractGPs' default 1e-18)."""
        return FinitePosteriorGP(self, np.asarray(τ, dtype=np.float64), float(σ2))


class FinitePosteriorGP:
    """fp(τ, σ²) of a posterior: what rand draws from (posterior draws K7)."""

    def __init__(self, fp, τ, σ2):
        self.fp, self.x, self.σ2 = fp, τ, σ2


def posterior(fx, y):
    return PosteriorGP(fx, y)


def predict(cov, τ, t, y, σ2, *, ctx=None):
    """predict(cov, τ, t, y, σ²)  (src/celerite_solver.jl:348-374): posterior mean of the zero-mean GP at ascending τ."""
    ctx = ctx or get_context()
    a, b, c, d = celerite_coefs(cov)
    ser = ctx.upload_series(t, y, σ2)
    try:
        return ctx.celerite_predict(ser, a, b, c, d, τ)[0]
    finally:
        ser.free()


def mean(fp, τ=None, *, ctx=None):
    """mean(fp[, τ])  (src/scalable_GP.jl:61-67, 84-85): predict on y − m(t), plus m(τ)."""
    if not isinstance(fp, PosteriorGP):
        raise TypeError("mean expects posterior(f(t, σ²), y)")
    fx = fp.f
    τ = fx.x if τ is None else np.asarray(τ, dtype=np.float64)
    m = fx.f.mean
    mτ = m(τ) if callable(m) else np.full(τ.shape, float(m))
    return predict(fx.f.kernel, τ, fx.x, fp.y - fx.mean_vector(), fx.σ2, ctx=ctx) + mτ


def predict_var(cov, τ, t, σ2, y=None, *, ctx=None):
    """Posterior variance of the zero-mean GP's latent f at ascending τ: the diagonal of predict_cov
    (src/direct_solver.jl:28-119) in O((N + M)·R²), without measurement noise.  With y, (mean, var)."""
    ctx = ctx or get_context()
    a, b, c, d = celerite_coefs(cov)
    τ = np.asarray(τ, dtype=np.float64)
    ser = ctx.upload_series(t, np.zeros_like(t) if y is None else y, σ2)
    try:
        out = ctx.celerite_predict_var(ser, a, b, c, d, τ, return_mean=y is not None)
    finally:
        ser.free()
    return (out[0][0], out[1][0]) if y is not None else out[0]


def mean_and_var(fp, τ=None, *, ctx=None):
    """mean_and_var(fp[, τ])  (AbstractGPs): posterior mean and the variance of the latent f at τ (default: the data
    times), from one factorisation.  The mean function shifts the mean only."""
    if not isinstance(fp, PosteriorGP):
        raise TypeError("mean_and_var expects posterior(f(t, σ²), y)")
    fx = fp.f
    τ = fx.x if τ is None else np.asarray(τ, dtype=np.float64)
    m = fx.f.mean
    mτ = m(τ) if callable(m) else np.full(τ.shape, float(m))
    mu, v = predict_var(fx.f.kernel, τ, fx.x, fx.σ2, fp.y - fx.mean_vector(), ctx=ctx)
    return mu + mτ, v


def var(fp, τ=None, *, ctx=None):
    """var(fp[, τ])  (AbstractGPs; diag of cov(fp, τ), src/scalable_GP.jl:44-155): the posterior variance of the latent
    f at τ (default: the data times), measurement noise not included."""
    if not isinstance(fp, PosteriorGP):
        raise TypeError("var expects posterior(f(t, σ²), y)")
    fx = fp.f
    τ = fx.x if τ is None else np.asarray(τ, dtype=np.float64)
    return predict_var(fx.f.kernel, τ, fx.x, fx.σ2, ctx=ctx)


def std(fp, τ=None, *, ctx=None):
    """std(fp[, τ]) = √max(var, 0): at a data point with a tiny σ² the exact variance is close to 0 and rounding can
    make the computed one slightly negative; it is clamped to 0 rather than turned into NaN."""
    return np.sqrt(np.maximum(var(fp, τ, ctx=ctx), 0.0))


def predict_cov(cov, τ, t, σ2, y=None, *, ctx=None):
    """predict_cov(cov, τ, t, y, σ²)  (src/direct_solver.jl:28-119): the M × M posterior covariance of the zero-mean GP's
    latent f at ascending τ, without measurement noise, exactly symmetric; O((N + M)·R² + M·(N + M)·R) instead of the dense
    O(N³).  With y, (mean, cov)."""
    ctx = ctx or get_context()
    a, b, c, d = celerite_coefs(cov)
    τ = np.asarray(τ, dtype=np.float64)
    ser = ctx.upload_series(t, np.zeros_like(t) if y is None else y, σ2)
    try:
        out = ctx.celerite_predict_cov(ser, a, b, c, d, τ, return_mean=y is not None)
    finally:
        ser.free()
    return (out[0][0], out[1][0]) if y is not None else out[0]


def mean_and_cov(fp, τ=None, *, ctx=None):
    """mean_and_cov(fp[, τ])  (AbstractGPs): posterior mean and the covariance of the latent f at τ (default: the data
    times), from one factorisation.  The mean function shifts the mean only."""
    if not isinstance(fp, PosteriorGP):
        raise TypeError("mean_and_cov expects posterior(f(t, σ²), y)")
    fx = fp.f
    τ = fx.x if τ is None else np.asarray(τ, dtype=np.float64)
    m = fx.f.mean
    mτ = m(τ) if callable(m) else np.full(τ.shape, float(m))
    mu, C = predict_cov(fx.f.kernel, τ, fx.x, fx.σ2, fp.y - fx.mean_vector(), ctx=ctx)
    return mu + mτ, C


def cov(fp, τ=None, *, ctx=None):
    """cov(fp[, τ])  (AbstractGPs; predict_cov, src/direct_solver.jl:28-119): the M × M posterior covariance of the latent
    f at τ (default: the data times), measurement noise not included."""
    if not isinstance(fp, PosteriorGP):
        raise TypeError("cov expects posterior(f(t, σ²), y)")
    fx = fp.f
    τ = fx.x if τ is None else np.asarray(τ, dtype=np.float64)
    return predict_cov(fx.f.kernel, τ, fx.x, fx.σ2, ctx=ctx)


def simulate(cov, τ, σ2, q, *, ctx=None):
    """simulate(rng, cov, τ, σ²)  (src/celerite_solver.jl:497-549) with the standard-normal draws q supplied by the caller
    (q = randn(rng, N) in the reference)."""
    ctx = ctx or get_context()
    a, b, c, d = celerite_coefs(cov)
    τ = np.asarray(τ, dtype=np.float64)
    ser = ctx.upload_series(τ, np.zeros_like(τ), σ2)
    try:
        return ctx.celerite_simulate(ser, a, b, c, d, np.asarray(q, dtype=np.float64).reshape(1, -1))[0]
    finally:
        ser.free()


def posterior_draws(fpx, q, *, ctx=None):
    """rand(rng, fp(τ, σ²), n) for fpx = posterior(f(t, σ²), y)(τ, σ²): draws of the latent f at τ conditioned on the data,
    plus noise of variance σ², by Matheron's rule (a prior draw on the merged grid of t and τ, corrected by the posterior
    mean of its residual at the data).  q [N + M] or [S, N + M] holds standard normals in merged-grid order (a data point
    first at a tie); the result is [M] or [S, M].  The mean function is handled as in mean: the draws are made for y − m(t)
    and m(τ) is added.  For the same q the draws differ from those of a dense Cholesky of cov(fp, τ); their distribution
    is the same."""
    fp = fpx.fp
    fx = fp.f
    τ = fpx.x
    q = np.asarray(q, dtype=np.float64)
    one = q.ndim == 1
    ctx = ctx or get_context()
    a, b, c, d = celerite_coefs(fx.f.kernel)
    m = fx.f.mean
    mτ = m(τ) if callable(m) else np.full(τ.shape, float(m))
    ser = ctx.upload_series(fx.x, fp.y - fx.mean_vector(), fx.σ2)
    try:
        out = ctx.celerite_posterior_draws(ser, a, b, c, d, τ, q.reshape(1, -1, q.shape[-1]), sigma2_tau=fpx.σ2)[0]
    finally:
        ser.free()
    out += mτ
    return out[0] if one else out


def rand(fx, q, t=None, *, ctx=None):
    """rand(rng, f(t, σ²)[, t'])  (src/scalable_GP.jl:133-155): one realisation on the GP's own times with its noise
    variances, or on other times t' without noise; the mean function is added.  For fx = posterior(...)(τ, σ²), draws of
    the posterior (posterior_draws)."""
    if isinstance(fx, FinitePosteriorGP):
        if t is not None:
            raise TypeError("rand(fp(τ, σ²), q) takes no second time vector")
        return posterior_draws(fx, q, ctx=ctx)
    if not isinstance(fx, FiniteScalableGP):
        raise TypeError("rand expects ScalableGP(...)(t, σ²)")
    m = fx.f.mean
    if t is None:
        return simulate(fx.f.kernel, fx.x, fx.σ2, q, ctx=ctx) + fx.mean_vector()
    t = np.asarray(t, dtype=np.float64)
    mt = m(t) if callable(m) else np.full(t.shape, float(m))
    return simulate(fx.f.kernel, t, np.zeros_like(t), q, ctx=ctx) + mt


def lombscargle(t, y, dy=None, *, frequencies, ctx=None):
    """lombscargle(t, y[, dy]; frequencies)  (LombScargle.jl's defaults: fit_mean, center_data, :standard normalisation):
    the generalised Lomb–Scargle power of y [N] or of each row of y [B × N] at the positive frequencies (inverse unit of t),
    [F] or [B × F], weighted by 1/dy² when the errors dy are given.  The times may come in any order; they must be distinct.
    Where the formula divides zero by zero (a constant row, N = 1, a frequency at which the basis is degenerate on these
    times) the power is NaN."""
    ctx = ctx or get_context()
    t = np.asarray(t, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    one = y.ndim == 1
    Y = np.atleast_2d(y)
    if t.ndim != 1 or Y.ndim != 2 or Y.shape[1] != t.shape[0]:
        raise ValueError(f"y must be [N] or [B, N] with N = {t.shape[0]}, got {list(y.shape)}")
    s2 = np.ones_like(t) if dy is None else np.broadcast_to(np.asarray(dy, dtype=np.float64), t.shape) ** 2
    order = np.argsort(t, kind="stable")   # the periodogram does not depend on the order of the points
    ser = ctx.upload_series(t[order], np.zeros_like(t), s2[order])
    try:
        out = ctx.lombscargle(ser, frequencies, y_batch=Y[:, order], weighted=dy is not None)
    finally:
        ser.free()
    return out[0] if one else out


# ----------------------------------------------------------------------------------------------- batched entry
class BatchedLikelihood:
    """Vectorised log-likelihood of the samplers' model (examples/ultranest/single_pl.jl:65-93):
        Θ row = [psd parameters…, variance, ν, μ]  →  logpdf(ScalableGP(μ, approx(𝓟, f_min, f_max, J, variance))(t, ν·σ²), y)
    The series (and its trig/exp table) is uploaded once; each call runs K1 + K2 on the whole batch."""

    def __init__(self, t, y, σ2, psd_model="SingleBendingPowerLaw", n_components=20, basis_function="SHO",
                 f_min=None, f_max=None, S_low=20.0, S_high=20.0, is_integrated_power=True, ctx=None, log_shift=False,
                 n_features=0, gradient="forward", periodic_mean=False):
        # n_features: Θ rows end with (S₀, f₀, Q) per QPO feature added to the continuum (docs/src/adding_features.md)
        self.n_features = int(n_features)
        if self.n_features and log_shift:
            raise ValueError("PSD features and the log-shift transform cannot be combined in one fused call")
        # periodic_mean: Θ rows end with (A, ϕ, T₀) and the mean is μ + A·sin(2πt/T₀ + ϕ)
        # (examples/ultranest/single_pl_periodicity.jl)
        self.periodic_mean = bool(periodic_mean)
        if self.periodic_mean and (self.n_features or log_shift):
            raise ValueError("the periodic mean cannot be combined with PSD features or the log-shift transform in one fused call")
        # gradient: "forward" (one K5g direction per Θ column) or "reverse" (one K5r sweep); only the gradient with features has
        # both — without them c and d are fixed by the spectral grid and the fused approx-path gradient serves every column
        if gradient not in ("forward", "reverse"):
            raise ValueError(f"gradient must be 'forward' or 'reverse', not {gradient!r}")
        if gradient == "reverse" and not self.n_features:
            raise ValueError("gradient='reverse' needs n_features > 0 (the approx path without features has one gradient kernel)")
        self.gradient_mode = gradient
        # log_shift: Θ rows carry a 7th column c and the data enter as yn = log(y − c), σ² = ν σ²/(y − c)²
        # (docs/src/ultranest.md:197-217); t, y, σ2 are then the untransformed flux and its measurement variance
        self.log_shift = bool(log_shift)
        self.ctx = ctx or get_context()
        t = np.asarray(t, dtype=np.float64)
        if f_min is None:
            f_min = 1.0 / (t[-1] - t[0])             # examples/ultranest/single_pl.jl:48
        if f_max is None:
            f_max = 1.0 / np.min(np.diff(t)) / 2.0
        if isinstance(psd_model, type):
            psd_model = psd_model.model_name
        self.spec = make_spec(psd_model, f_min, f_max, n_components, S_low, S_high, is_integrated_power, basis_function)
        self.series = self.ctx.upload_series(t, y, σ2)
        self.n_par = (backend.N_PSD_PAR[self.spec.psd_model] + 3 + int(self.log_shift) + 3 * self.n_features +
                      3 * int(self.periodic_mean))

    def __call__(self, theta):
        theta = np.atleast_2d(np.asarray(theta, dtype=np.float64))
        if self.n_features:
            return self.ctx.approx_features_logl(self.series, self.spec, self.n_features, theta)
        if self.log_shift:
            return self.ctx.approx_logl_logshift(self.series, self.spec, theta)
        if self.periodic_mean:
            return self.ctx.approx_logl_sine(self.series, self.spec, theta)
        return self.ctx.approx_logl(self.series, self.spec, theta)[0]

    def value_and_gradient(self, theta):
        """(logL [B], ∂logL/∂Θ [B × n_par]) — what ForwardDiff.gradient gives the reference's HMC/NUTS runs
        (test/test_likelihood.jl:55, examples/turing_distributed/single_pl.jl), for a whole batch of chains at once."""
        theta = np.atleast_2d(np.asarray(theta, dtype=np.float64))
        if self.n_features:
            if self.gradient_mode == "reverse":
                return self.ctx.approx_features_logl_grad_reverse(self.series, self.spec, self.n_features, theta)
            return self.ctx.approx_features_logl_grad(self.series, self.spec, self.n_features, theta)
        if self.log_shift:
            return self.ctx.approx_logl_logshift_grad(self.series, self.spec, theta)
        if self.periodic_mean:
            return self.ctx.approx_logl_sine_grad(self.series, self.spec, theta)
        return self.ctx.approx_logl_grad(self.series, self.spec, theta)

    def gradient(self, theta):
        return self.value_and_gradient(theta)[1]

    def close(self):
        self.series.free()


class BatchedCARMALikelihood:
    """Vectorised log-likelihood of the reference's CARMA(p, q) model (docs/src/carma.md:20-58):
        Θ row = [qa (p quadratic coefficients of the AR polynomial), qb (q, of the MA polynomial), variance, ν, μ(, c)]
        rα = quad2roots(qa), rβ = quad2roots(qb), β = roots2coeffs(rβ), 𝓒 = CARMA(p, q, rα, β, variance),
        logpdf(ScalableGP(μ, 𝓒)(t, σ²), yn)   with  yn = log(y − c), σ² = ν σ²/(y − c)²  when log_shift (else yn = y, σ² = ν σ²).
    Rows whose roots leave (−f_max, −f_min) × (−f_max, f_max) get −Inf, as the model's `@addlogprob! -Inf` does.  The decay
    rates and frequencies depend on Θ, so this goes through the generic coefficient entry (host arithmetic on p + q numbers per
    row, then ONE kernel call for the batch); the per-row data of the log-shift ride along as y_batch / s2_batch."""

    def __init__(self, t, y, σ2, p, q, f_min, f_max, log_shift=True, ctx=None):
        self.ctx = ctx or get_context()
        self.p, self.q, self.f_min, self.f_max, self.log_shift = int(p), int(q), float(f_min), float(f_max), bool(log_shift)
        if self.p < 1 or self.q < 0 or self.q > self.p:
            raise ValueError("need 1 <= p and 0 <= q <= p")
        self.y, self.σ2 = np.asarray(y, dtype=np.float64), np.asarray(σ2, dtype=np.float64)
        self.series = self.ctx.upload_series(t, self.y, self.σ2)
        self.n_par = self.p + self.q + 3 + int(self.log_shift)

    def _roots_ok(self, r):
        return bool(np.all((-self.f_max < r.real) & (r.real < -self.f_min) & (-self.f_max < r.imag) & (r.imag < self.f_max)))

    def coefficients(self, theta):
        """(ok [B], a, b, c, d [B × J]) for the rows of Θ; rows outside the root bounds keep placeholder coefficients."""
        theta = np.atleast_2d(np.asarray(theta, dtype=np.float64))
        if theta.shape[1] != self.n_par:
            raise ValueError(f"theta must have {self.n_par} columns")
        B, J = theta.shape[0], (self.p + 1) // 2
        ok = np.zeros(B, dtype=bool)
        a, b, c, d = (np.ones((B, J)) for _ in range(4))
        for i in range(B):
            rα = quad2roots(theta[i, :self.p])
            rβ = quad2roots(theta[i, self.p:self.p + self.q])
            if not (self._roots_ok(rα) and (self.q == 0 or self._roots_ok(rβ))):
                continue
            β = np.real(roots2coeffs(rβ)) if self.q > 0 else np.ones(1)
            a[i], b[i], c[i], d[i] = carma_celerite_coefs(self.p, rα, β, theta[i, self.p + self.q])
            ok[i] = True
        return ok, a, b, c, d

    def __call__(self, theta):
        theta = np.atleast_2d(np.asarray(theta, dtype=np.float64))
        ok, a, b, c, d = self.coefficients(theta)
        k = self.p + self.q
        out = np.full(theta.shape[0], -np.inf)
        if ok.any():
            sel = np.flatnonzero(ok)
            yb = sb = None
            if self.log_shift:
                shift = self.y[None, :] - theta[sel, k + 3:k + 4]
                with np.errstate(invalid="ignore", divide="ignore"):
                    yb, sb = np.log(shift), self.σ2[None, :] / shift ** 2
            out[sel] = self.ctx.celerite_logl(self.series, a[sel], b[sel], c[sel], d[sel], mu=theta[sel, k + 2], nu=theta[sel, k + 1],
                                              y_batch=yb, s2_batch=sb)
        return out

    def value_and_gradient(self, theta):
        """(logL [B], ∂logL/∂Θ [B × n_par]) in the column order of Θ.  The coefficients' Jacobian with respect to (qa, qb, variance)
        is formed on the host (carma_celerite_coefs_jacobian), the gradient with respect to the coefficients, ν, μ and, with the
        log shift, the data row comes from one reverse-mode call (K5r) for the batch, and the chain rule joins them.  Rows outside
        the root bounds get logL = −Inf and a zero gradient."""
        theta = np.atleast_2d(np.asarray(theta, dtype=np.float64))
        if theta.shape[1] != self.n_par:
            raise ValueError(f"theta must have {self.n_par} columns")
        B, k = theta.shape[0], self.p + self.q
        out, grad = np.full(B, -np.inf), np.zeros((B, self.n_par))
        rows = []
        for i in range(B):
            rα = quad2roots(theta[i, :self.p])
            rβ = quad2roots(theta[i, self.p:k])
            if self._roots_ok(rα) and (self.q == 0 or self._roots_ok(rβ)):
                rows.append((i, carma_celerite_coefs_jacobian(self.p, self.q, theta[i, :self.p], theta[i, self.p:k], theta[i, k])))
        if not rows:
            return out, grad
        sel = np.array([i for i, _ in rows])
        a, b, c, d = (np.array([co[0][j] for _, co in rows]) for j in range(4))
        jac = [np.array([co[1][j] for _, co in rows]) for j in range(4)]   # [n × J × (k + 1)] each
        yb = sb = None
        if self.log_shift:
            shift = self.y[None, :] - theta[sel, k + 3:k + 4]
            with np.errstate(invalid="ignore", divide="ignore"):
                yb, sb = np.log(shift), self.σ2[None, :] / shift ** 2
        L, g = self.ctx.celerite_logl_vjp(self.series, a, b, c, d, mu=theta[sel, k + 2], nu=theta[sel, k + 1], y_batch=yb,
                                          s2_batch=sb, data_grad=self.log_shift)
        out[sel] = L
        grad[sel, :k + 1] = sum(np.einsum("nj,njp->np", g[x], jac[j]) for j, x in enumerate("abcd"))
        grad[sel, k + 1], grad[sel, k + 2] = g["nu"], g["mu"]
        if self.log_shift:
            # yn = log(y − c): dyn/dc = −1/(y − c);  s2 = σ²/(y − c)²: ds2/dc = 2σ²/(y − c)³ (ν is applied inside the kernel)
            with np.errstate(invalid="ignore", divide="ignore"):
                grad[sel, k + 3] = np.sum(-g["y"] / shift + g["s2"] * 2.0 * self.σ2[None, :] / shift ** 3, axis=1)
        return out, grad

    def gradient(self, theta):
        return self.value_and_gradient(theta)[1]

    def close(self):
        self.series.free()
