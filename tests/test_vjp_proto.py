"""The K5r adjoint step rule (tests/tools/proto/vjp_math.py) against the dual-number oracle tests/tools/oracle_jvp.c by duality:
for random directions v over every input (a, b, c, d, μ, ν, y, σ²), ⟨∇logL, v⟩ equals the oracle's JVP along v.  And the host
Jacobian of the CARMA coefficients (carma_celerite_coefs_jacobian) against central differences of carma_celerite_coefs."""
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "tools", "proto"))
sys.path.insert(0, os.path.join(HERE, "tools"))
import oracle_jvp  # noqa: E402
import vjp_math as vm  # noqa: E402

GRAD_KEYS = (("a", "da"), ("b", "db"), ("c", "dc"), ("d", "dd"), ("y", "dy"), ("s2", "ds2"))


def _problem(rank, N, seed, B=2):
    """B coefficient sets of the given rank: complex terms, one real term when the rank is odd, mixed and negative signs."""
    rng = np.random.default_rng(seed)
    Jt = (rank + 1) // 2
    a = rng.normal(size=(B, Jt)); b = rng.normal(size=(B, Jt))
    c = rng.uniform(0.1, 2.0, (B, Jt)); d = rng.normal(scale=2.0, size=(B, Jt))
    a[:, 0] = np.abs(a[:, 0]) + 2.0 * Jt           # keeps most pivots positive; the sign of the others does not matter
    if rank % 2:
        b[:, -1] = 0.0; d[:, -1] = 0.0
    t = np.cumsum(rng.uniform(0.2, 1.5, N))
    y, s2 = rng.normal(size=N), rng.uniform(0.2, 0.4, N)
    mu, nu = rng.normal(size=B), rng.uniform(0.5, 1.5, B)
    yb, sb = rng.normal(size=(B, N)), rng.uniform(0.2, 0.4, (B, N))
    return rng, (a, b, c, d), t, y, s2, mu, nu, yb, sb


@pytest.mark.parametrize("rank", [2, 3, 5, 8, 12])
@pytest.mark.parametrize("N", [1, 2, 50])
def test_adjoint_equals_oracle_jvp_by_duality(rank, N):
    rng, (a, b, c, d), t, y, s2, mu, nu, yb, sb = _problem(rank, N, 100 * rank + N)
    B, Jt = a.shape
    L, G = vm.logl_vjp_batch(a, b, c, d, t, y, s2, mu, nu, y_batch=yb, s2_batch=sb)
    P = 6
    tan = {"da": rng.normal(size=(B, P, Jt)), "db": rng.normal(size=(B, P, Jt)), "dc": rng.normal(size=(B, P, Jt)),
           "dd": rng.normal(size=(B, P, Jt)), "dmu": rng.normal(size=(B, P)), "dnu": rng.normal(size=(B, P)),
           "dy": rng.normal(size=(B, P, N)), "ds2": rng.normal(size=(B, P, N))}
    Lo, Go = oracle_jvp.celerite_logl_jvp_batch(a, b, c, d, t, y, s2, mu=mu, nu=nu, y_batch=yb, s2_batch=sb, **tan)
    assert np.allclose(L, Lo, rtol=1e-12, atol=1e-12)
    dot = G["mu"][:, None] * tan["dmu"] + G["nu"][:, None] * tan["dnu"]
    for g, v in GRAD_KEYS:
        dot = dot + np.einsum("ij,ipj->ip", G[g], tan[v])
    assert np.all(np.abs(dot - Go) <= 1e-10 * np.maximum(1.0, np.abs(Go))), np.max(np.abs(dot - Go))


def test_real_terms_report_zero_b_d():
    _, (a, b, c, d), t, y, s2, mu, nu, _, _ = _problem(5, 40, 7)
    _, G = vm.logl_vjp_batch(a, b, c, d, t, y, s2, mu, nu)
    assert np.all(G["b"][:, -1] == 0.0) and np.all(G["d"][:, -1] == 0.0)


# ---------------------------------------------------------------------------------------------------- CARMA coefficient Jacobian
def _api():
    import pioran_b200  # noqa: F401  (registers the package's modules)
    return next(m for k, m in sys.modules.items() if k.endswith(".api") and hasattr(m, "carma_celerite_coefs_jacobian"))


@pytest.mark.parametrize("p", [1, 2, 3, 4, 5, 6])
def test_carma_coefficient_jacobian_matches_central_differences(p):
    api = _api()
    rng = np.random.default_rng(p)
    for q in range(p + 1):
        qa, qb, var = rng.uniform(0.3, 2.0, p), rng.uniform(0.3, 2.0, q), rng.uniform(0.5, 2.0)
        x0 = np.concatenate([qa, qb, [var]])

        def coefs(x):
            rα, rβ = api.quad2roots(x[:p]), api.quad2roots(x[p:p + q])
            β = np.real(api.roots2coeffs(rβ)) if q > 0 else np.ones(1)
            return np.concatenate(api.carma_celerite_coefs(p, rα, β, x[p + q]))

        co, jac = api.carma_celerite_coefs_jacobian(p, q, qa, qb, var)
        np.testing.assert_allclose(np.concatenate(co), coefs(x0), rtol=1e-12, atol=1e-14)
        J = np.concatenate(jac, axis=0)
        h = 1e-6
        cd = np.stack([(coefs(x0 + h * e) - coefs(x0 - h * e)) / (2 * h) for e in np.eye(x0.shape[0])], axis=1)
        scale = np.maximum(1.0, np.max(np.abs(cd), axis=0))   # per column: central differences carry rounding of |coefs| / h
        assert np.all(np.abs(J - cd) <= 1e-7 * scale[None, :]), (q, np.max(np.abs(J - cd) / scale[None, :]))
