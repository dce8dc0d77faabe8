"""The forward-mode oracle of the JVP and of the gradient with PSD features (tests/tools/oracle_jvp.c) — the reference of
tests/test_gpu_jvp.py — against the pinned value oracle and central differences of it."""
import os
import sys

import numpy as np
import pytest

from conftest import synthetic_series
from oracle import oracle as orc

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "tools"))
import oracle_jvp as oj  # noqa: E402

# real + complex terms with negative a, b, d (the rank-reduction set of test_gpu_parity.py), and a positive-definite SHO-like set
SETS = {
    "mixed_signs": (np.array([[1.2, 0.8, -0.3, 0.5], [2.0, 0.1, -0.05, 1.0]]), np.array([[0.0, 0.3, -0.1, 0.0], [0.0, -0.05, 0.02, 0.0]]),
                    np.array([[0.3, 0.2, 1.0, 2.0], [0.1, 0.5, 0.8, 3.0]]), np.array([[0.0, 1.5, -2.0, 0.0], [0.0, 0.7, 1.1, 0.0]])),
    "sho": (np.array([[0.7, 0.4, 0.2]]), np.array([[0.7, 0.4, 0.2]]), np.array([[0.9, 2.5, 6.0]]), np.array([[0.9, 2.5, 6.0]])),
}
NAMES = ("da", "db", "dc", "dd", "dmu", "dnu", "dy", "ds2")


def _series(N, seed):
    rng = np.random.default_rng(seed)
    return np.cumsum(rng.uniform(0.2, 1.5, N)), rng.normal(size=N), rng.uniform(0.2, 0.4, N)


def _tangents(rng, B, P, Jt, N):
    tan = {n: rng.normal(size=(B, P, Jt)) for n in ("da", "db", "dc", "dd")}
    tan.update(dmu=rng.normal(size=(B, P)), dnu=rng.normal(size=(B, P)), dy=rng.normal(size=(B, P, N)),
               ds2=rng.normal(size=(B, P, N)) * 0.1)
    return tan


def _logl_at(a, b, c, d, t, y, s2, mu, nu, tan, i, p, e):
    """orc.celerite_logl of set i moved by e along direction p."""
    s = lambda n, base: base + e * (tan[n][i, p] if n in tan else 0.0)
    return orc.celerite_logl(s("da", a[i]), s("db", b[i]), s("dc", c[i]), s("dd", d[i]), t, s("dy", y) - s("dmu", mu[i]),
                             s("dnu", nu[i]) * s("ds2", s2))


@pytest.mark.parametrize("which", sorted(SETS))
@pytest.mark.parametrize("N", [1, 2, 40])
def test_value_bit_equal_to_oracle(which, N):
    a, b, c, d = SETS[which]
    t, y, s2 = _series(N, 0)
    B = a.shape[0]
    mu, nu = np.full(B, 0.2), np.full(B, 1.1)
    L, _ = oj.celerite_logl_jvp_batch(a, b, c, d, t, y, s2, mu=mu, nu=nu, **_tangents(np.random.default_rng(1), B, 2, a.shape[1], N))
    for i in range(B):
        assert L[i] == orc.celerite_logl(a[i], b[i], c[i], d[i], t, y - mu[i], nu[i] * s2)


@pytest.mark.parametrize("which", sorted(SETS))
@pytest.mark.parametrize("N", [1, 2, 40])
def test_jvp_matches_central_differences(which, N):
    """One direction per input (P = 8) and all inputs together (the last direction)."""
    a, b, c, d = SETS[which]
    t, y, s2 = _series(N, 2)
    B, Jt = a.shape
    rng = np.random.default_rng(3)
    mu, nu = rng.normal(0, 0.3, B), rng.uniform(0.8, 1.3, B)
    full = _tangents(rng, B, 1, Jt, N)
    tan = {n: np.zeros((B, len(NAMES) + 1) + v.shape[2:]) for n, v in full.items()}
    for p, n in enumerate(NAMES):
        tan[n][:, p] = full[n][:, 0]
        tan[n][:, len(NAMES)] = full[n][:, 0]
    _, G = oj.celerite_logl_jvp_batch(a, b, c, d, t, y, s2, mu=mu, nu=nu, **tan)
    h = 1e-6
    for i in range(B):
        for p in range(len(NAMES) + 1):
            cd = (_logl_at(a, b, c, d, t, y, s2, mu, nu, tan, i, p, h) - _logl_at(a, b, c, d, t, y, s2, mu, nu, tan, i, p, -h)) / (2 * h)
            assert abs(G[i, p] - cd) <= 2e-7 * max(1.0, abs(cd)), (i, p, G[i, p], cd)


def test_long_double_twin_agrees():
    a, b, c, d = SETS["mixed_signs"]
    t, y, s2 = _series(40, 4)
    tan = _tangents(np.random.default_rng(5), 2, 3, 4, 40)
    _, G = oj.celerite_logl_jvp_batch(a, b, c, d, t, y, s2, **tan)
    _, Gl = oj.celerite_logl_jvp_batch(a, b, c, d, t, y, s2, long_double=True, **tan)
    assert np.abs(G - Gl).max() <= 1e-10 * np.abs(Gl).max()


def _features_theta(rng, B, f_min, f_max, nf):
    cols = [rng.uniform(0.0, 1.0, B), np.exp(rng.uniform(np.log(f_min), np.log(f_max), B)), rng.uniform(2.0, 3.5, B),
            np.exp(rng.normal(-1, 0.5, B)), rng.gamma(2, 0.5, B), rng.normal(0, 0.3, B)]
    for _ in range(nf):
        cols += [rng.uniform(0.5, 3, B), np.exp(rng.uniform(np.log(2 * f_min), np.log(f_max / 2), B)), rng.uniform(1.0, 15, B)]
    return np.column_stack(cols)


def _features_logl(th, nf, f_min, f_max, basis, integrated, t, y, s2):
    a, b, c, d = orc.approx_features("SBPL", th[:3], th[6:6 + 3 * nf].reshape(nf, 3), f_min, f_max, 20, th[3], basis=basis,
                                     is_integrated_power=integrated)
    return orc.celerite_logl(a, b, c, d, t, y - th[5], th[4] * s2)


@pytest.mark.parametrize("nf", [1, 2])
@pytest.mark.parametrize("integrated", [True, False])
@pytest.mark.parametrize("basis", ["SHO", "DRWCelerite"])
def test_features_dual_oracle_matches_central_differences(basis, integrated, nf):
    t, y, s2, f_min, f_max = synthetic_series(150, 9)
    th = _features_theta(np.random.default_rng(11 + nf), 3, f_min, f_max, nf)
    L, G = oj.approx_features_logl_grad_batch("SBPL", th, nf, f_min, f_max, 20, t, y, s2, basis=basis, is_integrated_power=integrated)
    for i in range(th.shape[0]):
        want = _features_logl(th[i], nf, f_min, f_max, basis, integrated, t, y, s2)
        assert abs(L[i] - want) <= 1e-11 * max(1.0, abs(want))
        for k in range(th.shape[1]):
            hp = 1e-4 * max(abs(th[i, k]), 1e-2)   # the features likelihood is noisy at ~1e-12: a wider step
            up, dn = th[i].copy(), th[i].copy()
            up[k] += hp
            dn[k] -= hp
            cd = (_features_logl(up, nf, f_min, f_max, basis, integrated, t, y, s2)
                  - _features_logl(dn, nf, f_min, f_max, basis, integrated, t, y, s2)) / (2 * hp)
            assert abs(G[i, k] - cd) <= 1e-5 * max(1.0, abs(cd)), (i, k, G[i, k], cd)
