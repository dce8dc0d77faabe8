"""The K5g step rule (tests/tools/proto/jvp_math.py, the reference of tests/test_gpu_jvp.py) against the oracle: its value is the
oracle's logl, and its directional derivatives match central differences of the oracle's logl along a, b, c, d, μ, ν, y and σ²,
one at a time and together, on real and complex terms, negative coefficients, and N = 1, 2."""
import os
import sys

import numpy as np
import pytest

from oracle import oracle as orc

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "tools", "proto"))
import jvp_math as jm  # noqa: E402

# real + complex terms with negative a, b, d (the set of test_gpu_parity.py's rank-reduction test), and a positive-definite SHO-like set
SETS = {
    "mixed_signs": (np.array([1.2, 0.8, -0.3, 0.5]), np.array([0.0, 0.3, -0.1, 0.0]),
                    np.array([0.3, 0.2, 1.0, 2.0]), np.array([0.0, 1.5, -2.0, 0.0])),
    "sho": (np.array([0.7, 0.4, 0.2]), np.array([0.7, 0.4, 0.2]),
            np.array([0.9, 2.5, 6.0]), np.array([0.9, 2.5, 6.0])),
}
NAMES = ("da", "db", "dc", "dd", "dmu", "dnu", "dy", "ds2")


def _series(N, seed=0):
    rng = np.random.default_rng(seed)
    t = np.cumsum(rng.uniform(0.2, 1.5, N))
    return t, rng.normal(size=N), rng.uniform(0.2, 0.4, N)


def _direction(rng, name, Jt, N):
    if name in ("dmu", "dnu"):
        return float(rng.normal())
    return rng.normal(size=N if name in ("dy", "ds2") else Jt)


def _cd_tol(cd):
    return 2e-7 * max(1.0, abs(cd))   # central differences at h = 1e-6 carry ~1e-9 … 1e-8 of rounding noise


@pytest.mark.parametrize("which", sorted(SETS))
@pytest.mark.parametrize("N", [1, 2, 40])
def test_value_equals_oracle(which, N):
    a, b, c, d = SETS[which]
    t, y, s2 = _series(N)
    L, _ = jm.logl_jvp(a, b, c, d, t, y, s2, 0.2, 1.1, dnu=np.ones(1))
    want = orc.celerite_logl(a, b, c, d, t, y - 0.2, 1.1 * s2)
    assert abs(L - want) <= 1e-12 * max(1.0, abs(want))


@pytest.mark.parametrize("which", sorted(SETS))
@pytest.mark.parametrize("N", [1, 2, 40])
def test_each_direction_matches_central_differences(which, N):
    a, b, c, d = SETS[which]
    t, y, s2 = _series(N, 1)
    rng = np.random.default_rng(2)
    mu, nu = -0.1, 0.9
    dirs = {n: _direction(rng, n, len(a), N) for n in NAMES}
    tan = {n: np.zeros((len(NAMES),) + np.shape(v)) for n, v in dirs.items()}   # P = 8: one direction per input
    for p, n in enumerate(NAMES):
        tan[n][p] = dirs[n]
    _, g = jm.logl_jvp(a, b, c, d, t, y, s2, mu, nu, **tan)
    for p, n in enumerate(NAMES):
        cd = jm.central_difference(a, b, c, d, t, y, s2, mu, nu, {n: dirs[n]})
        assert abs(g[p] - cd) <= _cd_tol(cd), (n, g[p], cd)


@pytest.mark.parametrize("which", sorted(SETS))
def test_all_directions_together_match_central_differences(which):
    a, b, c, d = SETS[which]
    N = 40
    t, y, s2 = _series(N, 3)
    rng = np.random.default_rng(4)
    dirs = {n: _direction(rng, n, len(a), N) for n in NAMES}
    _, g = jm.logl_jvp(a, b, c, d, t, y, s2, 0.3, 1.2, **{n: np.array([v]) for n, v in dirs.items()})
    cd = jm.central_difference(a, b, c, d, t, y, s2, 0.3, 1.2, dirs)
    assert abs(g[0] - cd) <= _cd_tol(cd)


def test_real_terms_ignore_db_dd():
    """b = d = 0 for a term of every set: the term takes one row and its db, dd tangents are exactly without effect."""
    a, b, c, d = SETS["mixed_signs"]
    t, y, s2 = _series(30, 5)
    real = (b == 0) & (d == 0)
    tan = np.where(real, 1.0, 0.0)[None]
    _, g = jm.logl_jvp(a, b, c, d, t, y, s2, db=tan, dd=tan)
    assert g[0] == 0.0
    cd = jm.central_difference(a, b, c, d, t, y, s2, 0.0, 1.0, {"db": tan[0], "dd": tan[0]})
    assert abs(cd) <= 1e-8
