"""The posterior-variance recursion K6 (tests/tools/proto/postvar_math.py) against the dense posterior covariance diagonal
k(0) − k(τ, t)ᵀ (K + diag σ²)⁻¹ k(τ, t), solved here with a Cholesky factor: the series and prediction grids of
tests/test_posterior.py, explicit sets with real terms, and the shortest series."""
import os
import sys

import numpy as np
import pytest
from scipy.linalg import cho_factor, cho_solve

from conftest import GOLDEN
from oracle import oracle as orc

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "tools", "proto"))
import postvar_math as pm  # noqa: E402

A = np.loadtxt(os.path.join(GOLDEN, "simu.txt"))
T, Y, YERR = (np.ascontiguousarray(c) for c in A.T)
S2 = YERR ** 2
F0 = 1 / (T[-1] - T[0]) / 100
FM = 1 / np.min(np.diff(T)) / 2 * 20
VAR = np.var(Y, ddof=1)


def grids():   # tests/test_posterior.py::grids
    rng = np.random.default_rng(7)
    return {
        "data times": T,
        "fine grid": np.linspace(T.min(), T.max(), 1000),
        "beyond the data": np.linspace(T.min() - 30, T.max() + 30, 1000),
        "random": np.sort(rng.random(1000)) * (T[-1] - T[0]) * 2 + (T[0] - T[-1] / 2),
    }


EDGE = np.sort(np.concatenate([[T[0] - 5, T[0] - 1e-3, T[0]], np.linspace(T[3], T[4], 7), T[10:13],
                               [0.5 * (T[20] + T[21])] * 3, [T[-1], T[-1] + 1e-3, T[-1] + 40]]))


def dense_var(a, b, c, d, t, s2, tau):
    K = pm.kernel(a, b, c, d, t[:, None] - t[None, :]) + np.diag(s2)
    k = pm.kernel(a, b, c, d, tau[:, None] - t[None, :])
    return np.sum(a) - np.einsum("mn,nm->m", k, cho_solve(cho_factor(K, lower=True), k.T))


def check(a, b, c, d, t, s2, tau, what):
    got = pm.predict_var(a, b, c, d, t, s2, tau)
    want = dense_var(np.asarray(a), np.asarray(b), np.asarray(c), np.asarray(d), t, s2, tau)
    err = np.max(np.abs(got - want)) / np.sum(a)
    assert err <= 1e-12, f"{what}: {err:.2e}"
    return got


@pytest.mark.parametrize("basis", ["SHO", "DRWCelerite"])
def test_recursion_matches_dense_on_the_posterior_grids(basis):
    a, b, c, d = orc.approx("SBPL", [0.82, 0.01, 3.3], F0, FM, 20, VAR, basis=basis)
    for name, tau in list(grids().items()) + [("edge points", EDGE)]:
        check(a, b, c, d, T, S2, tau, f"{basis}, {name}")


def test_far_points_recover_the_prior_variance():
    a, b, c, d = orc.approx("SBPL", [0.82, 0.01, 3.3], F0, FM, 20, VAR, basis="SHO")
    got = pm.predict_var(a, b, c, d, T, S2, np.array([T[0] - 1e7, T[-1] + 1e7]))
    assert np.allclose(got, np.sum(a), rtol=1e-12, atol=0)


def _mixed(J, seed, n_real):
    rng = np.random.default_rng(seed)
    a, b = rng.uniform(0.2, 1.0, J), rng.uniform(-0.1, 0.1, J)
    c = 10 ** rng.uniform(-3, 0.5, J)
    d = c * rng.uniform(0, 1.5, J)
    b[:n_real] = 0.0
    d[:n_real] = 0.0
    return a, b, c, d


@pytest.mark.parametrize("J,n_real,N,seed", [(3, 1, 60, 1), (12, 3, 400, 2), (6, 6, 150, 3)])
def test_recursion_matches_dense_with_real_terms(J, n_real, N, seed):
    a, b, c, d = _mixed(J, seed, n_real)
    rng = np.random.default_rng(seed + 10)
    t = np.sort(rng.uniform(0, 4 * N, N))
    s2 = rng.uniform(0.01, 0.05, N)
    tau = np.sort(np.concatenate([[t[0] - 3, t[0]], np.linspace(t[0] - 1, t[-1] + 2, 300), t[5:8], t[5:6],
                                  [t[-1], t[-1] + 5]]))
    check(a, b, c, d, t, s2, tau, f"J={J}, {n_real} real, N={N}")


@pytest.mark.parametrize("N", [1, 2])
def test_shortest_series(N):
    a, b, c, d = _mixed(4, 9, 1)
    t = np.array([3.0, 4.5])[:N]
    s2 = np.array([0.02, 0.03])[:N]
    tau = np.array([1.0, 3.0, 3.7, 4.5, 9.0])
    check(a, b, c, d, t, s2, tau, f"N={N}")
