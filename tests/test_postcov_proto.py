"""The posterior-covariance walk K8 (tests/tools/proto/postcov_math.py) against the dense posterior covariance
K_ττ − K_τt (K + diag σ²)⁻¹ K_tτ, solved here with a Cholesky factor: the series and prediction grids of
tests/test_posterior.py, explicit sets with real terms, the shortest series and a single prediction point."""
import os
import sys

import numpy as np
import pytest

from conftest import GOLDEN
from oracle import oracle as orc

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "tools", "proto"))
import postcov_math as cm  # noqa: E402
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


def check(a, b, c, d, t, s2, tau, what):
    a, b, c, d = (np.asarray(x, dtype=np.float64) for x in (a, b, c, d))
    got = cm.predict_cov(a, b, c, d, t, s2, tau)
    assert np.array_equal(got, got.T), f"{what}: not exactly symmetric"
    err, ld = cm.conditioned_error(got, a, b, c, d, t, s2, tau, 1e-12)
    if ld is not None:
        # An ill-conditioned solve: then the FP64 dense covariance is itself off the 80-bit one, and the walk must be at
        # least as close to the 80-bit covariance as the dense one.
        assert ld[0] <= max(1e-12, ld[1]), f"{what}: {err:.2e} from the dense covariance; 80-bit: {ld[0]:.2e} against {ld[1]:.2e}"
    return got


def test_merged_grid_puts_tau_first_at_a_tie():
    G, code = cm.merged_grid_tau_first([1.0, 2.0, 3.0], [0.5, 2.0, 2.0, 3.5])
    assert np.array_equal(G, [0.5, 1.0, 2.0, 2.0, 2.0, 3.0, 3.5])
    assert np.array_equal(code, [-1, 0, -2, -3, 1, 2, -4])


@pytest.mark.parametrize("basis", ["SHO", "DRWCelerite"])
def test_walk_matches_dense_on_the_posterior_grids(basis):
    a, b, c, d = orc.approx("SBPL", [0.82, 0.01, 3.3], F0, FM, 20, VAR, basis=basis)
    for name, tau in list(grids().items()) + [("edge points", EDGE)]:
        check(a, b, c, d, T, S2, tau, f"{basis}, {name}")


def test_diagonal_is_the_posterior_variance():
    a, b, c, d = orc.approx("SBPL", [0.82, 0.01, 3.3], F0, FM, 20, VAR, basis="SHO")
    got = cm.predict_cov(a, b, c, d, T, S2, EDGE)
    var = pm.predict_var(a, b, c, d, T, S2, EDGE)
    assert np.max(np.abs(np.diag(got) - var)) <= 1e-13 * np.sum(a)


def test_far_points_recover_the_prior_covariance():
    a, b, c, d = orc.approx("SBPL", [0.82, 0.01, 3.3], F0, FM, 20, VAR, basis="SHO")
    tau = np.array([T[0] - 1e7, T[0] - 1e7 + 0.5, T[-1] + 1e7])
    got = cm.predict_cov(a, b, c, d, T, S2, tau)
    want = pm.kernel(np.asarray(a), np.asarray(b), np.asarray(c), np.asarray(d), tau[:, None] - tau[None, :])
    # rows at absolute times |x| ≈ 1e7 carry the argument rounding of cos(d x), sin(d x) (about d·|x|·ε) into the
    # off-diagonal prior term, which the dense route forms from the lag: 1e-12·Σa at these points
    assert np.allclose(got, want, rtol=0, atol=1e-11 * np.sum(a))


def _mixed(J, seed, n_real):
    rng = np.random.default_rng(seed)
    a, b = rng.uniform(0.2, 1.0, J), rng.uniform(-0.1, 0.1, J)
    c = 10 ** rng.uniform(-3, 0.5, J)
    d = c * rng.uniform(0, 1.5, J)
    b[:n_real] = 0.0
    d[:n_real] = 0.0
    return a, b, c, d


@pytest.mark.parametrize("J,n_real,N,seed", [(3, 1, 60, 1), (12, 3, 400, 2), (6, 6, 150, 3)])
def test_walk_matches_dense_with_real_terms(J, n_real, N, seed):
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
    check(a, b, c, d, t, s2, np.array([1.0, 3.0, 3.0, 3.7, 4.5, 9.0]), f"N={N}")


def test_single_prediction_point():
    a, b, c, d = _mixed(5, 4, 2)
    for x in (T[0] - 2, 0.5 * (T[7] + T[8]), T[9], T[-1] + 2):
        check(a, b, c, d, T, S2, np.array([x]), f"M=1 at {x}")
