"""The posterior-draw recursion K7 (tests/tools/proto/postdraw_math.py) against a dense Matheron draw with the same q
(postdraw_math.dense_draws: the Cholesky factor of K(G, G) + diag(noise) times q on the merged grid, then a dense solve for
the correction); in exact arithmetic the two agree.  The series and grids of
tests/test_posterior.py, explicit sets with real terms, the shortest series and a single prediction point."""
import os
import sys

import numpy as np
import pytest

from conftest import GOLDEN
from oracle import oracle as orc

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "tools", "proto"))
import postdraw_math as dm  # noqa: E402
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


def _chol_ld(A):
    A = A.astype(np.longdouble)
    L = np.zeros_like(A)
    for j in range(len(A)):
        v = A[j:, j] - L[j:, :j] @ L[j, :j]
        L[j, j] = np.sqrt(v[0])
        L[j + 1:, j] = v[1:] / L[j, j]
    return L


def _kernel_ld(a, b, c, d, lag):
    lag = np.abs(lag.astype(np.longdouble))
    out = np.zeros_like(lag)
    for aa, bb, cc, dd in zip(*(x.astype(np.longdouble) for x in (a, b, c, d))):
        out += np.exp(-cc * lag) * (aa * np.cos(dd * lag) + bb * np.sin(dd * lag))
    return out


def dense_draws_ld(a, b, c, d, t, y, s2, tau, q, mu, sigma2_tau):
    """dense_draws in 80-bit arithmetic, with the Cholesky factor and the triangular solves written out."""
    G, code = dm.merged_grid(t, tau)
    noise = np.where(code >= 0, s2[np.maximum(code, 0)], sigma2_tau).astype(np.longdouble)
    L = _chol_ld(_kernel_ld(a, b, c, d, G[:, None] - G[None, :]) + np.diag(noise))
    dat, pre = np.flatnonzero(code >= 0), np.flatnonzero(code < 0)
    dat, pre = dat[np.argsort(code[dat])], pre[np.argsort(-code[pre] - 1)]
    u = np.atleast_2d(q).astype(np.longdouble) @ L.T
    Lk = _chol_ld(_kernel_ld(a, b, c, d, t[:, None] - t[None, :]) + np.diag(s2.astype(np.longdouble)))
    z = (y - mu - u[:, dat]).T
    for i in range(len(t)):
        z[i] = (z[i] - Lk[i, :i] @ z[:i]) / Lk[i, i]
    for i in range(len(t) - 1, -1, -1):
        z[i] = (z[i] - Lk[i + 1:, i] @ z[i + 1:]) / Lk[i, i]
    return mu + u[:, pre] + (_kernel_ld(a, b, c, d, tau[:, None] - t[None, :]) @ z).T


def check(a, b, c, d, t, y, s2, tau, what, S=2, mu=0.3, sigma2_tau=1e-18, seed=0):
    a, b, c, d = (np.asarray(x, dtype=np.float64) for x in (a, b, c, d))
    q = np.random.default_rng(seed).standard_normal((S, len(t) + len(tau)))
    got = dm.posterior_draws(a, b, c, d, t, y, s2, tau, q, mu, sigma2_tau)
    want = dm.dense_draws(a, b, c, d, t, y, s2, tau, q, mu, sigma2_tau)
    err = np.max(np.abs(got - want)) / np.sqrt(np.sum(a))
    if err > 1e-12:
        # An ill-conditioned merged covariance, such as a τ point on a data point with σ²_τ far below the data noise
        # (pivot ≈ 1e-8·Σa on "data times"): then the FP64 dense draw is itself off the 80-bit draw, and the recursion
        # must be at least as close to the 80-bit draw as the dense one.
        ld = dense_draws_ld(a, b, c, d, t, y, s2, tau, q, mu, sigma2_tau)
        e_rec, e_dense = (float(np.max(np.abs(x - ld))) / np.sqrt(np.sum(a)) for x in (got, want))
        assert e_rec <= max(1e-12, e_dense), f"{what}: {err:.2e} from the dense draw; 80-bit: {e_rec:.2e} against {e_dense:.2e}"


def test_merged_grid_puts_data_first_at_a_tie():
    G, code = dm.merged_grid([1.0, 2.0, 3.0], [0.5, 2.0, 2.0, 3.5])
    assert np.array_equal(G, [0.5, 1.0, 2.0, 2.0, 2.0, 3.0, 3.5])
    assert np.array_equal(code, [-1, 0, 1, -2, -3, 2, -4])


@pytest.mark.parametrize("basis", ["SHO", "DRWCelerite"])
def test_recursion_matches_dense_on_the_posterior_grids(basis):
    a, b, c, d = orc.approx("SBPL", [0.82, 0.01, 3.3], F0, FM, 20, VAR, basis=basis)
    for name, tau in grids().items():
        check(a, b, c, d, T, Y, S2, tau, f"{basis}, {name}")


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
    y = rng.normal(size=N)
    tau = np.sort(np.concatenate([[t[0] - 3, t[0]], np.linspace(t[0] - 1, t[-1] + 2, 300), t[5:8], [t[-1], t[-1] + 5]]))
    check(a, b, c, d, t, y, s2, tau, f"J={J}, {n_real} real, N={N}", S=3, seed=seed)


@pytest.mark.parametrize("N", [1, 2])
def test_shortest_series(N):
    a, b, c, d = _mixed(4, 9, 1)
    t, y, s2 = np.array([3.0, 4.5])[:N], np.array([0.3, -0.2])[:N], np.array([0.02, 0.03])[:N]
    check(a, b, c, d, t, y, s2, np.array([1.0, 3.0, 3.7, 4.5, 9.0]), f"N={N}", S=4)


def test_single_prediction_point_and_duplicates_with_noise():
    a, b, c, d = _mixed(5, 4, 2)
    check(a, b, c, d, T, Y, S2, np.array([0.5 * (T[7] + T[8])]), "M=1", S=3)
    # repeated τ: with σ²_τ > 0 the merged covariance stays positive definite
    tau = np.sort(np.concatenate([np.linspace(T[2], T[9], 20), [T[5]] * 3]))
    check(a, b, c, d, T, Y, S2, tau, "repeated τ", S=3, sigma2_tau=1e-6 * np.sum(a))
