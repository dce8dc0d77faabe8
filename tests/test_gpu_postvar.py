"""K6 (csrc/postvar.cuh): the posterior predictive variance of the celerite GP through the C ABI and the Python interface,
against the dense diagonal k(0) − k(τ, t)ᵀ (K + diag νσ²)⁻¹ k(τ, t) solved with a Cholesky factor in the test, on the series
and prediction grids of tests/test_posterior.py; plus the mean it returns alongside (bit for bit pioran_celerite_predict),
the NaN row of a non-positive-definite set, θ-chunking at N = 1e5, the rank limit and the argument checks."""
import ctypes as C
import os
import sys

import numpy as np
import pytest
from scipy.linalg import cho_factor, cho_solve

from conftest import GOLDEN
from oracle import oracle as orc

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "tools", "proto"))
import postvar_math as pm  # noqa: E402

pytestmark = pytest.mark.gpu

A = np.loadtxt(os.path.join(GOLDEN, "simu.txt"))
T, Y, YERR = (np.ascontiguousarray(c) for c in A.T)
S2 = YERR ** 2
F0 = 1 / (T[-1] - T[0]) / 100
FM = 1 / np.min(np.diff(T)) / 2 * 20
VAR = np.var(Y, ddof=1)
TOL = 1e-9   # of Σa


def grids():   # tests/test_posterior.py::grids
    rng = np.random.default_rng(7)
    return {
        "data times": T,
        "fine grid": np.linspace(T.min(), T.max(), 1000),
        "beyond the data": np.linspace(T.min() - 30, T.max() + 30, 1000),
        "random": np.sort(rng.random(1000)) * (T[-1] - T[0]) * 2 + (T[0] - T[-1] / 2),
    }


EDGE = np.sort(np.concatenate([[T[0] - 5, T[0] - 1e-3, T[0]], np.linspace(T[3], T[4], 40), T[10:13], T[10:11],
                               [0.5 * (T[20] + T[21])] * 3, [T[-1], T[-1] + 1e-3, T[-1] + 40]]))


@pytest.fixture(scope="module")
def pb():
    import pioran_b200
    return pioran_b200


@pytest.fixture(scope="module")
def ctx(pb):
    return pb.get_context(0)


def dense_var(a, b, c, d, t, s2, tau):
    K = pm.kernel(a, b, c, d, t[:, None] - t[None, :]) + np.diag(s2)
    k = pm.kernel(a, b, c, d, tau[:, None] - t[None, :])
    return np.sum(a) - np.einsum("mn,nm->m", k, cho_solve(cho_factor(K, lower=True), k.T))


def _batch(basis, J, B, seed):
    """B coefficient sets of the reference's approximation (tests/test_posterior.py::_theta_batch), with per-set ν and μ."""
    rng = np.random.default_rng(seed)
    a1 = rng.uniform(0.0, 1.2, B)
    th = np.stack([a1, 10 ** rng.uniform(-2.5, -1.0, B), a1 + rng.uniform(0.5, 2.5, B)], axis=1)
    mu, nu = rng.normal(Y.mean(), 0.3, B), rng.uniform(0.5, 2.0, B)
    co = [orc.approx("SBPL", list(th[i]), F0, FM, J, VAR * rng.uniform(0.5, 2.0), basis=basis) for i in range(B)]
    a, b, c, d = (np.stack([x[k] for x in co]) for k in range(4))
    return a, b, c, d, mu, nu


def _explicit(n_complex, n_real, B, seed):
    rng = np.random.default_rng(seed)
    Jt = n_complex + n_real
    a = rng.uniform(0.2, 1.0, (B, Jt)); b = rng.uniform(-0.1, 0.1, (B, Jt))
    c = 10 ** rng.uniform(-2.5, 0.0, (B, Jt)); d = c * rng.uniform(0.0, 1.5, (B, Jt))
    b[:, n_complex:] = 0.0; d[:, n_complex:] = 0.0
    return a, b, c, d


def _check_dense(got, a, b, c, d, nu, tau, what):
    for i in range(a.shape[0]):
        want = dense_var(a[i], b[i], c[i], d[i], T, nu[i] * S2, tau)
        err = np.max(np.abs(got[i] - want)) / np.sum(a[i])
        assert err <= TOL, f"{what}, set {i}: {err:.2e}"


@pytest.mark.parametrize("basis", ["SHO", "DRWCelerite"])
def test_var_matches_dense_on_the_posterior_grids(ctx, basis):
    a, b, c, d, mu, nu = _batch(basis, 20, 12, 11)
    ser = ctx.upload_series(T, Y, S2)
    try:
        R = 40 if basis == "SHO" else 60
        for name, tau in list(grids().items()) + [("edge points", EDGE)]:
            mean, var = ctx.celerite_predict_var(ser, a, b, c, d, tau, mu=mu, nu=nu)
            assert ctx.last_kernel_name() == f"postvar<{(R + 15) // 16}>"
            _check_dense(var, a, b, c, d, nu, tau, f"{basis}, {name}")
            assert np.array_equal(mean, ctx.celerite_predict(ser, a, b, c, d, tau, mu=mu, nu=nu)), name
    finally:
        ser.free()


@pytest.mark.parametrize("basis,J", [("SHO", 40), ("DRWCelerite", 30), ("DRWCelerite", 40)])   # test_posterior.WIDE_CASES
def test_var_wide_ranks(ctx, basis, J):
    a, b, c, d, mu, nu = _batch(basis, J, 5, 17)
    ser = ctx.upload_series(T, Y, S2)
    try:
        for name, tau in grids().items():
            mean, var = ctx.celerite_predict_var(ser, a, b, c, d, tau, mu=mu, nu=nu)
            _check_dense(var, a, b, c, d, nu, tau, f"{basis} J={J}, {name}")
            assert np.array_equal(mean, ctx.celerite_predict(ser, a, b, c, d, tau, mu=mu, nu=nu)), name
    finally:
        ser.free()


def test_rank_128_mixed_terms_and_rank_129_refused(pb, ctx):
    a, b, c, d = _explicit(60, 8, 3, 5)                                 # rank 2·60 + 8 = 128
    nu = np.array([1.0, 0.7, 1.9])
    ser = ctx.upload_series(T, Y, S2)
    try:
        tau = grids()["random"]
        var = ctx.celerite_predict_var(ser, a, b, c, d, tau, nu=nu, return_mean=False)
        _check_dense(var, a, b, c, d, nu, tau, "rank 128")
        assert ctx.last_kernel_name() == "postvar<8>"
        a, b, c, d = _explicit(64, 1, 2, 6)                             # rank 129
        with pytest.raises(pb.PioranError) as e:
            ctx.celerite_predict_var(ser, a, b, c, d, tau)
        assert e.value.code == -5
    finally:
        ser.free()


def test_edge_points_and_shortest_series(ctx):
    a, b, c, d, mu, nu = _batch("SHO", 20, 3, 3)
    ser = ctx.upload_series(T, Y, S2)
    try:
        var = ctx.celerite_predict_var(ser, a, b, c, d, EDGE, nu=nu, return_mean=False)
        _check_dense(var, a, b, c, d, nu, EDGE, "edge points")
        far = ctx.celerite_predict_var(ser, a, b, c, d, [T[-1] + 1e7], nu=nu, return_mean=False)   # M = 1, beyond t_N
        assert np.allclose(far[:, 0], a.sum(axis=1), rtol=1e-12, atol=0)
        one = ctx.celerite_predict_var(ser, a, b, c, d, EDGE[5:6], nu=nu, return_mean=False)        # M = 1 in a gap
        assert np.all(np.abs(one[:, 0] - var[:, 5]) <= 1e-13 * a.sum(axis=1))
    finally:
        ser.free()
    ae, be, ce, de = _explicit(3, 2, 2, 8)
    for N in (1, 2):
        t, y, s2 = np.array([3.0, 4.5])[:N], np.array([0.3, -0.2])[:N], np.array([0.02, 0.03])[:N]
        tau = np.array([1.0, 3.0, 3.0, 3.7, 4.5, 9.0])
        ser = ctx.upload_series(t, y, s2)
        try:
            var = ctx.celerite_predict_var(ser, ae, be, ce, de, tau, return_mean=False)
        finally:
            ser.free()
        for i in range(2):
            want = pm.predict_var(ae[i], be[i], ce[i], de[i], t, s2, tau)
            assert np.max(np.abs(var[i] - want)) <= TOL * ae[i].sum(), f"N={N}"


def test_mean_is_predict_and_var_ignores_mu(ctx):
    a, b, c, d, mu, nu = _batch("DRWCelerite", 20, 6, 21)
    tau = grids()["fine grid"]
    ser = ctx.upload_series(T, Y, S2)
    try:
        m1, v1 = ctx.celerite_predict_var(ser, a, b, c, d, tau, mu=mu, nu=nu)
        m2, v2 = ctx.celerite_predict_var(ser, a, b, c, d, tau, mu=mu + 0.8, nu=nu)
        v3 = ctx.celerite_predict_var(ser, a, b, c, d, tau, nu=nu, return_mean=False)
        assert np.array_equal(m1, ctx.celerite_predict(ser, a, b, c, d, tau, mu=mu, nu=nu))
        assert np.array_equal(m2, ctx.celerite_predict(ser, a, b, c, d, tau, mu=mu + 0.8, nu=nu))
        assert np.array_equal(v1, v2) and np.array_equal(v1, v3)
    finally:
        ser.free()


def test_non_positive_definite_set_gets_a_nan_row(ctx):
    a, b, c, d, mu, nu = _batch("SHO", 20, 5, 31)
    a[2] = -a[2]                                  # Σa < 0: the first pivot is negative
    tau = grids()["random"]
    ser = ctx.upload_series(T, Y, S2)
    try:
        var = ctx.celerite_predict_var(ser, a, b, c, d, tau, nu=nu, return_mean=False)
        keep = [0, 1, 3, 4]
        ref = ctx.celerite_predict_var(ser, a[keep], b[keep], c[keep], d[keep], tau, nu=nu[keep], return_mean=False)
    finally:
        ser.free()
    assert np.all(np.isnan(var[2]))
    assert np.array_equal(var[keep], ref)


def test_long_series_is_chunked_and_matches_single_set_calls(ctx):
    """N = 1e5 at rank 40: a set needs ≈ 34 MB of workspace, so 70 sets run as three θ-chunks of at most 1 GiB."""
    rng = np.random.default_rng(2)
    N = 100_000
    t = np.cumsum(rng.uniform(0.5, 1.5, N))
    s2 = rng.uniform(0.01, 0.05, N)
    y = rng.normal(size=N)
    B = 70
    co = [orc.approx("SBPL", [0.8, 10 ** rng.uniform(-4, -3), 3.0], 1 / (t[-1] - t[0]), 0.5, 20, 1.0, basis="SHO")
          for _ in range(B)]
    a, b, c, d = (np.stack([x[k] for x in co]) for k in range(4))
    nu = rng.uniform(0.5, 2.0, B)
    tau = np.sort(rng.uniform(t[0] - 10, t[-1] + 10, 1000))
    ser = ctx.upload_series(t, y, s2)
    try:
        mean, var = ctx.celerite_predict_var(ser, a, b, c, d, tau, nu=nu)
        for i in (0, 33, 69):
            m1, v1 = ctx.celerite_predict_var(ser, a[i:i + 1], b[i:i + 1], c[i:i + 1], d[i:i + 1], tau, nu=nu[i:i + 1])
            assert np.array_equal(v1[0], var[i]) and np.array_equal(m1[0], mean[i]), i
    finally:
        ser.free()
    assert np.all(np.isfinite(var))
    assert np.all(var >= -1e-9 * a.sum(axis=1)[:, None]) and np.all(var <= a.sum(axis=1)[:, None] * (1 + 1e-12))


def test_python_interface(pb):
    a, b, c, d = orc.approx("SBPL", [0.82, 0.01, 3.3], F0, FM, 20, VAR, basis="SHO")
    cov = pb.SumOfCelerite(a, b, c, d)
    tau = EDGE
    want = dense_var(a, b, c, d, T, S2, tau)
    f = pb.ScalableGP(0.7, cov)
    fp = pb.posterior(f(T, S2), Y)
    v = pb.var(fp, tau)
    assert np.max(np.abs(v - want)) <= TOL * np.sum(a)
    assert np.array_equal(pb.std(fp, tau), np.sqrt(np.maximum(v, 0.0)))
    m, v2 = pb.mean_and_var(fp, tau)
    assert np.array_equal(v2, v)
    assert np.array_equal(m, pb.mean(fp, tau))
    assert np.max(np.abs(pb.var(fp) - dense_var(a, b, c, d, T, S2, T))) <= TOL * np.sum(a)   # default τ: the data times
    # a custom mean shifts the mean only
    g = pb.ScalableGP(pb.CustomMean(lambda x: 0.1 * np.sin(x)), cov)
    gp = pb.posterior(g(T, S2), Y)
    mg, vg = pb.mean_and_var(gp, tau)
    assert np.array_equal(vg, v)
    assert np.array_equal(mg, pb.mean(gp, tau))
    # near-noiseless data: the variance at the data times is at rounding level, and std stays finite wherever var is
    tiny = pb.posterior(f(T, S2 * 1e-8), Y)
    vt, st = pb.var(tiny, T), pb.std(tiny, T)
    assert np.array_equal(np.isfinite(vt), np.isfinite(st)) and np.all(st[np.isfinite(st)] >= 0.0)


def test_argument_checks(ctx):
    a, b, c, d = _explicit(3, 1, 2, 4)
    tau = np.linspace(T[0], T[-1], 20)
    ser = ctx.upload_series(T, Y, S2)
    dp = C.POINTER(C.c_double)
    p = lambda x: x.ctypes.data_as(dp) if x is not None else None
    mean, var = np.empty((2, 20)), np.empty((2, 20))
    lib = ctx.lib
    call = lambda sid, B, M, tv, vout: lib.pioran_celerite_predict_var(ctx.h, sid, B, a.shape[1], p(a), p(b), p(c), p(d),
                                                                       None, None, M, p(tv), p(mean), vout)
    try:
        assert call(ser.id, 2, 20, tau, None) == -1                  # no var_out
        assert call(ser.id, 0, 20, tau, p(var)) == -1                # B = 0
        assert call(ser.id, 2, 0, tau, p(var)) == -1                 # M = 0
        assert call(ser.id, 2, 20, tau[::-1].copy(), p(var)) == -1   # descending τ
        assert call(ser.id + 1000, 2, 20, tau, p(var)) == -1         # unknown series
        assert lib.pioran_celerite_predict_var(ctx.h, ser.id, 2, a.shape[1], None, p(b), p(c), p(d), None, None, 20,
                                               p(tau), None, p(var)) == -1
        assert call(ser.id, 2, 20, tau, p(var)) == 0
        _check_dense(var, a, b, c, d, np.ones(2), tau, "explicit")
    finally:
        ser.free()
