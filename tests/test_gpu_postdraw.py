"""K7 (csrc/postdraw.cuh): draws from the posterior of the celerite GP by Matheron's rule, through the C ABI and the Python
interface.  Same q: against the oracle composition of the reference's routines on the merged grid G of t and τ,
    u = sim(a, b, c, d, G, noise_G, q),   draw = μ + u(τ) + pred(a, b, c, d, τ, t, ỹ − μ − u(t), ν σ²),
on the series and grids of tests/test_posterior.py.  Many q: the sample mean, variance and covariance against predict,
predict_var and the dense posterior covariance.  Plus edge cases, the NaN block of a non-positive-definite set, a custom
mean, θ-chunking, launch amortisation over draws, device groups and the argument checks."""
import ctypes as C
import os
import sys

import numpy as np
import pytest
from scipy.linalg import cho_factor, cho_solve

from conftest import GOLDEN, periodic_mean
from oracle import oracle as orc

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "tools", "proto"))
import postdraw_math as dm  # noqa: E402
import postvar_math as pm  # noqa: E402

pytestmark = pytest.mark.gpu

A = np.loadtxt(os.path.join(GOLDEN, "simu.txt"))
T, Y, YERR = (np.ascontiguousarray(c) for c in A.T)
S2 = YERR ** 2
F0 = 1 / (T[-1] - T[0]) / 100
FM = 1 / np.min(np.diff(T)) / 2 * 20
VAR = np.var(Y, ddof=1)
TOL = 1e-9   # of √Σa


def grids():   # tests/test_posterior.py::grids
    rng = np.random.default_rng(7)
    return {
        "data times": T,
        "fine grid": np.linspace(T.min(), T.max(), 1000),
        "beyond the data": np.linspace(T.min() - 30, T.max() + 30, 1000),
        "random": np.sort(rng.random(1000)) * (T[-1] - T[0]) * 2 + (T[0] - T[-1] / 2),
    }


EDGE = np.sort(np.concatenate([[T[0] - 5, T[0] - 1e-3, T[0]], np.linspace(T[3], T[4], 40), T[10:13], T[10:11],
                               [0.5 * (T[20] + T[21])] * 3, [T[-1], T[-1] + 1e-3, T[-1] + 40]]))   # test_gpu_postvar.EDGE


@pytest.fixture(scope="module")
def pb():
    import pioran_b200
    return pioran_b200


@pytest.fixture(scope="module")
def ctx(pb):
    return pb.get_context(0)


def _batch(basis, J, B, seed):   # test_gpu_postvar._batch
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


def _q(B, S, NG, seed):
    return np.random.default_rng(seed).standard_normal((B, S, NG))


def oracle_draws(a, b, c, d, t, y, s2, tau, q, mu, sigma2_tau):
    """The reference-order composition for one set: sim on G, then pred of the residual at the data."""
    G, code = dm.merged_grid(t, tau)
    noise = np.where(code >= 0, s2[np.maximum(code, 0)], sigma2_tau)
    dat, pre = np.flatnonzero(code >= 0), np.flatnonzero(code < 0)
    dat, pre = dat[np.argsort(code[dat])], pre[np.argsort(-code[pre] - 1)]
    out = []
    for qs in np.atleast_2d(q):
        u = orc.celerite_simulate(a, b, c, d, G, noise, qs)
        out.append(mu + u[pre] + orc.celerite_predict(a, b, c, d, tau, t, y - mu - u[dat], s2))
    return np.array(out)


def _check_oracle(got, a, b, c, d, mu, nu, tau, q, what, sigma2_tau=1e-18, t=T, y=Y, s2=S2):
    """≤ TOL·√Σa from the oracle composition, or conditioning: prediction points closer together than the data's
    resolution with σ²_τ = 1e-18 leave pivots of the merged factor near rounding level, and then two correct FP64 routes
    differ.  Such a set must be no farther from the oracle than 4× the distance between the oracle and the dense draw."""
    for i in range(a.shape[0]):
        want = oracle_draws(a[i], b[i], c[i], d[i], t, y, nu[i] * s2, tau, q[i], mu[i], sigma2_tau)
        sa = np.sqrt(np.sum(a[i]))
        err = np.max(np.abs(got[i] - want)) / sa
        if err > TOL:
            dense = dm.dense_draws(a[i], b[i], c[i], d[i], t, y, nu[i] * s2, tau, q[i], mu[i], sigma2_tau)
            e_ref = np.max(np.abs(want - dense)) / sa
            assert e_ref > TOL / 4 and err <= 4 * e_ref, f"{what}, set {i}: {err:.2e} from the oracle, which is {e_ref:.2e} from the dense draw"


@pytest.mark.parametrize("basis", ["SHO", "DRWCelerite"])
def test_draws_match_the_oracle_on_the_posterior_grids(ctx, basis):
    a, b, c, d, mu, nu = _batch(basis, 20, 12, 11)
    R = 40 if basis == "SHO" else 60
    ser = ctx.upload_series(T, Y, S2)
    try:
        cases = [(name, tau, 1e-18) for name, tau in grids().items()]
        cases.append(("edge points", EDGE, 1e-8 * float(np.min(a.sum(axis=1)))))   # repeated τ: σ²_τ > 0
        for k, (name, tau, s2t) in enumerate(cases):
            q = _q(12, 3, len(T) + len(tau), 100 + k)
            got = ctx.celerite_posterior_draws(ser, a, b, c, d, tau, q, mu=mu, nu=nu, sigma2_tau=s2t)
            assert got.shape == (12, 3, len(tau))
            assert ctx.last_kernel_name() == f"postdraw<{1 if R <= 32 else 2 if R <= 64 else 4}>"
            _check_oracle(got, a, b, c, d, mu, nu, tau, q, f"{basis}, {name}", sigma2_tau=s2t)
    finally:
        ser.free()


@pytest.mark.parametrize("basis,J", [("SHO", 40), ("DRWCelerite", 30), ("DRWCelerite", 40)])
def test_draws_wide_ranks(ctx, basis, J):
    a, b, c, d, mu, nu = _batch(basis, J, 4, 17)
    ser = ctx.upload_series(T, Y, S2)
    try:
        for k, (name, tau) in enumerate(grids().items()):
            q = _q(4, 2, len(T) + len(tau), 200 + k)
            got = ctx.celerite_posterior_draws(ser, a, b, c, d, tau, q, mu=mu, nu=nu)
            assert ctx.last_kernel_name() == "postdraw<4>"
            _check_oracle(got, a, b, c, d, mu, nu, tau, q, f"{basis} J={J}, {name}")
    finally:
        ser.free()


def test_rank_128_mixed_terms_and_rank_129_refused(pb, ctx):
    a, b, c, d = _explicit(60, 8, 3, 5)                                 # rank 2·60 + 8 = 128
    mu, nu = np.array([0.1, -0.2, 0.0]), np.array([1.0, 0.7, 1.9])
    tau = grids()["random"]
    q = _q(3, 2, len(T) + len(tau), 5)
    ser = ctx.upload_series(T, Y, S2)
    try:
        got = ctx.celerite_posterior_draws(ser, a, b, c, d, tau, q, mu=mu, nu=nu)
        _check_oracle(got, a, b, c, d, mu, nu, tau, q, "rank 128")
        assert ctx.last_kernel_name() == "postdraw<4>"
        a, b, c, d = _explicit(64, 1, 2, 6)                             # rank 129
        with pytest.raises(pb.PioranError) as e:
            ctx.celerite_posterior_draws(ser, a, b, c, d, tau, q[:2])
        assert e.value.code == -5
    finally:
        ser.free()


def test_sample_statistics_match_predict_predict_var_and_the_dense_covariance(ctx):
    a, b, c, d = (x[None] for x in orc.approx("SBPL", [0.82, 0.01, 3.3], F0, FM, 20, VAR, basis="SHO"))
    tau = grids()["fine grid"]
    S, M = 8192, len(tau)
    s2t = 1e-18
    q = _q(1, S, len(T) + M, 12345)
    ser = ctx.upload_series(T, Y, S2)
    try:
        draws = ctx.celerite_posterior_draws(ser, a, b, c, d, tau, q, mu=[0.4])[0]
        mean, var = ctx.celerite_predict_var(ser, a, b, c, d, tau, mu=[0.4])
    finally:
        ser.free()
    mean, var = mean[0], var[0] + s2t
    suma = float(a.sum())
    m_hat, v_hat = draws.mean(axis=0), draws.var(axis=0, ddof=1)
    se = np.sqrt(np.maximum(var, 0.0) / S)
    assert np.all(np.abs(m_hat - mean) <= 5 * se + 1e-12 * np.sqrt(suma))
    floor = 1e-6 * suma   # points where the variance is near 0 (next to precise data)
    assert np.all(np.abs(v_hat - var) <= 6 * np.sqrt(2 / S) * var + floor)
    # the covariance of fixed point pairs against the dense posterior covariance
    K = pm.kernel(a[0], b[0], c[0], d[0], T[:, None] - T[None, :]) + np.diag(S2)
    ks = pm.kernel(a[0], b[0], c[0], d[0], tau[:, None] - T[None, :])
    pairs = [(0, 1), (100, 103), (400, 460), (700, 999), (250, 251)]
    idx = sorted({i for p in pairs for i in p})
    kf = cho_factor(K, lower=True)
    sub = ks[idx]
    cov = pm.kernel(a[0], b[0], c[0], d[0], tau[idx][:, None] - tau[idx][None, :]) - sub @ cho_solve(kf, sub.T)
    at = {i: k for k, i in enumerate(idx)}
    for i, j in pairs:
        cij, cii, cjj = cov[at[i], at[j]], cov[at[i], at[i]], cov[at[j], at[j]]
        got = np.cov(draws[:, i], draws[:, j])[0, 1]
        se_c = np.sqrt((cii * cjj + cij ** 2) / S)
        assert abs(got - cij) <= 5 * se_c + 1e-9 * suma, (i, j, got, cij, se_c)


def test_edge_cases(ctx):
    a, b, c, d, mu, nu = _batch("SHO", 20, 3, 3)
    ser = ctx.upload_series(T, Y, S2)
    try:
        # every τ a data time; before and after the data; a single point; a single draw
        for k, tau in enumerate([T.copy(), np.array([T[0] - 50, T[0] - 1, T[-1] + 1, T[-1] + 50]),
                                 np.array([0.5 * (T[7] + T[8])])]):
            for S in (1, 2):
                q = _q(3, S, len(T) + len(tau), 300 + k)
                got = ctx.celerite_posterior_draws(ser, a, b, c, d, tau, q, mu=mu, nu=nu)
                assert got.shape == (3, S, len(tau))
                _check_oracle(got, a, b, c, d, mu, nu, tau, q, f"case {k}, S={S}")
    finally:
        ser.free()
    ae, be, ce, de = _explicit(3, 2, 2, 8)
    one = np.ones(2)
    for N in (1, 2):
        t, y, s2 = np.array([3.0, 4.5])[:N], np.array([0.3, -0.2])[:N], np.array([0.02, 0.03])[:N]
        tau = np.array([1.0, 3.0, 3.7, 4.5, 9.0])
        q = _q(2, 3, N + len(tau), 40 + N)
        ser = ctx.upload_series(t, y, s2)
        try:
            got = ctx.celerite_posterior_draws(ser, ae, be, ce, de, tau, q)
        finally:
            ser.free()
        _check_oracle(got, ae, be, ce, de, np.zeros(2), one, tau, q, f"N={N}", t=t, y=y, s2=s2)


def test_repeated_tau_needs_noise(pb, ctx):
    a, b, c, d, mu, nu = _batch("DRWCelerite", 20, 2, 4)
    tau = np.sort(np.concatenate([np.linspace(T[2], T[9], 20), [T[5] + 0.1] * 3]))
    q = _q(2, 2, len(T) + len(tau), 9)
    ser = ctx.upload_series(T, Y, S2)
    try:
        with pytest.raises(pb.PioranError) as e:
            ctx.celerite_posterior_draws(ser, a, b, c, d, tau, q, sigma2_tau=0.0)
        assert e.value.code == -1
        s2t = 1e-6 * float(np.min(a.sum(axis=1)))
        got = ctx.celerite_posterior_draws(ser, a, b, c, d, tau, q, mu=mu, nu=nu, sigma2_tau=s2t)
        _check_oracle(got, a, b, c, d, mu, nu, tau, q, "repeated τ", sigma2_tau=s2t)
        # distinct τ with σ²_τ = 0 is allowed
        ctx.celerite_posterior_draws(ser, a, b, c, d, np.unique(tau), q[:, :, :len(T) + len(np.unique(tau))], sigma2_tau=0.0)
    finally:
        ser.free()


def test_non_positive_definite_set_gets_a_nan_block(ctx):
    a, b, c, d, mu, nu = _batch("SHO", 20, 5, 31)
    a[2] = -a[2]                                  # Σa < 0: the first pivot is negative
    tau = grids()["random"]
    q = _q(5, 3, len(T) + len(tau), 6)
    keep = [0, 1, 3, 4]
    ser = ctx.upload_series(T, Y, S2)
    try:
        got = ctx.celerite_posterior_draws(ser, a, b, c, d, tau, q, mu=mu, nu=nu)
        ref = ctx.celerite_posterior_draws(ser, a[keep], b[keep], c[keep], d[keep], tau, q[keep], mu=mu[keep], nu=nu[keep])
    finally:
        ser.free()
    assert np.all(np.isnan(got[2]))
    assert np.array_equal(got[keep], ref)


def test_custom_mean_on_the_periodic_chain(ctx, pb, golden_periodic):
    """Sinusoidal mean of the reference's periodic run: y_batch = y − m_θ(t), μ = 0, and m_θ(τ) added by the caller."""
    g = golden_periodic
    rows = g.chain[::397][:6]
    th = rows[:, 2:8]
    spec = pb.make_spec(g.model, g.f_min, g.f_max, 20)
    a, b, c, d = ctx.approx_coeffs(spec, th[:, :4])
    nu = th[:, 4]
    B, N = len(rows), len(g.t)
    yb = np.stack([g.y - periodic_mean(g.t, r) for r in rows])
    tau = np.linspace(g.t[0] - 5, g.t[-1] + 5, 700)
    q = _q(B, 2, N + len(tau), 77)
    ser = ctx.upload_series(g.t, g.y, g.s2)
    try:
        got = ctx.celerite_posterior_draws(ser, a, b, c, d, tau, q, nu=nu, y_batch=yb)
    finally:
        ser.free()
    for i in range(B):
        want = oracle_draws(a[i], b[i], c[i], d[i], g.t, yb[i], nu[i] * g.s2, tau, q[i], 0.0, 1e-18)
        assert np.max(np.abs(got[i] - want)) <= TOL * np.sqrt(np.sum(a[i])), i
        full = got[i] + periodic_mean(tau, rows[i])
        assert np.all(np.isfinite(full))


def test_long_series_is_chunked_and_matches_single_set_calls(ctx):
    """N = 1e5 at rank 40: a set with S = 2 needs ≈ 71 MB of workspace, so 40 sets run as three θ-chunks of at most 1 GiB."""
    rng = np.random.default_rng(2)
    N = 100_000
    t = np.cumsum(rng.uniform(0.5, 1.5, N))
    s2 = rng.uniform(0.01, 0.05, N)
    y = rng.normal(size=N)
    B = 40
    co = [orc.approx("SBPL", [0.8, 10 ** rng.uniform(-4, -3), 3.0], 1 / (t[-1] - t[0]), 0.5, 20, 1.0, basis="SHO")
          for _ in range(B)]
    a, b, c, d = (np.stack([x[k] for x in co]) for k in range(4))
    nu = rng.uniform(0.5, 2.0, B)
    tau = np.sort(rng.uniform(t[0] - 10, t[-1] + 10, 1000))
    q = _q(B, 2, N + len(tau), 8)
    ser = ctx.upload_series(t, y, s2)
    try:
        got = ctx.celerite_posterior_draws(ser, a, b, c, d, tau, q, nu=nu)
        for i in (0, 17, 39):
            one = ctx.celerite_posterior_draws(ser, a[i:i + 1], b[i:i + 1], c[i:i + 1], d[i:i + 1], tau, q[i:i + 1], nu=nu[i:i + 1])
            assert np.array_equal(one[0], got[i]), i
    finally:
        ser.free()
    assert np.all(np.isfinite(got))


def test_launch_count_does_not_grow_with_draws(ctx):
    a, b, c, d, mu, nu = _batch("DRWCelerite", 20, 6, 5)
    tau = grids()["fine grid"]
    ser = ctx.upload_series(T, Y, S2)
    try:
        counts = []
        for S in (1, 32):
            q = _q(6, S, len(T) + len(tau), S)
            n0 = ctx.launch_count
            ctx.celerite_posterior_draws(ser, a, b, c, d, tau, q, mu=mu, nu=nu)
            counts.append(ctx.launch_count - n0)
            assert ctx.last_kernel_name() == "postdraw<2>"
    finally:
        ser.free()
    assert counts[0] == counts[1] > 0


def _ndev():   # test_gpu_group._ndev
    try:
        rt = C.CDLL("libcudart.so")
    except OSError:
        import torch
        return torch.cuda.device_count()
    n = C.c_int(0)
    rt.cudaGetDeviceCount(C.byref(n))
    return n.value


@pytest.mark.parametrize("devices", [[0], [0, 1]])
def test_device_group_matches_single_device(pb, ctx, devices):
    if len(devices) > _ndev():
        pytest.skip("needs %d GPUs" % len(devices))
    grp = pb.Context(devices)
    a, b, c, d, mu, nu = _batch("SHO", 20, 7, 23)
    tau = grids()["random"]
    q = _q(7, 3, len(T) + len(tau), 23)
    yb = Y[None] + np.random.default_rng(3).normal(0, 0.1, (7, len(T)))
    s1, sg = ctx.upload_series(T, Y, S2), grp.upload_series(T, Y, S2)
    try:
        one = ctx.celerite_posterior_draws(s1, a, b, c, d, tau, q, mu=mu, nu=nu, y_batch=yb, sigma2_tau=1e-9)
        two = grp.celerite_posterior_draws(sg, a, b, c, d, tau, q, mu=mu, nu=nu, y_batch=yb, sigma2_tau=1e-9)
    finally:
        s1.free(); sg.free()
    assert np.array_equal(one, two)


def test_python_interface(pb, ctx):
    a, b, c, d = orc.approx("SBPL", [0.82, 0.01, 3.3], F0, FM, 20, VAR, basis="SHO")
    cov = pb.SumOfCelerite(a, b, c, d)
    tau = grids()["random"]
    NG = len(T) + len(tau)
    q = _q(1, 4, NG, 51)[0]
    ser = ctx.upload_series(T, Y - 0.7, S2)
    try:
        want = ctx.celerite_posterior_draws(ser, a, b, c, d, tau, q[None])[0] + 0.7
    finally:
        ser.free()
    fp = pb.posterior(pb.ScalableGP(0.7, cov)(T, S2), Y)
    fpx = fp(tau)
    assert isinstance(fpx, pb.FinitePosteriorGP) and fpx.σ2 == 1e-18
    got = pb.rand(fpx, q)
    assert got.shape == (4, len(tau)) and np.array_equal(got, want)
    one = pb.rand(fpx, q[0])
    assert one.shape == (len(tau),) and np.array_equal(one, want[0])
    # a custom mean: the draws are made for y − m(t), and m(τ) is added
    m = pb.CustomMean(lambda x: 0.1 * np.sin(x))
    ser = ctx.upload_series(T, Y - m(T), S2)
    try:
        want = ctx.celerite_posterior_draws(ser, a, b, c, d, tau, q[None], sigma2_tau=1e-6)[0] + m(tau)
    finally:
        ser.free()
    got = pb.rand(pb.posterior(pb.ScalableGP(m, cov)(T, S2), Y)(tau, 1e-6), q)
    assert np.array_equal(got, want)
    # rand of a prior finite GP is unchanged
    fx = pb.ScalableGP(0.7, cov)(T, S2)
    qp = np.random.default_rng(1).standard_normal(len(T))
    assert np.array_equal(pb.rand(fx, qp), pb.simulate(cov, T, S2, qp) + 0.7)


def test_argument_checks(ctx):
    a, b, c, d = _explicit(3, 1, 2, 4)
    tau = np.linspace(T[0], T[-1], 20)
    NG = len(T) + 20
    q = _q(2, 3, NG, 1)
    ser = ctx.upload_series(T, Y, S2)
    dp = C.POINTER(C.c_double)
    p = lambda x: x.ctypes.data_as(dp) if x is not None else None
    out = np.empty((2, 3, 20))
    lib = ctx.lib
    call = lambda sid=ser.id, B=2, M=20, tv=tau, s2t=1e-18, S=3, qq=p(q), o=p(out): lib.pioran_celerite_posterior_draws(
        ctx.h, sid, B, a.shape[1], p(a), p(b), p(c), p(d), None, None, None, M, p(tv), s2t, S, qq, o)
    try:
        assert call(o=None) == -1                                    # no draws_out
        assert call(qq=None) == -1                                   # no q
        assert call(B=0) == -1 and call(M=0) == -1 and call(S=0) == -1
        assert call(tv=tau[::-1].copy()) == -1                       # descending τ
        assert call(s2t=-1e-9) == -1 and call(s2t=float("nan")) == -1
        dup = tau.copy(); dup[5] = dup[4]
        assert call(tv=dup, s2t=0.0) == -1                           # repeated τ, no noise
        assert call(tv=dup, s2t=1e-9) == 0
        assert call(sid=ser.id + 1000) == -1                         # unknown series
        assert lib.pioran_celerite_posterior_draws(ctx.h, ser.id, 2, a.shape[1], None, p(b), p(c), p(d), None, None, None,
                                                   20, p(tau), 1e-18, 3, p(q), p(out)) == -1
        assert call() == 0
        _check_oracle(out, a, b, c, d, np.zeros(2), np.ones(2), tau, q, "explicit")
    finally:
        ser.free()
