"""K8 (csrc/postcov.cuh): the full posterior covariance of the celerite GP through the C ABI and the Python interface, against
the dense K_ττ − K_τt (K + diag νσ²)⁻¹ K_tτ solved with a Cholesky factor in the test (an 80-bit solve where the FP64 one is
itself off), on the series and prediction grids of tests/test_posterior.py; plus its agreement with predict_var (diagonal),
predict (mean, bit for bit) and the sample covariance of K7 draws, exact symmetry, the NaN matrix of a non-positive-definite
set, the θ-chunk and column-range paths, device groups, the rank limit and the argument checks."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

from conftest import GOLDEN
from oracle import oracle as orc

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "tools", "proto"))
import postcov_math as cm  # noqa: E402

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


def _check_dense(got, a, b, c, d, nu, tau, what, t=T, s2=S2):
    for i in range(a.shape[0]):
        assert np.array_equal(got[i], got[i].T), f"{what}, set {i}: not exactly symmetric"
        err, ld = cm.conditioned_error(got[i], a[i], b[i], c[i], d[i], t, nu[i] * s2, tau, TOL)
        if ld is not None:   # ill-conditioned: at least as close to the 80-bit covariance as the FP64 dense route
            assert ld[0] <= max(TOL, ld[1]), f"{what}, set {i}: {err:.2e}; 80-bit: {ld[0]:.2e} against {ld[1]:.2e}"


@pytest.mark.parametrize("basis", ["SHO", "DRWCelerite"])
def test_cov_matches_dense_on_the_posterior_grids(ctx, basis):
    a, b, c, d, mu, nu = _batch(basis, 20, 6, 11)
    R = 40 if basis == "SHO" else 60
    ser = ctx.upload_series(T, Y, S2)
    try:
        for name, tau in list(grids().items()) + [("edge points", EDGE)]:
            mean, cov = ctx.celerite_predict_cov(ser, a, b, c, d, tau, mu=mu, nu=nu)
            assert ctx.last_kernel_name() == f"postcov<{1 if R <= 32 else 2 if R <= 64 else 4}>"
            _check_dense(cov, a, b, c, d, nu, tau, f"{basis}, {name}")
            assert np.array_equal(mean, ctx.celerite_predict(ser, a, b, c, d, tau, mu=mu, nu=nu)), name
            var = ctx.celerite_predict_var(ser, a, b, c, d, tau, mu=mu, nu=nu, return_mean=False)
            diag = np.diagonal(cov, axis1=1, axis2=2)
            assert np.all(np.abs(diag - var) <= TOL * a.sum(axis=1)[:, None]), name
    finally:
        ser.free()


@pytest.mark.parametrize("basis,J", [("SHO", 40), ("DRWCelerite", 30), ("DRWCelerite", 40)])   # test_posterior.WIDE_CASES
def test_cov_wide_ranks(ctx, basis, J):
    a, b, c, d, mu, nu = _batch(basis, J, 3, 17)
    ser = ctx.upload_series(T, Y, S2)
    try:
        for name in ("fine grid", "random"):
            tau = grids()[name]
            cov = ctx.celerite_predict_cov(ser, a, b, c, d, tau, mu=mu, nu=nu, return_mean=False)
            _check_dense(cov, a, b, c, d, nu, tau, f"{basis} J={J}, {name}")
    finally:
        ser.free()


def test_rank_128_mixed_terms_and_rank_129_refused(pb, ctx):
    a, b, c, d = _explicit(60, 8, 3, 5)                                 # rank 2·60 + 8 = 128
    nu = np.array([1.0, 0.7, 1.9])
    ser = ctx.upload_series(T, Y, S2)
    try:
        tau = grids()["random"]
        cov = ctx.celerite_predict_cov(ser, a, b, c, d, tau, nu=nu, return_mean=False)
        _check_dense(cov, a, b, c, d, nu, tau, "rank 128")
        assert ctx.last_kernel_name() == "postcov<4>"
        a, b, c, d = _explicit(64, 1, 2, 6)                             # rank 129
        with pytest.raises(pb.PioranError) as e:
            ctx.celerite_predict_cov(ser, a, b, c, d, tau)
        assert e.value.code == -5
    finally:
        ser.free()


def test_edge_points_shortest_series_and_single_point(ctx):
    a, b, c, d, mu, nu = _batch("SHO", 20, 3, 3)
    ser = ctx.upload_series(T, Y, S2)
    try:
        cov = ctx.celerite_predict_cov(ser, a, b, c, d, EDGE, nu=nu, return_mean=False)
        _check_dense(cov, a, b, c, d, nu, EDGE, "edge points")
        for k in (0, 5, len(EDGE) - 1):                                  # M = 1: before, inside and after the data
            one = ctx.celerite_predict_cov(ser, a, b, c, d, EDGE[k:k + 1], nu=nu, return_mean=False)
            assert one.shape == (3, 1, 1)
            assert np.all(np.abs(one[:, 0, 0] - cov[:, k, k]) <= 1e-13 * a.sum(axis=1)), k
    finally:
        ser.free()
    ae, be, ce, de = _explicit(3, 2, 2, 8)
    for N in (1, 2):
        t, y, s2 = np.array([3.0, 4.5])[:N], np.array([0.3, -0.2])[:N], np.array([0.02, 0.03])[:N]
        tau = np.array([1.0, 3.0, 3.0, 3.7, 4.5, 9.0])
        ser = ctx.upload_series(t, y, s2)
        try:
            cov = ctx.celerite_predict_cov(ser, ae, be, ce, de, tau, return_mean=False)
        finally:
            ser.free()
        _check_dense(cov, ae, be, ce, de, np.ones(2), tau, f"N={N}", t=t, s2=s2)


def test_mean_is_predict_and_cov_ignores_mu(ctx):
    a, b, c, d, mu, nu = _batch("DRWCelerite", 20, 4, 21)
    tau = grids()["fine grid"]
    ser = ctx.upload_series(T, Y, S2)
    try:
        m1, c1 = ctx.celerite_predict_cov(ser, a, b, c, d, tau, mu=mu, nu=nu)
        m2, c2 = ctx.celerite_predict_cov(ser, a, b, c, d, tau, mu=mu + 0.8, nu=nu)
        c3 = ctx.celerite_predict_cov(ser, a, b, c, d, tau, nu=nu, return_mean=False)
        assert np.array_equal(m1, ctx.celerite_predict(ser, a, b, c, d, tau, mu=mu, nu=nu))
        assert np.array_equal(m2, ctx.celerite_predict(ser, a, b, c, d, tau, mu=mu + 0.8, nu=nu))
        assert np.array_equal(c1, c2) and np.array_equal(c1, c3)
    finally:
        ser.free()


def test_sample_covariance_of_posterior_draws(ctx):
    """8 192 K7 draws of fp(τ, σ²_τ): their sample covariance against K8 + σ²_τ·I, entry by entry within 6 standard errors
    of a Wishart estimate, Var(Ĉ_ij) ≈ (C_ij² + C_ii C_jj) / S."""
    a, b, c, d, mu, nu = _batch("SHO", 20, 1, 41)
    tau = np.linspace(T[100], T[140], 48)
    s2tau = 1e-4 * a.sum()
    S = 8192
    q = np.random.default_rng(5).standard_normal((1, S, len(T) + len(tau)))
    ser = ctx.upload_series(T, Y, S2)
    try:
        draws = ctx.celerite_posterior_draws(ser, a, b, c, d, tau, q, mu=mu, nu=nu, sigma2_tau=s2tau)[0]
        cov = ctx.celerite_predict_cov(ser, a, b, c, d, tau, mu=mu, nu=nu, return_mean=False)[0]
    finally:
        ser.free()
    want = cov + s2tau * np.eye(len(tau))
    got = np.cov(draws, rowvar=False)
    se = np.sqrt((want ** 2 + np.outer(np.diag(want), np.diag(want))) / S)
    z = np.abs(got - want) / se
    assert z.max() <= 6.0, f"largest deviation {z.max():.1f} standard errors"


def test_non_positive_definite_set_gets_a_nan_matrix(ctx):
    a, b, c, d, mu, nu = _batch("SHO", 20, 5, 31)
    a[2] = -a[2]                                  # Σa < 0: the first pivot is negative
    tau = grids()["random"]
    ser = ctx.upload_series(T, Y, S2)
    try:
        cov = ctx.celerite_predict_cov(ser, a, b, c, d, tau, nu=nu, return_mean=False)
        keep = [0, 1, 3, 4]
        ref = ctx.celerite_predict_cov(ser, a[keep], b[keep], c[keep], d[keep], tau, nu=nu[keep], return_mean=False)
    finally:
        ser.free()
    assert np.all(np.isnan(cov[2]))
    assert np.array_equal(cov[keep], ref)


def _cap(N, M, R, sets=0.0, cols=0):
    """A workspace cap that holds `sets` whole sets, or one set's workspace and `cols` columns of rows and mirror rows."""
    ws = 8 * (N * 128 + 2 * N + M * (3 * R + 3))   # 128: at least the leading dimension of the stored factor
    return int(sets * (ws + 8 * M * M)) if sets else ws + 8 * 2 * cols * M


def test_theta_chunks_and_column_ranges_are_bit_equal(ctx):
    a, b, c, d, mu, nu = _batch("DRWCelerite", 20, 5, 13)
    tau = grids()["beyond the data"]
    M = len(tau)
    ser = ctx.upload_series(T, Y, S2)
    try:
        m0, c0 = ctx.celerite_predict_cov(ser, a, b, c, d, tau, mu=mu, nu=nu)
        n0 = ctx.launch_count
        for cap in (_cap(len(T), M, 60, sets=2.5), _cap(len(T), M, 60, cols=300), _cap(len(T), M, 60, cols=7)):
            ctx.set_postcov_workspace(cap)
            m1, c1 = ctx.celerite_predict_cov(ser, a, b, c, d, tau, mu=mu, nu=nu)
            assert np.array_equal(m1, m0) and np.array_equal(c1, c0), cap
        assert ctx.launch_count - n0 > 3 * 5 * 4    # the column ranges ran as more launches
    finally:
        ctx.set_postcov_workspace(0)
        ser.free()


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
    s1, sg = ctx.upload_series(T, Y, S2), grp.upload_series(T, Y, S2)
    try:
        one = ctx.celerite_predict_cov(s1, a, b, c, d, tau, mu=mu, nu=nu)
        two = grp.celerite_predict_cov(sg, a, b, c, d, tau, mu=mu, nu=nu)
        assert np.array_equal(one[0], two[0]) and np.array_equal(one[1], two[1])
        # the workspace cap reaches every child: column ranges on each device, as many launches as on one device
        cap = _cap(len(T), len(tau), 40, cols=200)
        ctx.set_postcov_workspace(cap); grp.set_postcov_workspace(cap)
        n1, ng = ctx.launch_count, grp.launch_count
        one_c = ctx.celerite_predict_cov(s1, a, b, c, d, tau, mu=mu, nu=nu)
        two_c = grp.celerite_predict_cov(sg, a, b, c, d, tau, mu=mu, nu=nu)
        assert ctx.launch_count - n1 == grp.launch_count - ng
        assert np.array_equal(one_c[1], one[1]) and np.array_equal(two_c[1], one[1])
    finally:
        ctx.set_postcov_workspace(0)
        s1.free(); sg.free()


def test_python_interface(pb):
    a, b, c, d = orc.approx("SBPL", [0.82, 0.01, 3.3], F0, FM, 20, VAR, basis="SHO")
    kern = pb.SumOfCelerite(a, b, c, d)
    tau = EDGE
    want = cm.dense_cov(*(np.asarray(x) for x in (a, b, c, d)), T, S2, tau)
    f = pb.ScalableGP(0.7, kern)
    fp = pb.posterior(f(T, S2), Y)
    C_ = pb.cov(fp, tau)
    assert C_.shape == (len(tau), len(tau)) and np.max(np.abs(C_ - want)) <= TOL * np.sum(a)
    m, C2 = pb.mean_and_cov(fp, tau)
    assert np.array_equal(C2, C_)
    assert np.array_equal(m, pb.mean(fp, tau))
    assert np.max(np.abs(np.diag(C_) - pb.var(fp, tau))) <= TOL * np.sum(a)
    assert np.max(np.abs(pb.cov(fp) - cm.dense_cov(*(np.asarray(x) for x in (a, b, c, d)), T, S2, T))) <= TOL * np.sum(a)
    # a custom mean shifts the mean only
    g = pb.ScalableGP(pb.CustomMean(lambda x: 0.1 * np.sin(x)), kern)
    gp = pb.posterior(g(T, S2), Y)
    mg, cg = pb.mean_and_cov(gp, tau)
    assert np.array_equal(cg, C_)
    assert np.array_equal(mg, pb.mean(gp, tau))
    assert np.array_equal(pb.predict_cov(kern, tau, T, S2), C_)


def test_argument_checks(ctx):
    a, b, c, d = _explicit(3, 1, 2, 4)
    tau = np.linspace(T[0], T[-1], 20)
    ser = ctx.upload_series(T, Y, S2)
    dp = C.POINTER(C.c_double)
    p = lambda x: x.ctypes.data_as(dp) if x is not None else None
    mean, cov = np.empty((2, 20)), np.empty((2, 20, 20))
    lib = ctx.lib
    call = lambda sid, B, M, tv, cout: lib.pioran_celerite_predict_cov(ctx.h, sid, B, a.shape[1], p(a), p(b), p(c), p(d),
                                                                       None, None, M, p(tv), p(mean), cout)
    try:
        assert call(ser.id, 2, 20, tau, None) == -1                  # no cov_out
        assert call(ser.id, 0, 20, tau, p(cov)) == -1                # B = 0
        assert call(ser.id, 2, 0, tau, p(cov)) == -1                 # M = 0
        assert call(ser.id, 2, 20, tau[::-1].copy(), p(cov)) == -1   # descending τ
        assert call(ser.id + 1000, 2, 20, tau, p(cov)) == -1         # unknown series
        assert lib.pioran_celerite_predict_cov(ctx.h, ser.id, 2, a.shape[1], None, p(b), p(c), p(d), None, None, 20,
                                               p(tau), None, p(cov)) == -1
        assert lib.pioran_ctx_set_postcov_workspace(ctx.h, -1) == -1
        assert call(ser.id, 2, 20, tau, p(cov)) == 0
        _check_dense(cov, a, b, c, d, np.ones(2), tau, "explicit")
    finally:
        ser.free()
