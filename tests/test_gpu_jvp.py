"""K5g (csrc/jvp.cuh): forward-mode derivatives of the explicit-coefficient likelihood, and the gradient with PSD features built on
it, through the C ABI.  References: the forward-mode oracle tests/tools/oracle_jvp.c (the reference's own sweep on dual numbers,
checked against the pinned value oracle and its central differences by tests/test_oracle_jvp.py), central differences of the
GPU's own values, and the K5 gradient."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

from conftest import assert_parity, periodic_mean, rel_err, synthetic_series
from oracle import oracle as orc

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "tools"))
import oracle_jvp as oj  # noqa: E402

pytestmark = pytest.mark.gpu
RTOL = 1e-8          # the _check rule of test_gpu_grad.py
NAMES = ("da", "db", "dc", "dd", "dmu", "dnu", "dy", "ds2")


@pytest.fixture(scope="module")
def pb():
    import pioran_b200
    return pioran_b200


@pytest.fixture(scope="module")
def ctx(pb):
    return pb.get_context(0)


def _check(got, want, rtol=RTOL):
    scale = np.maximum(np.abs(want), np.abs(want).max(axis=0, keepdims=True))
    scale = np.where(scale > 0, scale, 1.0)
    err = np.abs(got - want) / scale
    assert np.all(np.isfinite(got)), "non-finite derivative"
    assert err.max() <= rtol, f"derivative parity {err.max():.3e}"
    return err.max()


def _coeffs(R, B, seed, mixed=False):
    """B positive-definite coefficient sets of rank R: SHO-form complex terms (a = b, c = d), one real term when R is odd.
    mixed: the first complex term of every set but the first is real (b = d = 0), so the batch keeps it at two rows."""
    rng = np.random.default_rng(seed)
    nc, nr = R // 2, R % 2
    Jt = nc + nr
    a = rng.uniform(0.1, 1.0, (B, Jt)) / Jt
    c = np.exp(rng.uniform(np.log(0.05), np.log(5.0), (B, Jt)))
    b, d = a.copy(), c.copy()
    b[:, nc:], d[:, nc:] = 0.0, 0.0
    if mixed and nc:
        b[1:, 0], d[1:, 0] = 0.0, 0.0
    return a, b, c, d


def _tangents(rng, B, P, Jt, N, a, c):
    s = {"da": np.abs(a).mean(), "db": np.abs(a).mean(), "dc": c.mean(), "dd": c.mean()}
    tan = {n: rng.normal(size=(B, P, Jt)) * s[n] for n in ("da", "db", "dc", "dd")}
    tan.update(dmu=rng.normal(size=(B, P)), dnu=rng.normal(size=(B, P)) * 0.3,
               dy=rng.normal(size=(B, P, N)), ds2=rng.normal(size=(B, P, N)) * 0.05)
    return tan


def _ndev():
    rt = C.CDLL("libcudart.so")
    n = C.c_int(0)
    rt.cudaGetDeviceCount(C.byref(n))
    return n.value


def _check_ld(got, want, want_ld, rtol=RTOL, slack=4.0):
    """_check, with the conditioning exemption of conftest.assert_parity for entries where the FP64 oracle itself is off its 80-bit
    twin: such an entry passes when the GPU lies within `slack` times that distance of the 80-bit value."""
    scale = np.maximum(np.abs(want_ld), np.abs(want_ld).max(axis=0, keepdims=True))
    scale = np.where(scale > 0, scale, 1.0)
    err = np.abs(got - want) / scale
    e_ref, e_gpu = np.abs(want - want_ld) / scale, np.abs(got - want_ld) / scale
    bad = (err > rtol) & ~((e_ref > rtol / slack) & (e_gpu <= slack * e_ref))
    assert np.all(np.isfinite(got)), "non-finite derivative"
    assert not bad.any(), f"derivative parity {err[bad].max():.3e} at {np.argwhere(bad)[:4].tolist()}"
    assert (err > rtol).sum() <= max(1, got.size // 50), "too many entries needed the conditioning exemption"
    return err.max()


def _ld(a, b, c, d, t, y, s2, mu, nu):
    return lambda i: orc.celerite_logl(a[i], b[i], c[i], d[i], t, y - mu[i], nu[i] * s2, long_double=True)


@pytest.mark.parametrize("N", [1, 2, 333])
@pytest.mark.parametrize("R", [2, 5, 16, 17, 32, 33, 48, 64, 65, 80, 96])
def test_jvp_vs_reference(ctx, R, N):
    rng = np.random.default_rng(R * 1000 + N)
    t = np.cumsum(rng.uniform(0.2, 1.5, N)); y = rng.normal(size=N); s2 = rng.uniform(0.2, 0.4, N)
    ser = ctx.upload_series(t, y, s2)
    B, P = 3, 7
    a, b, c, d = _coeffs(R, B, R + N, mixed=R > 4)
    mu, nu = rng.normal(0, 0.3, B), rng.uniform(0.8, 1.5, B)
    tan = _tangents(rng, B, P, a.shape[1], N, a, c)
    L, G = ctx.celerite_logl_jvp(ser, a, b, c, d, mu=mu, nu=nu, **tan)
    wl, wg = oj.celerite_logl_jvp_batch(a, b, c, d, t, y, s2, mu=mu, nu=nu, **tan)
    assert_parity(L, wl, np.arange(B), _ld(a, b, c, d, t, y, s2, mu, nu))
    assert rel_err(L, ctx.celerite_logl(ser, a, b, c, d, mu=mu, nu=nu)).max() <= 1e-9
    _check(G, wg)
    # P = 1: the first direction alone gives the first column
    L1, G1 = ctx.celerite_logl_jvp(ser, a, b, c, d, mu=mu, nu=nu, **{n: v[:, :1] for n, v in tan.items()})
    assert np.array_equal(L1, L) and np.array_equal(G1[:, 0], G[:, 0])
    ser.free()


def test_negative_coefficients_and_real_terms(ctx):
    """The rank-reduction set of test_gpu_parity.py (negative a, b, d; real terms), one direction per input."""
    rng = np.random.default_rng(3)
    N = 150
    t = np.cumsum(rng.uniform(0.2, 1.5, N)); y = rng.normal(size=N); s2 = np.full(N, 0.3)
    ser = ctx.upload_series(t, y, s2)
    a = np.array([[1.2, 0.8, -0.3, 0.5], [2.0, 0.1, -0.05, 1.0]])
    b = np.array([[0.0, 0.3, -0.1, 0.0], [0.0, -0.05, 0.02, 0.0]])
    c = np.array([[0.3, 0.2, 1.0, 2.0], [0.1, 0.5, 0.8, 3.0]])
    d = np.array([[0.0, 1.5, -2.0, 0.0], [0.0, 0.7, 1.1, 0.0]])
    B, P = 2, len(NAMES)
    full = _tangents(rng, B, 1, 4, N, a, c)
    tan = {n: np.zeros((B, P) + v.shape[2:]) for n, v in full.items()}
    for p, n in enumerate(NAMES):
        tan[n][:, p] = full[n][:, 0]
    L, G = ctx.celerite_logl_jvp(ser, a, b, c, d, **tan)
    wl, wg = oj.celerite_logl_jvp_batch(a, b, c, d, t, y, s2, **tan)
    assert rel_err(L, orc.celerite_logl_batch(a, b, c, d, t, y, s2)).max() <= 1e-9
    _check(G, wg)
    ser.free()


def test_jvp_vs_central_differences_of_gpu_values(ctx):
    rng = np.random.default_rng(5)
    N = 333
    t = np.cumsum(rng.uniform(0.2, 1.5, N)); y = rng.normal(size=N); s2 = rng.uniform(0.2, 0.4, N)
    ser = ctx.upload_series(t, y, s2)
    a, b, c, d = _coeffs(33, 1, 7)
    mu, nu = np.array([0.2]), np.array([1.1])
    tan = _tangents(rng, 1, 1, a.shape[1], N, a, c)
    _, G = ctx.celerite_logl_jvp(ser, a, b, c, d, mu=mu, nu=nu, **tan)
    h = 1e-6
    vals = []
    for e in (h, -h):
        s = lambda n, base: base + e * tan[n][:, 0]
        vals.append(ctx.celerite_logl(ser, s("da", a), s("db", b), s("dc", c), s("dd", d), mu=s("dmu", mu), nu=s("dnu", nu),
                                      y_batch=s("dy", y[None]), s2_batch=s("ds2", s2[None])))
    cd = (vals[0] - vals[1]) / (2 * h)
    assert abs(G[0, 0] - cd[0]) <= 1e-6 * max(1.0, abs(cd[0])), (G[0, 0], cd[0])
    ser.free()


@pytest.mark.parametrize("basis", ["SHO", "DRWCelerite"])
def test_norm_nu_mu_directions_equal_k5(pb, ctx, golden_single, basis):
    """On approx coefficients the JVP directions norm (da = a/norm, db = b/norm), ν and μ are K5's last three columns."""
    g = golden_single
    th = g.theta[::97][:24]
    spec = pb.make_spec(g.model, g.f_min, g.f_max, 20, basis_function=basis)
    ser = ctx.upload_series(g.t, g.y, g.s2)
    a, b, c, d = ctx.approx_coeffs(spec, th[:, :4])
    B, Jt = a.shape
    norm, nu, mu = th[:, 3], th[:, 4], th[:, 5]
    da, db = np.zeros((B, 3, Jt)), np.zeros((B, 3, Jt))
    da[:, 0], db[:, 0] = a / norm[:, None], b / norm[:, None]
    dnu, dmu = np.zeros((B, 3)), np.zeros((B, 3))
    dnu[:, 1], dmu[:, 2] = 1.0, 1.0
    L, G = ctx.celerite_logl_jvp(ser, a, b, c, d, mu=mu, nu=nu, da=da, db=db, dnu=dnu, dmu=dmu)
    kl, kg = ctx.approx_logl_grad(ser, spec, th)
    assert rel_err(L, kl).max() <= 1e-9
    _check(G, kg[:, 3:6])
    ser.free()


def test_periodic_mean(ctx, pb, golden_periodic):
    """Sinusoidal mean A·sin(2πt/T₀ + ϕ) + μ of the reference's periodic run: its parameters enter as dy tangents."""
    g = golden_periodic
    rows = g.chain[::211][:16]
    th = rows[:, 2:8]
    spec = pb.make_spec(g.model, g.f_min, g.f_max, 20)
    ser = ctx.upload_series(g.t, g.y, g.s2)
    a, b, c, d = ctx.approx_coeffs(spec, th[:, :4])
    B, N = len(rows), len(g.t)
    yb = np.stack([g.y - periodic_mean(g.t, r) + r[7] for r in rows])      # the constant μ rides as mu
    mu, nu = rows[:, 7], th[:, 4]
    A, phi, T0 = rows[:, 8:9], rows[:, 9:10], rows[:, 10:11]
    arg = 2 * np.pi * g.t[None] / T0 + phi
    dy = np.zeros((B, 5, N))
    dy[:, 2] = -np.sin(arg)                                                 # ∂ỹ/∂A
    dy[:, 3] = -A * np.cos(arg)                                             # ∂ỹ/∂ϕ
    dy[:, 4] = A * np.cos(arg) * 2 * np.pi * g.t[None] / T0 ** 2            # ∂ỹ/∂T₀
    dnu, dmu = np.zeros((B, 5)), np.zeros((B, 5))
    dnu[:, 0], dmu[:, 1] = 1.0, 1.0
    L, G = ctx.celerite_logl_jvp(ser, a, b, c, d, mu=mu, nu=nu, y_batch=yb, dnu=dnu, dmu=dmu, dy=dy)
    assert rel_err(L, rows[:, 1]).max() <= 1e-9
    wl, wg = oj.celerite_logl_jvp_batch(a, b, c, d, g.t, g.y, g.s2, mu=mu, nu=nu, y_batch=yb, dnu=dnu, dmu=dmu, dy=dy)
    _check(G, wg)
    # central differences of the GPU value along each of ν, μ, A, ϕ, T₀
    for p, col in enumerate((6, 7, 8, 9, 10)):                              # chain columns of ν, μ, A, ϕ, T₀
        hp = 1e-6 * np.maximum(np.abs(rows[:, col]), 1e-3)
        vals = []
        for e in (hp, -hp):
            r2 = rows.copy()
            r2[:, col] += e
            y2 = np.stack([g.y - periodic_mean(g.t, r) + r[7] for r in r2])
            vals.append(ctx.celerite_logl(ser, a, b, c, d, mu=r2[:, 7], nu=r2[:, 6], y_batch=y2))
        cd = (vals[0] - vals[1]) / (2 * hp)
        assert np.all(np.abs(G[:, p] - cd) <= 1e-5 * np.maximum(1.0, np.abs(cd))), (p, G[:, p], cd)
    ser.free()


def _features_theta(rng, B, f_min, f_max, nf):
    cols = [rng.uniform(0.0, 1.0, B), np.exp(rng.uniform(np.log(f_min), np.log(f_max), B)), rng.uniform(2.0, 3.5, B),
            np.exp(rng.normal(-1, 0.5, B)), rng.gamma(2, 0.5, B), rng.normal(0, 0.3, B)]
    for _ in range(nf):
        cols += [rng.uniform(0.5, 3, B), np.exp(rng.uniform(np.log(2 * f_min), np.log(f_max / 2), B)), rng.uniform(1.0, 15, B)]
    return np.column_stack(cols)


@pytest.mark.parametrize("nf", [1, 2])
@pytest.mark.parametrize("integrated", [True, False])
@pytest.mark.parametrize("basis", ["SHO", "DRWCelerite"])
def test_features_gradient(pb, ctx, basis, integrated, nf):
    t, y, s2, f_min, f_max = synthetic_series(400, 9)
    rng = np.random.default_rng(11 + nf)
    like = pb.BatchedLikelihood(t, y, s2, "SingleBendingPowerLaw", 20, basis, f_min=f_min, f_max=f_max, ctx=ctx, n_features=nf,
                                is_integrated_power=integrated)
    B = 12
    th = _features_theta(rng, B, f_min, f_max, nf)
    L, G = like.value_and_gradient(th)
    assert rel_err(L, like(th)).max() <= 1e-9
    kw = dict(basis=basis, is_integrated_power=integrated)
    wl, wg = oj.approx_features_logl_grad_batch("SBPL", th, nf, f_min, f_max, 20, t, y, s2, **kw)
    _, wg_ld = oj.approx_features_logl_grad_batch("SBPL", th, nf, f_min, f_max, 20, t, y, s2, long_double=True, **kw)
    assert rel_err(L, wl).max() <= 1e-9
    _check_ld(G, wg, wg_ld)
    like.close()


@pytest.mark.parametrize("basis", ["SHO", "DRWCelerite"])
def test_features_with_zero_amplitude_reduce_to_k5(pb, ctx, basis):
    t, y, s2, f_min, f_max = synthetic_series(400, 4)
    rng = np.random.default_rng(21)
    B = 10
    th = _features_theta(rng, B, f_min, f_max, 1)
    th[:, 6] = 0.0                                                   # S₀ = 0: the feature contributes nothing
    like = pb.BatchedLikelihood(t, y, s2, "SingleBendingPowerLaw", 20, basis, f_min=f_min, f_max=f_max, ctx=ctx, n_features=1)
    L, G = like.value_and_gradient(th)
    spec = pb.make_spec("SingleBendingPowerLaw", f_min, f_max, 20, basis_function=basis)
    kl, kg = ctx.approx_logl_grad(like.series, spec, th[:, :6])
    assert rel_err(L, kl).max() <= 1e-9
    _check(G[:, :6], kg)
    scale = np.abs(G).max()
    assert np.abs(G[:, 7:9]).max() <= 1e-12 * scale
    like.close()


@pytest.mark.parametrize("devices", [[0], [0, 1]])
def test_device_group_matches_single_context(pb, ctx, devices):
    """Rows split over the devices of a group, with per-row data (y_batch, s2_batch) and data tangents (dy, ds2) cut at the
    same offsets; the two-device case runs where two GPUs are visible."""
    if len(devices) > _ndev():
        pytest.skip("needs %d GPUs" % len(devices))
    grp = pb.Context(devices)
    rng = np.random.default_rng(8)
    N, B = 200, 5
    t = np.cumsum(rng.uniform(0.2, 1.5, N)); y = rng.normal(size=N); s2 = np.full(N, 0.3)
    s1, sg = ctx.upload_series(t, y, s2), grp.upload_series(t, y, s2)
    a, b, c, d = _coeffs(21, B, 9)
    tan = _tangents(rng, B, 3, a.shape[1], N, a, c)
    data = dict(mu=rng.normal(size=B), nu=rng.uniform(0.8, 1.2, B), y_batch=rng.normal(size=(B, N)),
                s2_batch=rng.uniform(0.2, 0.4, (B, N)))
    want = ctx.celerite_logl_jvp(s1, a, b, c, d, **data, **tan)
    got = grp.celerite_logl_jvp(sg, a, b, c, d, **data, **tan)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    t2, y2, v2, f_min, f_max = synthetic_series(300, 2)
    th = _features_theta(rng, 9, f_min, f_max, 1)
    l1 = pb.BatchedLikelihood(t2, y2, v2, "SingleBendingPowerLaw", 20, "SHO", f_min=f_min, f_max=f_max, ctx=ctx, n_features=1)
    lg = pb.BatchedLikelihood(t2, y2, v2, "SingleBendingPowerLaw", 20, "SHO", f_min=f_min, f_max=f_max, ctx=grp, n_features=1)
    w, g = l1.value_and_gradient(th), lg.value_and_gradient(th)
    assert np.array_equal(w[0], g[0]) and np.array_equal(w[1], g[1])
    l1.close(); lg.close(); s1.free(); sg.free()
    grp.close()


def test_errors_and_null_tangents(pb, ctx):
    from pioran_b200 import _lib
    rng = np.random.default_rng(1)
    N = 50
    t = np.cumsum(rng.uniform(0.2, 1.5, N)); y = rng.normal(size=N); s2 = np.full(N, 0.3)
    ser = ctx.upload_series(t, y, s2)
    a, b, c, d = _coeffs(97, 1, 3)                                   # rank 97
    with pytest.raises(_lib.PioranError) as e:
        ctx.celerite_logl_jvp(ser, a, b, c, d, dmu=np.ones((1, 1)))
    assert e.value.code == -5
    a, b, c, d = _coeffs(10, 2, 3)
    dp = C.POINTER(C.c_double)
    p = lambda x: x.ctypes.data_as(dp) if x is not None else None
    L, G = np.empty(2), np.full((2, 3), np.nan)
    lib = ctx.lib
    args = lambda P, gout: (ctx.h, ser.id, 2, a.shape[1], P, p(a), p(b), p(c), p(d), None, None, None, None,
                            *([None] * 8), p(L), gout)
    assert lib.pioran_celerite_logl_jvp(*args(0, p(G))) == -1
    assert lib.pioran_celerite_logl_jvp(*args(3, None)) == -1
    assert lib.pioran_celerite_logl_jvp(*args(3, p(G))) == 0
    assert np.array_equal(G, np.zeros((2, 3)))
    assert rel_err(L, ctx.celerite_logl(ser, a, b, c, d)).max() <= 1e-9
    spec = pb.make_spec("SingleBendingPowerLaw", 0.01, 1.0, 20)
    th = np.ones((1, 6 + 27))
    with pytest.raises(_lib.PioranError) as e:
        ctx.approx_features_logl_grad(ser, spec, 9, th)
    assert e.value.code == -5
    ser.free()
