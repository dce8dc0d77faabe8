"""K5r (csrc/vjp.cuh): the reverse-mode gradient of the explicit-coefficient likelihood, the reverse gradient with PSD features and
the CARMA gradient built on it, through the C ABI and the Python classes.  References: the dual-number oracle
tests/tools/oracle_jvp.c on unit directions, the K5g kernel by duality, a dense solve for the data gradients, the forward features
entry, and central differences of the GPU's own CARMA values."""
import ctypes as C

import numpy as np
import pytest

import os
import sys

from conftest import rel_err, synthetic_series

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "tools"))
import oracle_jvp as oj  # noqa: E402

pytestmark = pytest.mark.gpu
RTOL = 1e-8


@pytest.fixture(scope="module")
def pb():
    import pioran_b200
    return pioran_b200


@pytest.fixture(scope="module")
def ctx(pb):
    return pb.get_context(0)


def _check(got, want, rtol=RTOL):
    """|got − want| within rtol of the column scale (the _check rule of test_gpu_jvp.py)."""
    got, want = np.atleast_2d(got), np.atleast_2d(want)
    scale = np.maximum(np.abs(want), np.abs(want).max(axis=0, keepdims=True))
    scale = np.where(scale > 0, scale, 1.0)
    err = np.abs(got - want) / scale
    assert np.all(np.isfinite(got)), "non-finite gradient"
    assert err.max() <= rtol, f"gradient parity {err.max():.3e} at {np.unravel_index(err.argmax(), err.shape)}"


def _coeffs(R, B, seed, mixed=False, negative=False):
    """B coefficient sets of rank R (SHO-form complex terms, one real term when R is odd).  mixed: the first complex term of every
    set but the first is real, so the batch keeps it at two rows.  negative: some b and d flipped in sign."""
    rng = np.random.default_rng(seed)
    nc, nr = R // 2, R % 2
    Jt = nc + nr
    a = rng.uniform(0.1, 1.0, (B, Jt)) / Jt
    c = np.exp(rng.uniform(np.log(0.05), np.log(5.0), (B, Jt)))
    b, d = a.copy(), c.copy()
    if negative:
        b[:, ::2] *= -0.5
        d[:, 1::2] *= -1.0
    b[:, nc:], d[:, nc:] = 0.0, 0.0
    if mixed and nc:
        b[1:, 0], d[1:, 0] = 0.0, 0.0
    return a, b, c, d


def _series(rng, N):
    return np.cumsum(rng.uniform(0.2, 1.5, N)), rng.normal(size=N), rng.uniform(0.2, 0.4, N)


def _unit_oracle(a, b, c, d, t, y, s2, mu, nu, yb=None, sb=None):
    """The oracle's gradient with respect to a, b, c, d, μ, ν from P = 4 Jt + 2 unit directions."""
    B, Jt = a.shape
    P = 4 * Jt + 2
    tan = {k: np.zeros((B, P, Jt)) for k in ("da", "db", "dc", "dd")}
    for q, k in enumerate(("da", "db", "dc", "dd")):
        tan[k][:, q * Jt:(q + 1) * Jt, :] = np.eye(Jt)[None]
    dmu, dnu = np.zeros((B, P)), np.zeros((B, P))
    dmu[:, 4 * Jt], dnu[:, 4 * Jt + 1] = 1.0, 1.0
    L, G = oj.celerite_logl_jvp_batch(a, b, c, d, t, y, s2, mu=mu, nu=nu, y_batch=yb, s2_batch=sb, dmu=dmu, dnu=dnu, **tan)
    return L, G


def _flat(g):
    return np.concatenate([g["a"], g["b"], g["c"], g["d"], g["mu"][:, None], g["nu"][:, None]], axis=1)


def _dense(a, b, c, d, t, y, s2, mu, nu):
    """Data gradients of one set from a dense solve: g_y = −α, g_s2 = ν·½(α² − diag (K + Σ)⁻¹), α = (K + Σ)⁻¹ (y − μ)."""
    tau = np.abs(t[:, None] - t[None, :])
    K = sum(np.exp(-c[m] * tau) * (a[m] * np.cos(d[m] * tau) + b[m] * np.sin(d[m] * tau)) for m in range(a.shape[0]))
    inv = np.linalg.inv(K + np.diag(nu * s2))
    alpha = inv @ (y - mu)
    return -alpha, nu * 0.5 * (alpha ** 2 - np.diag(inv))


@pytest.mark.parametrize("N", [1, 2, 333])
@pytest.mark.parametrize("R", [2, 5, 16, 17, 32, 33, 48, 64, 65, 80, 96])
def test_vjp_vs_reference(ctx, R, N):
    rng = np.random.default_rng(R * 1000 + N + 7)
    t, y, s2 = _series(rng, N)
    ser = ctx.upload_series(t, y, s2)
    B = 3
    a, b, c, d = _coeffs(R, B, R + N, mixed=R > 4, negative=R % 3 == 0)
    mu, nu = rng.normal(0, 0.3, B), rng.uniform(0.8, 1.5, B)
    L, g = ctx.celerite_logl_vjp(ser, a, b, c, d, mu=mu, nu=nu, data_grad=True)
    assert ctx.last_kernel_name() == f"vjp<{max(1, (R + 15) // 16)}>"
    assert rel_err(L, ctx.celerite_logl(ser, a, b, c, d, mu=mu, nu=nu)).max() <= 1e-9
    wl, wg = _unit_oracle(a, b, c, d, t, y, s2, mu, nu)
    assert rel_err(L, wl).max() <= 1e-9
    _check(_flat(g), wg)
    if R % 2:                                                         # the real term: exactly zero b and d partials
        assert np.all(g["b"][:, -1] == 0.0) and np.all(g["d"][:, -1] == 0.0)
    # data gradients against a dense solve, and the μ, ν identities
    for i in range(B):
        gy, gs2 = _dense(a[i], b[i], c[i], d[i], t, y, s2, mu[i], nu[i])
        _check(g["y"][i], gy)
        _check(g["s2"][i], gs2)
    _check(g["mu"], -g["y"].sum(axis=1))
    _check(g["nu"], (s2[None, :] * g["s2"]).sum(axis=1) / nu)
    # duality against K5g along random directions over every input
    P = 3
    tan = {k: rng.normal(size=(B, P, a.shape[1])) for k in ("da", "db", "dc", "dd")}
    tan.update(dmu=rng.normal(size=(B, P)), dnu=rng.normal(size=(B, P)), dy=rng.normal(size=(B, P, N)), ds2=rng.normal(size=(B, P, N)))
    _, jv = ctx.celerite_logl_jvp(ser, a, b, c, d, mu=mu, nu=nu, **tan)
    dot = g["mu"][:, None] * tan["dmu"] + g["nu"][:, None] * tan["dnu"]
    for k, v in (("a", "da"), ("b", "db"), ("c", "dc"), ("d", "dd"), ("y", "dy"), ("s2", "ds2")):
        dot = dot + np.einsum("ij,ipj->ip", g[k], tan[v])
    _check(dot, jv)
    ser.free()


def test_negative_coefficients_batch_rows_and_nan(ctx):
    """The rank-reduction set of test_gpu_parity.py (negative a, b, d; real terms) with per-row data; a NaN coefficient
    propagates to its own row only."""
    rng = np.random.default_rng(3)
    N = 150
    t, y, s2 = _series(rng, N)
    ser = ctx.upload_series(t, y, s2)
    a = np.array([[1.2, 0.8, -0.3, 0.5], [2.0, 0.1, -0.05, 1.0], [1.5, 0.4, 0.2, 0.7]])
    b = np.array([[0.0, 0.3, -0.1, 0.0], [0.0, -0.05, 0.02, 0.0], [0.0, 0.1, 0.05, 0.0]])
    c = np.array([[0.3, 0.2, 1.0, 2.0], [0.1, 0.5, 0.8, 3.0], [0.4, 0.3, 0.9, 1.0]])
    d = np.array([[0.0, 1.5, -2.0, 0.0], [0.0, 0.7, -1.0, 0.0], [0.0, 2.0, 1.0, 0.0]])
    mu, nu = np.array([0.1, -0.2, 0.0]), np.array([1.3, 0.9, 1.0])
    yb, sb = rng.normal(size=(3, N)), rng.uniform(0.2, 0.4, (3, N))
    L, g = ctx.celerite_logl_vjp(ser, a, b, c, d, mu=mu, nu=nu, y_batch=yb, s2_batch=sb)
    wl, wg = _unit_oracle(a, b, c, d, t, y, s2, mu, nu, yb, sb)
    assert rel_err(L, wl).max() <= 1e-9
    _check(_flat(g), wg)
    assert np.all(g["b"][:, [0, 3]] == 0.0) and np.all(g["d"][:, [0, 3]] == 0.0)
    a2 = a.copy()
    a2[1, 2] = np.nan
    L2, g2 = ctx.celerite_logl_vjp(ser, a2, b, c, d, mu=mu, nu=nu, y_batch=yb, s2_batch=sb)
    assert np.isnan(L2[1]) and np.isnan(g2["a"][1]).all()
    assert np.array_equal(L2[[0, 2]], L[[0, 2]]) and np.array_equal(g2["c"][[0, 2]], g["c"][[0, 2]])
    ser.free()


def test_workspace_chunks(pb):
    """A cap that fits three sets splits a batch of 8 into three θ-chunks (data gradients copied back chunk by chunk); every
    output is bit-equal to the single-chunk run."""
    ctx = pb.Context(0)                                               # its own context: the cap is per context
    rng = np.random.default_rng(5)
    N, B, R = 333, 8, 33
    t, y, s2 = _series(rng, N)
    ser = ctx.upload_series(t, y, s2)
    a, b, c, d = _coeffs(R, B, 4, mixed=True)
    kw = dict(mu=rng.normal(0, 0.3, B), nu=rng.uniform(0.8, 1.5, B), y_batch=rng.normal(size=(B, N)),
              s2_batch=rng.uniform(0.2, 0.4, (B, N)), data_grad=True)
    L1, g1 = ctx.celerite_logl_vjp(ser, a, b, c, d, **kw)
    TS, K = 3, 20                                                     # K = ⌈√333⌉ rounded up to a multiple of 4
    per = 8 * (N * (2 * 16 * TS + 2) + (-(-N // K) + K) * 256 * TS * TS)
    ctx.set_vjp_workspace(3 * per + per // 2)
    n0 = ctx.launch_count
    L2, g2 = ctx.celerite_logl_vjp(ser, a, b, c, d, **kw)
    assert ctx.launch_count - n0 == 3
    ctx.set_vjp_workspace(0)
    assert np.array_equal(L1, L2)
    for k in g1:
        assert np.array_equal(g1[k], g2[k]), k
    ser.free()
    ctx.close()


def _features_theta(rng, B, f_min, f_max, nf):
    cols = [rng.uniform(0.0, 1.0, B), np.exp(rng.uniform(np.log(f_min), np.log(f_max), B)), rng.uniform(2.0, 3.5, B),
            np.exp(rng.normal(-1, 0.5, B)), rng.gamma(2, 0.5, B), rng.normal(0, 0.3, B)]
    for _ in range(nf):
        cols += [rng.uniform(0.5, 3, B), np.exp(rng.uniform(np.log(2 * f_min), np.log(f_max / 2), B)), rng.uniform(1.0, 15, B)]
    return np.column_stack(cols)


@pytest.mark.parametrize("nf", [1, 2])
@pytest.mark.parametrize("integrated", [True, False])
@pytest.mark.parametrize("basis", ["SHO", "DRWCelerite"])
def test_features_reverse_gradient(pb, ctx, basis, integrated, nf):
    t, y, s2, f_min, f_max = synthetic_series(400, 9)
    rng = np.random.default_rng(11 + nf)
    kw = dict(f_min=f_min, f_max=f_max, ctx=ctx, n_features=nf, is_integrated_power=integrated)
    rev = pb.BatchedLikelihood(t, y, s2, "SingleBendingPowerLaw", 20, basis, gradient="reverse", **kw)
    fwd = pb.BatchedLikelihood(t, y, s2, "SingleBendingPowerLaw", 20, basis, **kw)
    th = _features_theta(rng, 12, f_min, f_max, nf)
    L, G = rev.value_and_gradient(th)
    assert ctx.last_kernel_name().startswith("vjp<")
    Lf, Gf = fwd.value_and_gradient(th)
    assert ctx.last_kernel_name().startswith("jvp<")
    assert rel_err(L, Lf).max() <= 1e-9
    _check(G, Gf)
    wl, wg = oj.approx_features_logl_grad_batch("SBPL", th, nf, f_min, f_max, 20, t, y, s2, basis=basis, is_integrated_power=integrated)
    assert rel_err(L, wl).max() <= 1e-9
    _check(G, wg)
    rev.close(); fwd.close()


def test_reverse_option_needs_features(pb, ctx):
    t, y, s2, f_min, f_max = synthetic_series(50, 1)
    with pytest.raises(ValueError):
        pb.BatchedLikelihood(t, y, s2, "SingleBendingPowerLaw", 20, "SHO", f_min=f_min, f_max=f_max, ctx=ctx, gradient="reverse")


def _carma_theta(rng, B, p, q, log_shift, cmax):
    cols = [rng.uniform(0.4, 1.8, (B, p)), rng.uniform(0.4, 1.8, (B, q)), rng.uniform(0.5, 2.0, (B, 1)),
            rng.uniform(0.8, 1.3, (B, 1)), rng.normal(0.0, 0.2, (B, 1))]
    if log_shift:
        cols.append(rng.uniform(0.0, cmax, (B, 1)))
    return np.concatenate(cols, axis=1)


@pytest.mark.parametrize("log_shift", [False, True])
@pytest.mark.parametrize("p,q", [(3, 1), (4, 2), (5, 2)])
def test_carma_gradient_matches_central_differences(pb, ctx, p, q, log_shift):
    rng = np.random.default_rng(10 * p + q)
    N = 200
    t = np.cumsum(rng.uniform(0.2, 1.0, N))
    y = np.exp(rng.normal(0.0, 0.3, N)) + 1.0
    s2 = (0.05 * y) ** 2
    like = pb.BatchedCARMALikelihood(t, y, s2, p, q, 1e-3, 10.0, log_shift=log_shift, ctx=ctx)
    B = 5
    th = _carma_theta(rng, B, p, q, log_shift, 0.8 * y.min())
    th[-1, 0] = -1.0                                                  # a root with positive real part: outside the bounds
    L, G = like.value_and_gradient(th)
    assert ctx.last_kernel_name().startswith("vjp<")
    assert np.array_equal(L[:-1], like(th)[:-1]) or rel_err(L[:-1], like(th)[:-1]).max() <= 1e-9
    assert L[-1] == -np.inf and np.all(G[-1] == 0.0)
    # five-point central differences at h = 1e-4: the two-point rule at h = 1e-6 carries ~1e-5 of the column scale of rounding
    # noise on the worse-conditioned rows (|logL| ~ 300), more than the tolerance
    cd = np.empty((B - 1, like.n_par))
    for k in range(like.n_par):
        h = 1e-4 * np.maximum(np.abs(th[:-1, k]), 1e-2)
        at = lambda s: like(th[:-1] + s * h[:, None] * np.eye(like.n_par)[k][None, :])
        cd[:, k] = (-at(2) + 8 * at(1) - 8 * at(-1) + at(-2)) / (12 * h)
    err = np.abs(G[:-1] - cd) / np.maximum(1.0, np.abs(cd).max(axis=0, keepdims=True))
    assert err.max() <= 1e-6, (np.unravel_index(err.argmax(), err.shape), err.max())
    assert np.array_equal(like.gradient(th), G)
    like.close()


def _ndev():
    rt = C.CDLL("libcudart.so")
    n = C.c_int(0)
    rt.cudaGetDeviceCount(C.byref(n))
    return n.value


@pytest.mark.parametrize("devices", [[0], [0, 1]])
def test_device_group_matches_single_context(pb, ctx, devices):
    if len(devices) > _ndev():
        pytest.skip("needs %d GPUs" % len(devices))
    grp = pb.Context(devices)
    rng = np.random.default_rng(8)
    N, B = 200, 5
    t, y, s2 = _series(rng, N)
    s1, sg = ctx.upload_series(t, y, s2), grp.upload_series(t, y, s2)
    a, b, c, d = _coeffs(21, B, 9)
    data = dict(mu=rng.normal(size=B), nu=rng.uniform(0.8, 1.2, B), y_batch=rng.normal(size=(B, N)),
                s2_batch=rng.uniform(0.2, 0.4, (B, N)), data_grad=True)
    wl, wg = ctx.celerite_logl_vjp(s1, a, b, c, d, **data)
    gl, gg = grp.celerite_logl_vjp(sg, a, b, c, d, **data)
    assert np.array_equal(gl, wl)
    for k in wg:
        assert np.array_equal(gg[k], wg[k]), k
    t2, y2, v2, f_min, f_max = synthetic_series(300, 2)
    th = _features_theta(rng, 9, f_min, f_max, 1)
    kw = dict(f_min=f_min, f_max=f_max, n_features=1, gradient="reverse")
    l1 = pb.BatchedLikelihood(t2, y2, v2, "SingleBendingPowerLaw", 20, "SHO", ctx=ctx, **kw)
    lg = pb.BatchedLikelihood(t2, y2, v2, "SingleBendingPowerLaw", 20, "SHO", ctx=grp, **kw)
    w, g = l1.value_and_gradient(th), lg.value_and_gradient(th)
    assert np.array_equal(w[0], g[0]) and np.array_equal(w[1], g[1])
    l1.close(); lg.close(); s1.free(); sg.free()
    grp.close()


def test_errors(pb, ctx):
    from pioran_b200 import _lib
    rng = np.random.default_rng(1)
    N = 50
    t, y, s2 = _series(rng, N)
    ser = ctx.upload_series(t, y, s2)
    a, b, c, d = _coeffs(97, 1, 3)                                   # rank 97
    with pytest.raises(_lib.PioranError) as e:
        ctx.celerite_logl_vjp(ser, a, b, c, d)
    assert e.value.code == -5
    a, b, c, d = _coeffs(10, 2, 3)
    dp = C.POINTER(C.c_double)
    p = lambda x: x.ctypes.data_as(dp) if x is not None else None
    L, ga = np.empty(2), np.empty((2, a.shape[1]))
    lib = ctx.lib
    args = lambda sid, B, gout: (ctx.h, sid, B, a.shape[1], p(a), p(b), p(c), p(d), None, None, None, None, p(L), gout,
                                 *([None] * 7))
    assert lib.pioran_celerite_logl_vjp(*args(ser.id, 2, None)) == -1          # no gradient output
    assert lib.pioran_celerite_logl_vjp(*args(ser.id + 1000, 2, p(ga))) == -1  # unknown series
    assert lib.pioran_celerite_logl_vjp(*args(ser.id, 0, p(ga))) == -1         # B = 0
    assert lib.pioran_celerite_logl_vjp(*args(ser.id, 2, p(ga))) == 0
    assert rel_err(L, ctx.celerite_logl(ser, a, b, c, d)).max() <= 1e-9
    spec = pb.make_spec("SingleBendingPowerLaw", 0.01, 1.0, 20)
    with pytest.raises(_lib.PioranError) as e:
        ctx.approx_features_logl_grad_reverse(ser, spec, 9, np.ones((1, 6 + 27)))
    assert e.value.code == -5
    ser.free()
