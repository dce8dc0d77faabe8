"""Sinusoidal-mean likelihood and gradient (pioran_approx_logl_sine, pioran_approx_logl_sine_grad): the reference's periodicity
run, examples/ultranest/single_pl_periodicity.jl, with m(t) = μ + A·sin(2πt/T₀ + ϕ) and Θ row [psd…, norm, ν, μ, A, ϕ, T₀]."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

from conftest import assert_parity, rel_err, synthetic_series

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "tools"))
import oracle_sine as orc  # noqa: E402

TOL = 1e-9
RTOL = 1e-8      # gradient entries against the oracle, on the scale of their column (test_gpu_grad.py)


@pytest.fixture(scope="module")
def pb():
    import pioran_b200
    return pioran_b200


@pytest.fixture(scope="module")
def ctx(pb):
    return pb.get_context(0)


def _check(got, want, ld=None, rtol=RTOL, slack=4.0):
    """Entries within rtol of their column's scale; with the 80-bit oracle `ld`, an entry may exceed rtol only where the FP64
    oracle is itself farther than rtol/slack from the 80-bit one, and then the GPU must lie within slack × that distance of it
    (the rule of conftest.assert_parity, per entry)."""
    scale = np.maximum(np.abs(want), np.abs(want).max(axis=0, keepdims=True))
    err = np.abs(got - want) / scale
    assert np.all(np.isfinite(got)), "non-finite gradient"
    bad = err > rtol
    if ld is not None and bad.any():
        e_ref, e_gpu = np.abs(want - ld) / scale, np.abs(got - ld) / scale
        bad &= ~((e_ref > rtol / slack) & (e_gpu <= slack * e_ref))
    assert not bad.any(), f"gradient parity {err[bad].max():.3e} (column {np.argwhere(bad)[0][1]})"


def _same_value(val, plain, ref, ld):
    """The gradient entry's value against the likelihood entry's.  The gradient entry takes its amplitudes from the dual-number
    K1 (approx_grad_kernel), whose rounding differs from the value K1's, and the sweep amplifies that difference by the row's
    condition: within 1e-12 relative where the FP64 oracle `ref` agrees with the 80-bit one `ld` to 1e-13; elsewhere both meet
    the parity rule of conftest.assert_parity against the oracle (the caller checks `val`, this checks `plain`)."""
    d = np.abs(val - plain)
    cond = np.abs(ref - ld) <= 1e-13 * np.abs(ld)
    assert np.all(d[cond] <= 1e-12 * np.abs(plain[cond])), np.max(d[cond] / np.abs(plain[cond]))
    e_ref, e_gpu = rel_err(ref, ld), rel_err(plain, ld)
    assert np.all((rel_err(plain, ref) <= 1e-9) | ((e_ref > 1e-9 / 4) & (e_gpu <= 4 * e_ref)))


def _mean_draws(rng, B, ysd):
    """(A, ϕ, T₀): an amplitude up to the spread of the series, T₀ between a day and the span of the golden series."""
    return np.column_stack([rng.uniform(0.0, ysd, B), rng.uniform(0.0, 2 * np.pi, B), np.exp(rng.uniform(0.0, np.log(700.0), B))])


def _prior(model, rng, B, f_min, f_max, y, alpha_max):
    """PSD rows over the prior's range; variance, ν, μ and (A, ϕ, T₀) near the series' own scale, so that the rows are as well
    conditioned as the ones a sampler spends its time on (the 80-bit oracle agrees with the FP64 one on all of them)."""
    f0, fM = f_min / 20.0, f_max * 20.0
    a1 = rng.uniform(0.0, 1.5, B)
    f1 = np.exp(rng.uniform(np.log(4 * f0), np.log(fM / 64), B))
    if model == "SingleBendingPowerLaw":
        psd = [a1, f1, a1 + rng.uniform(size=B) * (alpha_max - a1)]
    else:
        a2 = a1 + rng.uniform(size=B) * (0.5 * (alpha_max + a1) - a1)
        psd = [a1, f1, a2, f1 * np.exp(rng.uniform(np.log(2.0), np.log(16.0), B)), a2 + rng.uniform(size=B) * (alpha_max - a2)]
    rest = [y.var() * np.exp(rng.normal(0.0, 0.5, B)), rng.gamma(4.0, 0.25, B), rng.normal(y.mean(), 0.1 * y.std(), B)]
    return np.column_stack(psd + rest + [_mean_draws(rng, B, y.std())])


def _ld_value(model, f_min, f_max, J, basis, t, y, s2):
    return lambda row: orc.approx_logl_sine_grad_batch(model, row[None], f_min, f_max, J, t, y, s2, basis=basis, long_double=True)[0][0]


def _expected_kernel(R, ND):
    """blocked_grad_sine<NT, NTR, HALF, NTAN> of the gradient row layout (blocked.cuh blk_layout(R, true))."""
    NT = (R + 7) // 8
    if R % 8 in (0, 7):
        return f"blocked_grad_sine<{NT},{NT + 1},false,{ND + 1}>"
    return f"blocked_grad_sine<{NT},{NT},{'true' if 1 <= R % 8 <= 4 else 'false'},{ND + 1}>"


# ------------------------------------------------------------------------------------------------- value
@pytest.mark.gpu
def test_golden_pairs(pb, ctx, golden_periodic):
    """All 8 480 (θ, logℒ) pairs of simu_periodic_rednoise through the fused entry."""
    g = golden_periodic
    theta = np.ascontiguousarray(g.chain[:, 2:11])
    spec = pb.make_spec(g.model, g.f_min, g.f_max, 20)
    ser = ctx.upload_series(g.t, g.y, g.s2)
    got = ctx.approx_logl_sine(ser, spec, theta)
    assert np.median(rel_err(got, g.logl)) < 1e-12
    assert_parity(got, g.logl, theta, _ld_value("SBPL", g.f_min, g.f_max, 20, "SHO", g.t, g.y, g.s2), TOL)
    ser.free()


@pytest.mark.gpu
@pytest.mark.parametrize("model,basis,J", [("SingleBendingPowerLaw", "SHO", 20), ("SingleBendingPowerLaw", "DRWCelerite", 20),
                                           ("DoubleBendingPowerLaw", "SHO", 13), ("SingleBendingPowerLaw", "SHO", 10)])
def test_amplitude_zero_is_the_constant_mean(pb, ctx, golden_periodic, model, basis, J):
    """A = 0: ỹ = y exactly, so the value is pioran_approx_logl's and the gradient's other columns are
    pioran_approx_logl_grad's, bit for bit; ∂/∂ϕ and ∂/∂T₀ are exactly 0.  B = 5 also takes the one-CTA-per-θ value kernel."""
    g = golden_periodic
    rng = np.random.default_rng(3)
    nd = 3 if model == "SingleBendingPowerLaw" else 5
    for B in (5, 300):
        theta = _prior(model, rng, B, g.f_min, g.f_max, g.y, 4.0 if basis == "SHO" else 6.0)
        theta[:, nd + 3] = 0.0
        spec = pb.make_spec(model, g.f_min, g.f_max, J, basis_function=basis)
        ser = ctx.upload_series(g.t, g.y, g.s2)
        v = ctx.approx_logl_sine(ser, spec, theta)
        vp = ctx.approx_logl(ser, spec, theta[:, :nd + 3])[0]
        assert np.array_equal(v, vp, equal_nan=True)
        gv, gg = ctx.approx_logl_sine_grad(ser, spec, theta)
        gvp, ggp = ctx.approx_logl_grad(ser, spec, theta[:, :nd + 3])
        assert np.array_equal(gv, gvp, equal_nan=True) and np.array_equal(gg[:, :nd + 3], ggp, equal_nan=True)
        assert np.all(gg[:, nd + 4:] == 0.0)
        ser.free()


@pytest.mark.gpu
def test_value_rows_are_the_host_built_data(pb, ctx, golden_periodic):
    """The device transform against today's route: y − m_θ(t) built on the host, through the generic entry."""
    g = golden_periodic
    rows = g.chain[::97]
    theta = np.ascontiguousarray(rows[:, 2:11])
    spec = pb.make_spec(g.model, g.f_min, g.f_max, 20)
    ser = ctx.upload_series(g.t, g.y, g.s2)
    got = ctx.approx_logl_sine(ser, spec, theta)
    a, b, c, d = ctx.approx_coeffs(spec, theta[:, :4])
    yb = g.y[None] - theta[:, 6:7] * np.sin(2 * np.pi * g.t[None] / theta[:, 8:9] + theta[:, 7:8])
    gen = ctx.celerite_logl(ser, a, b, c, d, mu=theta[:, 5], nu=theta[:, 4], y_batch=yb)
    assert rel_err(got, gen).max() <= 1e-11
    ser.free()


# ------------------------------------------------------------------------------------------------- gradient
# (model, basis, J): R mod 8 = 0 (own data tile), 1 … 4 (HALF), 5 … 7 (7: own data tile in the gradient layout), up to 62
GRAD_CASES = [("SingleBendingPowerLaw", "SHO", 20), ("SingleBendingPowerLaw", "SHO", 31), ("SingleBendingPowerLaw", "SHO", 10),
              ("SingleBendingPowerLaw", "SHO", 3), ("SingleBendingPowerLaw", "DRWCelerite", 20), ("SingleBendingPowerLaw", "DRWCelerite", 5),
              ("SingleBendingPowerLaw", "DRWCelerite", 11), ("DoubleBendingPowerLaw", "SHO", 20), ("DoubleBendingPowerLaw", "SHO", 31),
              ("DoubleBendingPowerLaw", "DRWCelerite", 7), ("DoubleBendingPowerLaw", "DRWCelerite", 12), ("DoubleBendingPowerLaw", "SHO", 4)]


@pytest.mark.gpu
def test_gradient_golden_rows_vs_oracle(pb, ctx, golden_periodic):
    """Every 50th golden pair: value and all nine partials against the oracle's dual-number sweep."""
    g = golden_periodic
    theta = np.ascontiguousarray(g.chain[::50, 2:11])
    like = pb.BatchedLikelihood(g.t, g.y, g.s2, g.model, 20, "SHO", f_min=g.f_min, f_max=g.f_max, ctx=ctx, periodic_mean=True)
    val, grad = like.value_and_gradient(theta)
    assert ctx.last_kernel_name() == "blocked_grad_sine<5,6,false,4>"
    oval, ograd = orc.approx_logl_sine_grad_batch("SBPL", theta, g.f_min, g.f_max, 20, g.t, g.y, g.s2, nthreads=0)
    lval, lgrad = orc.approx_logl_sine_grad_batch("SBPL", theta, g.f_min, g.f_max, 20, g.t, g.y, g.s2, nthreads=0, long_double=True)
    assert_parity(val, oval, theta, lambda row: lval[np.flatnonzero((theta == row).all(axis=1))[0]], TOL)
    _check(grad, ograd, lgrad)
    like.close()


@pytest.mark.gpu
@pytest.mark.parametrize("model,basis,J", GRAD_CASES)
def test_gradient_prior_draws_vs_oracle(pb, ctx, golden_periodic, model, basis, J):
    g = golden_periodic
    rng = np.random.default_rng(J + 100 * len(model))
    omodel = "SBPL" if model == "SingleBendingPowerLaw" else "DBPL"
    theta = _prior(model, rng, 24, g.f_min, g.f_max, g.y, 4.0 if basis == "SHO" else 6.0)
    spec = pb.make_spec(model, g.f_min, g.f_max, J, basis_function=basis)
    ser = ctx.upload_series(g.t, g.y, g.s2)
    val, grad = ctx.approx_logl_sine_grad(ser, spec, theta)
    R = 2 * J if basis == "SHO" else 3 * J
    assert ctx.last_kernel_name() == _expected_kernel(R, 3 if omodel == "SBPL" else 5)
    oval, ograd = orc.approx_logl_sine_grad_batch(omodel, theta, g.f_min, g.f_max, J, g.t, g.y, g.s2, basis=basis, nthreads=0)
    lval, lgrad = orc.approx_logl_sine_grad_batch(omodel, theta, g.f_min, g.f_max, J, g.t, g.y, g.s2, basis=basis, nthreads=0,
                                                  long_double=True)
    assert_parity(val, oval, theta, lambda row: lval[np.flatnonzero((theta == row).all(axis=1))[0]], TOL)
    _check(grad, ograd, lgrad)
    _same_value(val, ctx.approx_logl_sine(ser, spec, theta), oval, lval)      # the gradient entry's value is the likelihood entry's
    ser.free()


@pytest.mark.gpu
def test_mean_partials_match_central_differences(pb, ctx, golden_periodic):
    """∂/∂A, ∂/∂ϕ, ∂/∂T₀ against central differences of the GPU value itself (independent of the oracle)."""
    g = golden_periodic
    theta = np.ascontiguousarray(g.chain[::1061, 2:11])
    spec = pb.make_spec(g.model, g.f_min, g.f_max, 20)
    ser = ctx.upload_series(g.t, g.y, g.s2)
    val, grad = ctx.approx_logl_sine_grad(ser, spec, theta)
    for k in (6, 7, 8):
        h = 1e-6 * np.maximum(1.0, np.abs(theta[:, k]))
        tp, tm = theta.copy(), theta.copy()
        tp[:, k] += h
        tm[:, k] -= h
        fd = (ctx.approx_logl_sine(ser, spec, tp) - ctx.approx_logl_sine(ser, spec, tm)) / (2 * h)
        noise = 2e-15 * np.abs(val).max() / h.min()
        assert np.allclose(grad[:, k], fd, rtol=2e-5, atol=1e-6 * np.abs(grad[:, k]).max() + noise), k
    ser.free()


@pytest.mark.gpu
def test_value_from_the_gradient_entry(pb, ctx, golden_periodic):
    g = golden_periodic
    theta = np.ascontiguousarray(g.chain[::7, 2:11])
    spec = pb.make_spec(g.model, g.f_min, g.f_max, 20)
    ser = ctx.upload_series(g.t, g.y, g.s2)
    val, _ = ctx.approx_logl_sine_grad(ser, spec, theta)
    plain = ctx.approx_logl_sine(ser, spec, theta)
    far = np.flatnonzero(~(np.abs(val - plain) <= 1e-12 * np.abs(plain)))      # the 80-bit oracle only where needed
    assert far.size <= 0.02 * theta.shape[0], far.size
    if far.size:
        oval = orc.approx_logl_sine_grad_batch("SBPL", theta[far], g.f_min, g.f_max, 20, g.t, g.y, g.s2, nthreads=0)[0]
        lval = orc.approx_logl_sine_grad_batch("SBPL", theta[far], g.f_min, g.f_max, 20, g.t, g.y, g.s2, nthreads=0,
                                               long_double=True)[0]
        _same_value(val[far], plain[far], oval, lval)
    ser.free()


# ------------------------------------------------------------------------------------------------- chunks, groups, limits
@pytest.mark.gpu
def test_theta_chunks_equal_single_set_calls(pb, ctx):
    """N = 1e5: 800 kB of ỹ per parameter vector, 1 342 per 1 GiB chunk; B = 2 689 runs three chunks.  Rank 20 keeps B = 1 on
    the warp-per-θ value kernel, so every row must equal its single-set call bit for bit."""
    t, y, s2, f_min, f_max = synthetic_series(100_000, 5)
    per_chunk = (1 << 30) // (8 * t.size)
    B = 2 * per_chunk + 5
    rng = np.random.default_rng(8)
    theta = _prior("SingleBendingPowerLaw", rng, B, f_min, f_max, y, 4.0)
    spec = pb.make_spec("SingleBendingPowerLaw", f_min, f_max, 10)
    ser = ctx.upload_series(t, y, s2)
    n0 = ctx.launch_count
    val = ctx.approx_logl_sine(ser, spec, theta)
    assert ctx.launch_count - n0 >= 3 * 3            # per chunk: transform, K1, K2
    gv, gg = ctx.approx_logl_sine_grad(ser, spec, theta)
    for i in (0, per_chunk - 1, per_chunk, 2 * per_chunk, B - 1):
        assert np.array_equal(ctx.approx_logl_sine(ser, spec, theta[i:i + 1]), val[i:i + 1])
        v1, g1 = ctx.approx_logl_sine_grad(ser, spec, theta[i:i + 1])
        assert np.array_equal(v1, gv[i:i + 1]) and np.array_equal(g1, gg[i:i + 1])
    ser.free()


def _ndev():
    import torch
    return torch.cuda.device_count()


@pytest.mark.gpu
def test_device_group_splits_the_batch(pb, golden_periodic):
    if _ndev() < 2:
        pytest.skip("needs 2 GPUs")
    g = golden_periodic
    theta = np.ascontiguousarray(g.chain[::41, 2:11])
    one, grp = pb.get_context(0), pb.Context([0, 1])
    try:
        spec = pb.make_spec(g.model, g.f_min, g.f_max, 20)
        s1, sg = one.upload_series(g.t, g.y, g.s2), grp.upload_series(g.t, g.y, g.s2)
        assert np.array_equal(grp.approx_logl_sine(sg, spec, theta), one.approx_logl_sine(s1, spec, theta))
        for a, b in zip(grp.approx_logl_sine_grad(sg, spec, theta), one.approx_logl_sine_grad(s1, spec, theta)):
            assert np.array_equal(a, b)
        s1.free()
    finally:
        grp.close()


@pytest.mark.gpu
def test_rank_limits_and_argument_checks(pb, ctx, golden_periodic):
    g = golden_periodic
    theta = np.ascontiguousarray(g.chain[:4, 2:11])
    ser = ctx.upload_series(g.t, g.y, g.s2)
    # value: ranks <= 64 (SHO J = 32); the first rank above, 66, is refused (2J and 3J never make 65)
    ctx.approx_logl_sine(ser, pb.make_spec(g.model, g.f_min, g.f_max, 32), theta)
    for basis, J in (("SHO", 33), ("DRWCelerite", 22)):
        with pytest.raises(pb.PioranError) as e:
            ctx.approx_logl_sine(ser, pb.make_spec(g.model, g.f_min, g.f_max, J, basis_function=basis), theta)
        assert e.value.code == -5
    # gradient: ranks <= 62; 63 (DRWCelerite J = 21) and 64 (SHO J = 32) are refused, and so is the scalar-pipe selection
    ctx.approx_logl_sine_grad(ser, pb.make_spec(g.model, g.f_min, g.f_max, 31), theta)
    for basis, J in (("DRWCelerite", 21), ("SHO", 32)):
        with pytest.raises(pb.PioranError) as e:
            ctx.approx_logl_sine_grad(ser, pb.make_spec(g.model, g.f_min, g.f_max, J, basis_function=basis), theta)
        assert e.value.code == -5
    spec = pb.make_spec(g.model, g.f_min, g.f_max, 20)
    ctx.set_sweep_kernel("scalar")
    try:
        with pytest.raises(pb.PioranError) as e:
            ctx.approx_logl_sine_grad(ser, spec, theta)
        assert e.value.code == -5
    finally:
        ctx.set_sweep_kernel("auto")
    # argument errors: PIORAN_EINVAL
    dp = C.POINTER(C.c_double)
    th, out, grad = theta.copy(), np.empty(4), np.empty((4, 9))
    p = lambda x: x.ctypes.data_as(dp)
    lib, h = ctx.lib, ctx.h
    assert lib.pioran_approx_logl_sine(h, ser.id, C.byref(spec), 0, p(th), p(out)) == -1
    assert lib.pioran_approx_logl_sine(h, ser.id, C.byref(spec), 4, None, p(out)) == -1
    assert lib.pioran_approx_logl_sine(h, ser.id, C.byref(spec), 4, p(th), None) == -1
    assert lib.pioran_approx_logl_sine(h, 987654, C.byref(spec), 4, p(th), p(out)) == -1
    assert lib.pioran_approx_logl_sine_grad(h, ser.id, C.byref(spec), 0, p(th), p(out), p(grad)) == -1
    assert lib.pioran_approx_logl_sine_grad(h, ser.id, C.byref(spec), 4, p(th), p(out), None) == -1
    assert lib.pioran_approx_logl_sine_grad(h, 987654, C.byref(spec), 4, p(th), p(out), p(grad)) == -1
    bad = pb.make_spec(g.model, g.f_min, g.f_max, 20)
    bad.psd_model = 7
    assert lib.pioran_approx_logl_sine(h, ser.id, C.byref(bad), 4, p(th), p(out)) == -1
    assert lib.pioran_approx_logl_sine_grad(h, ser.id, C.byref(bad), 4, p(th), p(out), p(grad)) == -1
    with pytest.raises(ValueError):
        ctx.approx_logl_sine(ser, spec, theta[:, :8])
    with pytest.raises(ValueError):
        ctx.approx_logl_sine_grad(ser, spec, theta[:, :6])
    ser.free()


# ------------------------------------------------------------------------------------------------- Python interface
@pytest.mark.gpu
def test_batched_likelihood_periodic_mean(pb, ctx, golden_periodic):
    g = golden_periodic
    theta = np.ascontiguousarray(g.chain[::331, 2:11])
    like = pb.BatchedLikelihood(g.t, g.y, g.s2, g.model, 20, "SHO", ctx=ctx, periodic_mean=True)
    assert like.n_par == 9
    assert np.array_equal(like(theta), ctx.approx_logl_sine(like.series, like.spec, theta))
    v, gr = like.value_and_gradient(theta)
    v2, g2 = ctx.approx_logl_sine_grad(like.series, like.spec, theta)
    assert np.array_equal(v, v2) and np.array_equal(gr, g2) and np.array_equal(like.gradient(theta), g2)
    assert rel_err(like(theta), g.chain[::331, 1]).max() <= TOL
    like.close()
    dbpl = pb.BatchedLikelihood(g.t, g.y, g.s2, "DoubleBendingPowerLaw", 20, "SHO", ctx=ctx, periodic_mean=True)
    assert dbpl.n_par == 11
    dbpl.close()
    # vectorized_callbacks with the periodic mean and a caller's prior over all nine columns
    lo, hi = theta.min(axis=0), theta.max(axis=0)
    loglike, transform, close = pb.sampler.vectorized_callbacks(g.t, g.y_raw, g.yerr, log_transform=False, ctx=ctx,
                                                                periodic_mean=True, prior=lambda u: lo + u * (hi - lo))
    cube = np.random.default_rng(2).uniform(size=(16, 9))
    th = transform(cube)
    want = pb.BatchedLikelihood(g.t, g.y, g.s2, g.model, 20, "SHO", ctx=ctx, periodic_mean=True)
    ref = want(th)
    ref[~np.isfinite(ref)] = -1e300
    assert np.array_equal(loglike(th), ref)
    want.close()
    close()


def test_periodic_mean_combinations_are_refused(pb):
    """No device is touched: the combinations are refused before any upload."""
    t = np.linspace(0.0, 10.0, 20)
    y, s2 = np.ones(20), np.full(20, 0.01)
    with pytest.raises(ValueError):
        pb.BatchedLikelihood(t, y, s2, periodic_mean=True, log_shift=True)
    with pytest.raises(ValueError):
        pb.BatchedLikelihood(t, y, s2, periodic_mean=True, n_features=1)
    with pytest.raises(ValueError):
        pb.sampler.vectorized_callbacks(t, y, np.full(20, 0.1), periodic_mean=True)
    with pytest.raises(ValueError):
        pb.sampler.vectorized_callbacks(t, y, np.full(20, 0.1), periodic_mean=True, prior=lambda u: u, device_prior=True)
