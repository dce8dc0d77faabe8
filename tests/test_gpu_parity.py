"""GPU parity tests proper (run with -m gpu on a B200): every value goes through the C ABI of
libpioran_b200.so and is compared with the CPU oracle, the reference's golden chains, or a size-independent
property.  Tolerance: BASELINE.json north_star — ≤ 1e-9 relative on logL in FP64 (|Δ|/max(1,|logL|))."""
import os

import numpy as np
import pytest

from conftest import GOLDEN, assert_parity, periodic_mean, prior_theta, rel_err, synthetic_series
from oracle import oracle as orc

pytestmark = pytest.mark.gpu
TOL = 1e-9


@pytest.fixture(scope="module")
def pb():
    import pioran_b200
    return pioran_b200


@pytest.fixture(scope="module")
def ctx(pb):
    return pb.get_context(0)


# ------------------------------------------------------------------------------------------------- K1
@pytest.mark.parametrize("basis", ["SHO", "DRWCelerite"])
@pytest.mark.parametrize("integrated", [True, False])
def test_k1_coefficients_vs_oracle(pb, ctx, golden_single, basis, integrated):
    g = golden_single
    th = g.theta[::37, :4].copy()
    if basis == "DRWCelerite":
        th[:, 2] += 1.5  # DRWCelerite allows α₂ up to 6
    spec = pb.make_spec(g.model, g.f_min, g.f_max, 20, is_integrated_power=integrated, basis_function=basis)
    a, b, c, d = ctx.approx_coeffs(spec, th)
    for i in range(len(th)):
        oa, ob, oc, od = orc.approx("SBPL", th[i, :3], g.f_min, g.f_max, 20, th[i, 3], is_integrated_power=integrated,
                                    basis=basis)
        scale = np.abs(oa).max()
        assert np.max(np.abs(a[i] - oa)) <= 1e-12 * scale
        assert np.max(np.abs(b[i] - ob)) <= 1e-12 * scale
        assert np.allclose(c[i], oc, rtol=1e-14) and np.allclose(d[i], od, rtol=1e-14)


def test_k1_golden_amplitudes_and_variance(pb, ctx):
    """test/test_psd.jl:38 via the coefficient formula a = A·f·π/√2, and Σa = va (test/test_psd.jl:114,141)."""
    from test_oracle import A1, A2_DRW, A2_SHO, F1, GOLD_AMPLITUDES, VARS
    f0, fM, J = 0.02, 1.52e2, 20
    spec = pb.make_spec("SingleBendingPowerLaw", f0 * 20, fM / 20, J, is_integrated_power=False)
    a, b, c, d = ctx.approx_coeffs(spec, np.array([[0.3, 0.02, 2.93, 1.0]]))
    fj = c[0] / (np.sqrt(2) * np.pi)
    amp = a[0] / (fj * np.pi / np.sqrt(2))
    # with is_integrated_power=false the amplitudes are the golden ones up to the common factor 1/Σ(A f)π/√2
    ratio = amp / GOLD_AMPLITUDES
    assert np.max(np.abs(ratio / ratio[0] - 1)) < 1e-11
    for basis, a2 in (("SHO", A2_SHO), ("DRWCelerite", A2_DRW)):
        spec = pb.make_spec("SingleBendingPowerLaw", 2.0e-3, 3.52e2, 25, is_integrated_power=False, basis_function=basis)
        th = np.column_stack([A1, F1, a2, VARS])
        a, b, c, d = ctx.approx_coeffs(spec, th)
        assert a.shape[1] == (25 if basis == "SHO" else 50)
        assert np.max(np.abs(a.sum(axis=1) / np.array(VARS) - 1)) < 1e-12


def test_api_mirror_approx_and_logpdf(pb, golden_single):
    """The reference-facing calls: approx → ScalableGP → logpdf, checked on the run's maximum-likelihood point."""
    import json
    g = golden_single
    with open(os.path.join(GOLDEN, "simu_single_maximum_likelihood.json")) as fh:
        ml = json.load(fh)
    α1, f1, α2, variance, ν, μ = ml["point"]
    P = pb.SingleBendingPowerLaw(α1, f1, α2)
    R = pb.approx(P, g.f_min, g.f_max, 20, variance, basis_function="SHO")
    assert isinstance(R, pb.SumOfCelerite) and len(R.a) == 20
    f = pb.ScalableGP(μ, R)
    val = pb.logpdf(f(g.t, ν * g.s2), g.y)
    assert abs(val - ml["logl"]) <= TOL * abs(ml["logl"])
    assert abs(pb.log_likelihood(R, g.t, g.y - μ, ν * g.s2) - val) <= 1e-12 * abs(val)


def _ld_twin(model, f_min, f_max, J, basis, t, y, s2):
    """row θ = [psd…, norm, ν, μ] → 80-bit evaluation of the same likelihood (oracle, conditioning triage only)."""
    npar = 3 if model == "SBPL" else 5

    def f(th):
        a, b, c, d = orc.approx(model, th[:npar], f_min, f_max, J, th[npar], basis=basis)
        return orc.celerite_logl(a, b, c, d, t, y - th[npar + 2], th[npar + 1] * s2, long_double=True)
    return f


# ------------------------------------------------------------------------------------------------- K2 vs golden chains
def _assert_chain(got, ref):
    r = rel_err(got, ref)
    assert np.all(np.isfinite(got))
    assert r.max() <= TOL, f"max rel {r.max():.3e} at row {int(r.argmax())}"
    assert np.median(r) < 1e-13


def test_fused_vs_chain_single(pb, ctx, golden_single):
    """All 6 475 (θ, logL) pairs of examples/ultranest/inference/simu_single (SHO J=20, N=485)."""
    g = golden_single
    like = pb.BatchedLikelihood(g.t, g.y, g.s2, g.model, 20, "SHO", ctx=ctx)
    _assert_chain(like(g.theta), g.logl)


def test_fused_vs_chain_double(pb, ctx, golden_double):
    """All 6 542 pairs of simu_double (DoubleBendingPowerLaw)."""
    g = golden_double
    like = pb.BatchedLikelihood(g.t, g.y, g.s2, g.model, 20, "SHO", ctx=ctx)
    _assert_chain(like(g.theta), g.logl)


def test_generic_vs_chain_periodic(pb, ctx, golden_periodic):
    """All 8 480 pairs of simu_periodic_rednoise: per-θ sinusoidal mean → y_batch on the generic path."""
    g = golden_periodic
    spec = pb.make_spec(g.model, g.f_min, g.f_max, 20)
    ser = ctx.upload_series(g.t, g.y, g.s2)
    a, b, c, d = ctx.approx_coeffs(spec, g.theta[:, :4])
    yb = np.stack([g.y - periodic_mean(g.t, row) for row in g.chain])
    got = ctx.celerite_logl(ser, a, b, c, d, nu=g.theta[:, 4], y_batch=yb)
    _assert_chain(got, g.logl)


def test_generic_equals_fused(pb, ctx, golden_single):
    g = golden_single
    sub = g.theta[::13]
    spec = pb.make_spec(g.model, g.f_min, g.f_max, 20)
    ser = ctx.upload_series(g.t, g.y, g.s2)
    fused = ctx.approx_logl(ser, spec, sub)[0]
    a, b, c, d = ctx.approx_coeffs(spec, sub[:, :4])
    gen = ctx.celerite_logl(ser, a, b, c, d, mu=sub[:, 5], nu=sub[:, 4])
    assert rel_err(gen, fused).max() < 1e-10


# ------------------------------------------------------------------------------------------------- K2 vs oracle
@pytest.mark.parametrize("basis,J", [("SHO", 20), ("DRWCelerite", 20), ("SHO", 30), ("SHO", 16), ("DRWCelerite", 12),
                                     ("SHO", 25), ("SHO", 32)])
def test_fused_vs_oracle_bases(pb, ctx, golden_single, basis, J):
    """Every compiled block size (R = 2J or 3J → BS 4…8), both bases; DRWCelerite logL has no literal in the
    reference, so it is pinned through the oracle (itself pinned by celerite ≡ dense)."""
    g = golden_single
    sub = g.theta[::97].copy()
    if basis == "DRWCelerite":
        sub[:, 2] += 1.0
    spec = pb.make_spec(g.model, g.f_min, g.f_max, J, basis_function=basis)
    ser = ctx.upload_series(g.t, g.y, g.s2)
    got = ctx.approx_logl(ser, spec, sub)[0]
    want = orc.approx_logl_batch("SBPL", sub, g.f_min, g.f_max, J, g.t, g.y, g.s2, basis=basis, nthreads=0)
    assert np.median(rel_err(got, want)) < 1e-12
    assert_parity(got, want, sub, _ld_twin("SBPL", g.f_min, g.f_max, J, basis, g.t, g.y, g.s2), TOL)


@pytest.mark.parametrize("N", [1, 2, 3, 15, 16, 17, 31, 32, 33, 100])
def test_small_and_ragged_lengths(pb, ctx, N):
    """Edge lengths around the 16-step TMA chunk and the 32-step log-ring, and the N=1 / N=2 corner cases."""
    rng = np.random.default_rng(N)
    t = np.cumsum(rng.uniform(0.1, 2.0, N))
    y = rng.normal(size=N)
    s2 = rng.uniform(0.01, 0.1, N)
    f_min, f_max = 1e-3, 5.0
    th = prior_theta(5, f_min, f_max, 0.0, 1.0, seed=N)
    spec = pb.make_spec("SingleBendingPowerLaw", f_min, f_max, 20)
    ser = ctx.upload_series(t, y, s2)
    got = ctx.approx_logl(ser, spec, th)[0]
    want = orc.approx_logl_batch("SBPL", th, f_min, f_max, 20, t, y, s2)
    assert rel_err(got, want).max() <= TOL
    a, b, c, d = ctx.approx_coeffs(spec, th[:, :4])
    gen = ctx.celerite_logl(ser, a, b, c, d, mu=th[:, 5], nu=th[:, 4])
    assert rel_err(gen, want).max() <= TOL


def test_generic_raw_coefficients_reference_benchmark_shape(pb, ctx):
    """benchmark/benchmarks.jl:76-91 shape: a = 5·U(0,1), b, c, d ~ U(0,1) raw coefficients, J_t ∈ {2…32}."""
    rng = np.random.default_rng(7)
    N = 200
    t = np.sort(rng.uniform(0, 100, N))
    y = rng.normal(size=N)
    s2 = rng.uniform(0.5, 1.0, N)
    ser = ctx.upload_series(t, y, s2)
    for Jt in (2, 4, 8, 16, 20, 32):
        B = 6
        a = 5 * rng.uniform(size=(B, Jt)); b = rng.uniform(size=(B, Jt)) * 0.2
        c = rng.uniform(size=(B, Jt)); d = rng.uniform(size=(B, Jt))
        got = ctx.celerite_logl(ser, a, b, c, d)
        want = orc.celerite_logl_batch(a, b, c, d, t, y, s2)
        assert rel_err(got, want).max() <= TOL, Jt


def test_real_terms_rank_reduction_and_carma_like_signs(pb, ctx):
    """Real terms (b=d=0) take one row; negative a/b/d coefficients (test/test_carma.jl:51-69 has such sets)."""
    rng = np.random.default_rng(3)
    N = 150
    t = np.cumsum(rng.uniform(0.2, 1.5, N)); y = rng.normal(size=N); s2 = np.full(N, 0.3)
    ser = ctx.upload_series(t, y, s2)
    a = np.array([[1.2, 0.8, -0.3, 0.5], [2.0, 0.1, -0.05, 1.0]])
    b = np.array([[0.0, 0.3, -0.1, 0.0], [0.0, -0.05, 0.02, 0.0]])
    c = np.array([[0.3, 0.2, 1.0, 2.0], [0.1, 0.5, 0.8, 3.0]])
    d = np.array([[0.0, 1.5, -2.0, 0.0], [0.0, 0.7, 1.1, 0.0]])
    got = ctx.celerite_logl(ser, a, b, c, d)
    want = orc.celerite_logl_batch(a, b, c, d, t, y, s2)
    assert rel_err(got, want).max() <= TOL


def test_nonfinite_semantics_match_reference(pb, ctx):
    """Negative first pivot → NaN (log without abs, celerite_solver.jl:126); indefinite later pivots stay finite."""
    t = np.array([0.0, 1.0, 2.5, 3.0]); y = np.array([0.1, -0.2, 0.3, 0.0]); s2 = np.full(4, 1e-2)
    ser = ctx.upload_series(t, y, s2)
    a = np.array([[-1.0, 0.0], [2.0, -1.5]]); b = np.zeros((2, 2))
    c = np.array([[0.5, 1.0], [0.1, 5.0]]); d = np.zeros((2, 2))
    got = ctx.celerite_logl(ser, a, b, c, d)
    want = orc.celerite_logl_batch(a, b, c, d, t, y, s2)
    assert np.isnan(got[0]) and np.isnan(want[0])
    assert np.isfinite(got[1]) and rel_err(got[1], want[1]) <= TOL


def test_multi_series_ragged(pb, ctx):
    """Config C3 in small: ragged series × per-series parameter batches in ONE call."""
    S, B = 5, 7
    sers, specs, want = [], [], []
    thetas = np.empty((S, B, 6))
    for s in range(S):
        t, y, s2, f_min, f_max = synthetic_series(60 + 37 * s, seed=2000 + s)
        th = prior_theta(B, f_min, f_max, y.mean(), y.std(), seed=s)
        thetas[s] = th
        sers.append(ctx.upload_series(t, y, s2))
        specs.append(pb.make_spec("SingleBendingPowerLaw", f_min, f_max, 20))
        want.append(orc.approx_logl_batch("SBPL", th, f_min, f_max, 20, t, y, s2))
    got = ctx.approx_logl(sers, specs, thetas, theta_per_series=True)
    assert got.shape == (S, B)
    assert rel_err(got, np.array(want)).max() <= TOL


def test_permutation_and_split_invariance(pb, ctx, golden_single):
    """Size-independent property: a row's value does not depend on its batch position or the batch split."""
    g = golden_single
    like = pb.BatchedLikelihood(g.t, g.y, g.s2, g.model, 20, "SHO", ctx=ctx)
    th = g.theta[:1000]
    full = like(th)
    perm = np.random.default_rng(0).permutation(len(th))
    assert np.array_equal(like(th[perm]), full[perm])
    parts = np.concatenate([like(th[:333]), like(th[333:334]), like(th[334:])])
    assert np.array_equal(parts, full)


@pytest.mark.parametrize("basis", ["SHO", "DRWCelerite"])
def test_dispatch_tiers_agree(pb, ctx, golden_single, basis):
    """The same rows through the tensor-pipe kernels the default dispatch picks as the batch grows (csrc/api.cu
    approx_logl_dev_locked): one 4-warp CTA per evaluation (blocked_wide, ≤ 296 evaluations), then the warp kernel (blocked)
    with 4-warp CTAs (≤ 592), 8-warp CTAs (≤ 1 184) and the full-size CTA.  Each batch is compared with the rows of the full
    batch, i.e. with the same kernel family; the scalar-pipe tiers of dispatch_shared and the oracle parity of every tier are
    in test_gpu_sweep_matrix.py."""
    g = golden_single
    like = pb.BatchedLikelihood(g.t, g.y, g.s2, g.model, 20, basis, ctx=ctx)
    th = g.theta[:3000].copy()
    if basis == "DRWCelerite":
        th[:, 2] += 1.0
    full = like(th)                    # full-size CTAs
    for B in (1, 7, 592, 593, 1184, 1185):
        part = like(th[:B])
        assert rel_err(part, full[:B]).max() <= 1e-12, (basis, B)
    like.close()


# ------------------------------------------------------------------------------------------------- BASELINE sizes
def test_config_c1_single_n1000_drw(pb, ctx):
    """BASELINE configs[0]: single logpdf, approx(SBPL, J=20, DRWCelerite) on a simulated N=1000 irregular series."""
    t, y, s2, f_min, f_max = synthetic_series(1000, seed=1234, basis="DRWCelerite")
    P = pb.SingleBendingPowerLaw(0.82, 0.01, 3.3)
    R = pb.approx(P, f_min, f_max, 20, 1.0, basis_function="DRWCelerite", ctx=ctx)
    assert len(R.a) == 40
    val = pb.logpdf(pb.ScalableGP(0.0, R)(t, s2), y, ctx=ctx)
    a, b, c, d = orc.approx("SBPL", [0.82, 0.01, 3.3], f_min, f_max, 20, 1.0, basis="DRWCelerite")
    want = orc.celerite_logl(a, b, c, d, t, y, s2)
    assert rel_err(val, want) <= TOL


def test_config_c2_full_size_subset_vs_oracle(pb, ctx):
    """BASELINE configs[1] at full size: 4 096 θ × N=10 000, DRWCelerite J=20.  All rows are evaluated on the GPU;
    a seeded subset is checked against the oracle, the rest through permutation invariance."""
    t, y, s2, f_min, f_max = synthetic_series(10000, seed=1235, basis="DRWCelerite")
    th = prior_theta(4096, f_min, f_max, y.mean(), y.std(), seed=42, alpha2_max=6.0)
    like = pb.BatchedLikelihood(t, y, s2, "SingleBendingPowerLaw", 20, "DRWCelerite", ctx=ctx)
    got = like(th)
    assert got.shape == (4096,) and np.isfinite(got).mean() > 0.99
    idx = np.random.default_rng(1).choice(4096, 24, replace=False)
    want = orc.approx_logl_batch("SBPL", th[idx], f_min, f_max, 20, t, y, s2, basis="DRWCelerite", nthreads=0)
    assert_parity(got[idx], want, th[idx], _ld_twin("SBPL", f_min, f_max, 20, "DRWCelerite", t, y, s2), TOL)
    perm = np.random.default_rng(2).permutation(4096)
    assert np.array_equal(like(th[perm]), got[perm], equal_nan=True)


def test_config_c3_multi_source_full_size(pb, ctx):
    """BASELINE configs[2] at full size on one GPU: 512 light curves (N ≈ 2 000, ragged) × 400 parameter vectors each,
    SHO J = 20 — one fused call over all series (per-series θ and f_min/f_max).  A seeded subset is checked against the
    oracle; single-series calls must reproduce the batched values bit for bit (work-item independence)."""
    import workloads as wl
    rng = np.random.default_rng(2000)
    S, B = 512, 400
    lengths = np.clip(np.rint(rng.normal(2000, 300, S)), 1000, 3000).astype(int)
    series, specs, thetas, raw = [], [], [], []
    for s in range(S):
        t, y, s2, f_min, f_max = wl.make_series_fast(int(lengths[s]), seed=2000 + s)
        raw.append((t, y, s2, f_min, f_max))
        series.append(ctx.upload_series(t, y, s2))
        specs.append(pb.make_spec("SingleBendingPowerLaw", f_min, f_max, 20))
        thetas.append(prior_theta(B, f_min, f_max, y.mean(), y.std(), seed=5000 + s))
    theta = np.stack(thetas)
    got = ctx.approx_logl(series, specs, theta, theta_per_series=True)
    assert got.shape == (S, B) and np.isfinite(got).mean() > 0.99
    for s in rng.choice(S, 6, replace=False):
        t, y, s2, f_min, f_max = raw[s]
        idx = rng.choice(B, 4, replace=False)
        want = orc.approx_logl_batch("SBPL", theta[s, idx], f_min, f_max, 20, t, y, s2, nthreads=0)
        assert_parity(got[s, idx], want, theta[s, idx], _ld_twin("SBPL", f_min, f_max, 20, "SHO", t, y, s2), TOL)
        single = ctx.approx_logl(series[s], specs[s], theta[s])[0]
        assert np.array_equal(single, got[s], equal_nan=True)
    for ser in series:
        ser.free()


@pytest.mark.parametrize("basis,J,B", [("SHO", 20, 37), ("DRWCelerite", 20, 5), ("SHO", 12, 700)])
def test_log_shift_fused_entry_vs_oracle(pb, ctx, basis, J, B):
    """Log-normally distributed series (docs/src/timeseries.md:16-21; likelihood of docs/src/ultranest.md:197-217):
    yn = log(y − c), σ² = ν σ²/(y − c)² per parameter vector.  The fused entry transforms on the device; the oracle gets the
    transformed arrays row by row.  Also: the same numbers through the generic entry's host-side y_batch / s2_batch, and NaN
    where y − c ≤ 0 (the reference's log throws DomainError)."""
    t, y, s2, f_min, f_max = synthetic_series(300, seed=77)
    flux = np.exp(0.4 * y) + 0.3                      # positive series
    sig2 = s2 * flux ** 2
    rng = np.random.default_rng(B)
    theta = np.empty((B, 7))
    theta[:, 0] = rng.uniform(0.0, 1.25, B)
    theta[:, 1] = np.exp(rng.uniform(np.log(f_min), np.log(f_max), B))
    theta[:, 2] = theta[:, 0] + rng.uniform(size=B) * (4.0 - theta[:, 0])
    theta[:, 3] = np.exp(rng.normal(-3.0, 1.0, B))
    theta[:, 4] = rng.gamma(2.0, 0.5, B)
    theta[:, 5] = rng.normal(np.log(flux).mean(), 0.5, B)
    theta[:, 6] = np.exp(rng.uniform(np.log(1e-6), np.log(flux.min() * 0.99), B))
    spec = pb.make_spec("SingleBendingPowerLaw", f_min, f_max, J, basis_function=basis)
    ser = ctx.upload_series(t, flux, sig2)
    got = ctx.approx_logl_logshift(ser, spec, theta)
    rows = np.unique(np.concatenate([[0, B - 1], rng.choice(B, size=min(B, 6), replace=False)]))
    for i in rows:
        yn = np.log(flux - theta[i, 6])
        s2n = sig2 / (flux - theta[i, 6]) ** 2
        want = orc.approx_logl_batch("SBPL", theta[i:i + 1, :6], f_min, f_max, J, t, yn, s2n, basis=basis)[0]
        if rel_err(got[i], want) > TOL:     # ill-conditioned draw: no farther from the 80-bit value than 4× the reference order
            a_, b_, c_, d_ = orc.approx("SBPL", theta[i, :3], f_min, f_max, J, theta[i, 3], basis=basis)
            ld = orc.celerite_logl(a_, b_, c_, d_, t, yn - theta[i, 5], theta[i, 4] * s2n, long_double=True)
            assert rel_err(got[i], ld) <= 4 * rel_err(want, ld), (i, got[i], want, ld)
    # generic entry with host-transformed per-θ data: same sweep, explicit coefficients
    sub = rows[:4]
    a, b, c, d = ctx.approx_coeffs(spec, theta[sub, :4])
    yb = np.log(flux[None, :] - theta[sub, 6:7])
    sb = sig2[None, :] / (flux[None, :] - theta[sub, 6:7]) ** 2
    gen = ctx.celerite_logl(ser, a, b, c, d, mu=theta[sub, 5], nu=theta[sub, 4], y_batch=yb, s2_batch=sb)
    assert np.max(np.abs(gen - got[sub]) / np.maximum(1.0, np.abs(got[sub]))) <= TOL
    # c above the smallest flux: log of a negative number
    bad = theta[:2].copy()
    bad[1, 6] = flux.min() * 1.5
    out = ctx.approx_logl_logshift(ser, spec, bad)
    assert np.isfinite(out[0]) and np.isnan(out[1])
    with pytest.raises(ValueError):
        ctx.approx_logl_logshift(ser, spec, theta[:, :6])
    ser.free()


def test_carma_covariance_through_generic_entry(pb, ctx):
    """SURVEY 8f #4: a covariance with parameter-dependent decay rates and frequencies — the reference's CARMA(3, 2) literal
    of test/test_carma.jl:53-70 — through log_likelihood(cov::CARMA, …) (src/celerite_solver.jl:272-282): coefficients on the
    host, then the generic kernel (one complex term with a negative frequency and a real term with a negative amplitude: rank 3).
    Checked against the oracle's celerite recursion and its dense Cholesky; batched over roots drawn around the literal."""
    rα = np.array([-0.042163209825323775 + 1.1115603157767922j, -0.042163209825323775 - 1.1115603157767922j, -0.7599101571312047])
    β = [3.9413022090550216, 11.38193903188344, 1.0]
    t, y, s2, _, _ = synthetic_series(400, seed=9)
    cov = pb.CARMA(3, 2, rα, β, 1.3)
    got = pb.log_likelihood(cov, t, y, s2, ctx=ctx)
    a, b, c, d = pb.celerite_coefs(cov)
    want = orc.celerite_logl(a, b, c, d, t, y, s2)
    assert rel_err(got, want) <= TOL
    nll, info = orc.direct_nll(a, b, c, d, t, y, s2)
    assert info == 0 and rel_err(-nll, want) <= 1e-8                             # celerite ≡ dense for this covariance
    rng = np.random.default_rng(2)
    B = 64
    coefs = []
    for i in range(B):
        quad = np.array([1.2 * np.exp(rng.normal(0, 0.3)), 0.09 * np.exp(rng.normal(0, 0.3)), 0.76 * np.exp(rng.normal(0, 0.3))])
        coefs.append(pb.carma_celerite_coefs(3, pb.quad2roots(quad), β, np.exp(rng.normal(0, 0.5))))
    A, Bc, Cc, D = (np.stack([k[j] for k in coefs]) for j in range(4))
    ser = ctx.upload_series(t, y, s2)
    gotb = ctx.celerite_logl(ser, A, Bc, Cc, D)
    ser.free()
    wantb = orc.celerite_logl_batch(A, Bc, Cc, D, t, y, s2, nthreads=0)
    ok = np.isfinite(wantb)
    assert ok.sum() >= B // 2
    assert np.max(np.abs(gotb[ok] - wantb[ok]) / np.maximum(1.0, np.abs(wantb[ok]))) <= TOL
