"""Device groups (pioran_ctx_create_multi, include/pioran_b200.h): one process, one context over several GPUs — what a sampler
that is a single process with one callback needs (reference: examples/ultranest/single_pl.jl:113-117).  A group of one device
exercises the whole forwarding layer on the single-GPU box; the two-device case runs where two GPUs are visible."""
import numpy as np
import pytest

from conftest import prior_theta, rel_err, synthetic_series

pytestmark = pytest.mark.gpu


def _ndev():
    import ctypes
    try:
        rt = ctypes.CDLL("libcudart.so")
    except OSError:
        import torch
        return torch.cuda.device_count()
    n = ctypes.c_int(0)
    rt.cudaGetDeviceCount(ctypes.byref(n))
    return n.value


@pytest.mark.parametrize("devices", [[0], [0, 1]])
def test_group_context_matches_single_device(devices):
    import pioran_b200 as pb
    if len(devices) > _ndev():
        pytest.skip("needs %d GPUs" % len(devices))
    one = pb.get_context(0)
    grp = pb.Context(devices)
    assert grp.device_count == len(devices)
    try:
        t, y, s2, f_min, f_max = synthetic_series(700, 3)
        th = prior_theta(1001, f_min, f_max, y.mean(), y.std(), 11, alpha2_max=3.5)
        for basis in ("SHO", "DRWCelerite"):
            spec = pb.make_spec("SingleBendingPowerLaw", f_min, f_max, 20, basis_function=basis)
            s1, sg = one.upload_series(t, y, s2), grp.upload_series(t, y, s2)
            want = one.approx_logl(s1, spec, th)[0]
            got = grp.approx_logl(sg, spec, th)[0]
            assert np.array_equal(got, want), basis           # same kernels, same inputs per row
            # gradients and explicit coefficients split the same way
            lw, gw = one.approx_logl_grad(s1, spec, th[:37])
            lg, gg = grp.approx_logl_grad(sg, spec, th[:37])
            assert np.array_equal(lg, lw) and np.array_equal(gg, gw)
            a, b, c, d = grp.approx_coeffs(spec, th[:53, :4])
            assert np.array_equal(grp.celerite_logl(sg, a, b, c, d, mu=th[:53, 5], nu=th[:53, 4]),
                                  one.celerite_logl(s1, a, b, c, d, mu=th[:53, 5], nu=th[:53, 4]))
            # the dense cross-check splits its parameter vectors the same way
            a9, b9, c9, d9 = grp.approx_coeffs(spec, th[:9, :4])
            nw, iw = one.direct_logl(s1, a9, b9, c9, d9, mu=th[:9, 5], nu=th[:9, 4])
            ng, ig = grp.direct_logl(sg, a9, b9, c9, d9, mu=th[:9, 5], nu=th[:9, 4])
            assert np.array_equal(ng, nw) and np.array_equal(ig, iw)
            s1.free(); sg.free()
        # several series in one call
        sers1, sersg, specs = [], [], []
        for k in range(3):
            tk, yk, sk, fm, fx = synthetic_series(200 + 37 * k, 20 + k)
            sers1.append(one.upload_series(tk, yk, sk)); sersg.append(grp.upload_series(tk, yk, sk))
            specs.append(pb.make_spec("SingleBendingPowerLaw", fm, fx, 12))
        want = one.approx_logl(sers1, specs, th[:101])
        got = grp.approx_logl(sersg, specs, th[:101])
        assert got.shape == (3, 101) and np.array_equal(got, want)
        # device-pointer entries and stream injection need a single-device context
        with pytest.raises(pb.PioranError) as e:
            grp.set_stream(0x1234)
        assert e.value.code == -5
        with pytest.raises(pb.PioranError):
            grp.approx_logl(pb.backend.Series(grp, 99, 10), specs[0], th[:4])      # unknown series id
    finally:
        grp.close()


def _features_theta(rng, B, f_min, f_max, nf):
    cols = [rng.uniform(0.0, 1.0, B), np.exp(rng.uniform(np.log(f_min), np.log(f_max), B)), rng.uniform(2.0, 3.5, B),
            np.exp(rng.normal(-1, 0.5, B)), rng.gamma(2, 0.5, B), rng.normal(0, 0.3, B)]
    for _ in range(nf):
        cols += [rng.uniform(0.5, 3, B), np.exp(rng.uniform(np.log(2 * f_min), np.log(f_max / 2), B)), rng.uniform(1.0, 15, B)]
    return np.column_stack(cols)


def _same(got, want, what):
    if isinstance(want, (tuple, list)):
        assert len(got) == len(want), what
        for k, (g, w) in enumerate(zip(got, want)):
            _same(g, w, f"{what}[{k}]")
    elif isinstance(want, dict):
        for k in want:
            _same(got[k], want[k], f"{what}[{k}]")
    else:
        assert np.array_equal(got, want), what


@pytest.mark.parametrize("devices", [[0], [0, 1]])
def test_group_entries_match_single_device(devices):
    """Every entry with a group branch gives the single-device result bit for bit: the splitting entries on every slice
    (per-row data and data tangents sliced by the series length), the entries that run on the first device, and the
    setters, which must reach every child."""
    import pioran_b200 as pb
    if len(devices) > _ndev():
        pytest.skip("needs %d GPUs" % len(devices))
    one = pb.get_context(0)
    grp = pb.Context(devices)
    rng = np.random.default_rng(17)
    try:
        t, y, s2, f_min, f_max = synthetic_series(700, 3)
        N = t.size
        th = prior_theta(37, f_min, f_max, y.mean(), y.std(), 11, alpha2_max=3.5)
        B = th.shape[0]
        s1, sg = one.upload_series(t, y, s2), grp.upload_series(t, y, s2)
        for basis in ("SHO", "DRWCelerite"):
            spec = pb.make_spec("SingleBendingPowerLaw", f_min, f_max, 20, basis_function=basis)

            def both(name, *args, **kw):
                want = getattr(one, name)(s1, *args, **kw)
                got = getattr(grp, name)(sg, *args, **kw)
                _same(got, want, f"{basis} {name}")

            # fused path
            th_ls = np.column_stack([th, y.min() - rng.uniform(0.5, 2.0, B)])
            both("approx_logl_logshift", spec, th_ls)
            both("approx_logl_logshift_grad", spec, th_ls)
            prior = pb.sampler.single_bending_power_law_prior(f_min, f_max, float(y.mean()), float(y.var()), alpha2_max=3.5)
            both("prior_transform_logl", spec, prior.device_spec(), rng.uniform(size=(B, 6)), return_theta=True)
            # PSD features
            for nf in (1, 2):
                thf = _features_theta(rng, 23, f_min, f_max, nf)
                both("approx_features_logl", spec, nf, thf)
                both("approx_features_logl_grad", spec, nf, thf)
                both("approx_features_logl_grad_reverse", spec, nf, thf)
            # explicit coefficients with per-θ data, data tangents and data gradients
            a, b, c, d = one.approx_coeffs(spec, th[:, :4])
            mu, nu = th[:, 5], th[:, 4]
            yb = y + rng.normal(0, 0.1, (B, N))
            sb = s2 * rng.uniform(0.5, 2.0, (B, N))
            both("celerite_logl", a, b, c, d, mu=mu, nu=nu, y_batch=yb, s2_batch=sb)
            P, Jt = 2, a.shape[1]
            tan = {k: rng.normal(size=(B, P, Jt)) for k in ("da", "db", "dc", "dd")}
            both("celerite_logl_jvp", a, b, c, d, mu=mu, nu=nu, y_batch=yb, s2_batch=sb, dmu=rng.normal(size=(B, P)),
                 dnu=rng.normal(size=(B, P)), dy=rng.normal(size=(B, P, N)), ds2=rng.normal(size=(B, P, N)), **tan)
            both("celerite_logl_vjp", a, b, c, d, mu=mu, nu=nu, y_batch=yb, s2_batch=sb, data_grad=True)
            # the single-device work of a group runs on its first device
            tau = np.sort(rng.uniform(t[0] - 5, t[-1] + 5, 90))
            both("celerite_predict", a[:9], b[:9], c[:9], d[:9], tau, mu=mu[:9], nu=nu[:9])
            both("celerite_predict_var", a[:9], b[:9], c[:9], d[:9], tau, mu=mu[:9], nu=nu[:9])
            both("celerite_simulate", a[:9], b[:9], c[:9], d[:9], rng.normal(size=(9, N)), nu=nu[:9])
            both("celerite_logl_scan", a[:3], b[:3], c[:3], d[:3], mu=mu[:3], nu=nu[:3])
            for ctx, ser in ((one, s1), (grp, sg)):
                ctx.scan_range_begin(ser, a[0], b[0], c[0], d[0], 0, N // 2, mu=mu[0], nu=nu[0])
            _same(grp.scan_range_end(None), one.scan_range_end(None), f"{basis} scan_range_end")
        s1.free(); sg.free()
        # a setter applied to a group reaches every child: with the automatic scan routing off, one evaluation of a long series
        # runs the sequential sweep on whichever device its slice lands on
        t, y, s2, f_min, f_max = synthetic_series(8192, 4)
        s1, sg = one.upload_series(t, y, s2), grp.upload_series(t, y, s2)
        spec = pb.make_spec("SingleBendingPowerLaw", f_min, f_max, 20)
        a, b, c, d = one.approx_coeffs(spec, th[:1, :4])
        for ctx in (one, grp):
            ctx.set_auto_scan(False)
        got = grp.celerite_logl(sg, a, b, c, d, mu=th[:1, 5], nu=th[:1, 4])
        want = one.celerite_logl(s1, a, b, c, d, mu=th[:1, 5], nu=th[:1, 4])
        assert not one.last_kernel_name().startswith("scan")
        _same(got, want, "celerite_logl without the scan routing")
        s1.free(); sg.free()
    finally:
        one.set_auto_scan(True)
        grp.close()


def test_resident_time_vector_drop_in():
    """log_likelihood(cov, τ, y, σ²; solver = :celerite_gpu) keeps τ on the device between calls (julia/b200_solver.jl:
    b200_resident_series; Python mirror api._resident_series): the second call uploads only y and σ²."""
    import pioran_b200 as pb
    from oracle import oracle as orc
    t, y, s2, f_min, f_max = synthetic_series(300, 5)
    cov = pb.approx(pb.SingleBendingPowerLaw(0.6, 0.02, 3.1), f_min, f_max, 20, 1.3, basis_function="DRWCelerite")
    a, b, c, d = pb.celerite_coefs(cov)
    pb.api.release_resident_series()
    for k, (mu, nu) in enumerate(((0.0, 1.0), (0.3, 1.7), (-0.2, 0.6))):
        got = pb.log_likelihood(cov, t, y - mu, nu * s2, solver="celerite_gpu")
        want = orc.celerite_logl(a, b, c, d, t, y - mu, nu * s2)
        assert rel_err(got, want) <= 1e-9
        assert len(pb.api._resident) == 1
    assert rel_err(pb.log_likelihood(cov, t, y, s2, solver=":celerite_matrix"), orc.celerite_logl(a, b, c, d, t, y, s2)) <= 1e-9
    pb.api.release_resident_series()
    assert len(pb.api._resident) == 0
