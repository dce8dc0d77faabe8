"""K9 (csrc/lsp.cuh): generalised Lomb–Scargle periodograms through the C ABI and the Python interface, against the numpy
restatement tests/tools/proto/lsp_math.py (its 80-bit evaluation at ill-conditioned frequencies) on rows drawn by
pioran_celerite_simulate: every tile dimension with a ragged tail, weighted and unweighted; results that are the same bit for
bit under chunking, batch position, the resident y and device groups; invariances; NaN for 0/0; launches; argument checks;
and `lombscargle` of the Python interface against scipy."""
import ctypes as C
import os
import sys

import numpy as np
import pytest
from scipy import signal

from conftest import GOLDEN
from oracle import oracle as orc

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "tools", "proto"))
import lsp_math as lm  # noqa: E402

pytestmark = pytest.mark.gpu

TS = np.loadtxt(os.path.join(GOLDEN, "simu_single_subset_time_series.txt"))
T, Y = np.ascontiguousarray(TS[:, 0]), np.log(TS[:, 1])
S2 = TS[:, 2] ** 2 / TS[:, 1] ** 2
TOL = 1e-9   # absolute: powers lie in [0, 1]
BMAX = 1000


def _irregular(N, seed):
    rng = np.random.default_rng(seed)
    t = np.cumsum(0.05 + rng.exponential(1.0, N))
    return t, rng.uniform(0.01, 0.05, N) ** 2


def _times(N):
    """The golden simu_single series (N = 485, on a 0.25-day grid), its first three points, or an irregular series."""
    if N == len(T):
        return T, S2
    if N == 3:
        return T[:3].copy(), S2[:3].copy()
    return _irregular(N, N)


@pytest.fixture(scope="module")
def pb():
    import pioran_b200
    return pioran_b200


@pytest.fixture(scope="module")
def ctx(pb):
    return pb.get_context(0)


@pytest.fixture(scope="module")
def series(ctx):
    """N → (t, s2, resident series, BMAX rows drawn by pioran_celerite_simulate, offset by the log-flux mean)."""
    out = {}
    for N in (3, len(T), 2000):
        t, s2 = _times(N)
        ser = ctx.upload_series(t, np.zeros(N), s2)
        f0, fm = 1 / (t[-1] - t[0]), 0.5 / np.min(np.diff(t))
        a, b, c, d = orc.approx("SBPL", [0.82, 0.01, 3.3], f0 / 10, fm * 10, 20, 0.3, basis="SHO")
        q = np.random.default_rng(N).standard_normal((BMAX, N))
        rows = ctx.celerite_simulate(ser, *(np.tile(np.asarray(x), (BMAX, 1)) for x in (a, b, c, d)), q) + Y.mean()
        out[N] = (t, s2, ser, rows)
    yield out
    for v in out.values():
        v[2].free()


def _check(got, t, rows, freq, s2, what):
    """|gpu − lsp_math| ≤ TOL, NaN where the oracle has NaN.  Beyond TOL only at an ill-conditioned frequency, and then the
    GPU must lie within max(TOL, 16 ε·cond) of the 80-bit evaluation, cond = lsp_math.condition (|CC·SS| / |CC·SS − CS²|):
    the rounding of any FP64 evaluation of the normalisers is amplified that much.  A frequency whose denominator vanishes
    to rounding only (cond > 1e12: three points at f = 1/T) is 0/0 in exact arithmetic, holds rounding noise in any precision
    and is not compared."""
    want = lm.lombscargle(t, rows, freq, s2)
    cond = lm.condition(t, freq, s2)
    sing = (cond > 1e12) & ~np.isnan(want[0])   # an exactly degenerate basis is 0/0 = NaN on both sides
    assert sing.sum() <= (len(t) == 3), f"{what}: {sing.sum()} singular frequencies"
    got, want, freq, cond = got[:, ~sing], want[:, ~sing], freq[~sing], cond[~sing]
    assert np.array_equal(np.isnan(got), np.isnan(want)), f"{what}: NaN pattern differs"
    err = np.abs(got - want)
    bad = np.argwhere(err > TOL)
    if len(bad):
        rws = np.unique(bad[:, 0])
        ld = lm.lombscargle(t, rows[rws], freq, s2, dtype=np.longdouble).astype(np.float64)
        idx = {r: k for k, r in enumerate(rws)}
        for i, j in bad:
            e_gpu = abs(got[i, j] - ld[idx[i], j])
            assert e_gpu <= max(TOL, 16 * np.finfo(np.float64).eps * cond[j]), (
                f"{what}: row {i}, f {freq[j]:.6g} (cond {cond[j]:.1e}): |gpu − f64| {err[i, j]:.2e}, |gpu − 80-bit| {e_gpu:.2e}")
        assert len(bad) <= max(1, got.size // 100), f"{what}: {len(bad)} entries needed the 80-bit route"


@pytest.mark.parametrize("weighted", [True, False])
@pytest.mark.parametrize("F", [1, 63, 64, 65, 1000])
@pytest.mark.parametrize("N", [3, 485, 2000])
@pytest.mark.parametrize("B", [1, 7, 64, 65, 1000])
def test_parity(ctx, series, B, N, F, weighted):
    t, s2, ser, rows = series[N]
    freq = lm.frequency_grid(t, F)
    got = ctx.lombscargle(ser, freq, y_batch=rows[:B], weighted=weighted)
    assert got.shape == (B, F)
    assert ctx.last_kernel_name() == "lsp<64,64,32>"
    _check(got, t, rows[:B], freq, s2 if weighted else None, f"B={B} N={N} F={F} weighted={weighted}")


def test_small_workspace_is_bit_for_bit(ctx, series):
    t, s2, ser, rows = series[len(T)]
    freq = lm.frequency_grid(t, 1000)
    want = ctx.lombscargle(ser, freq, y_batch=rows[:200])
    n0 = ctx.launch_count
    try:
        ctx.set_lsp_workspace(1 << 20)   # 32 frequency chunks of 32, row chunks of 64
        n1 = ctx.launch_count
        got = ctx.lombscargle(ser, freq, y_batch=rows[:200])
        assert ctx.launch_count - n1 > 10 * (n1 - n0)
    finally:
        ctx.set_lsp_workspace(0)
    assert np.array_equal(got, want, equal_nan=True)


def test_row_of_a_batch_is_a_one_row_call(ctx, series):
    t, s2, ser, rows = series[2000]
    freq = lm.frequency_grid(t, 65)
    for weighted in (True, False):
        P = ctx.lombscargle(ser, freq, y_batch=rows[:65], weighted=weighted)
        for i in (0, 31, 63, 64):
            assert np.array_equal(ctx.lombscargle(ser, freq, y_batch=rows[i], weighted=weighted)[0], P[i], equal_nan=True)


def test_resident_y(ctx):
    freq = lm.frequency_grid(T, 1000)
    ser = ctx.upload_series(T, Y, S2)
    try:
        for weighted in (True, False):
            got = ctx.lombscargle(ser, freq, weighted=weighted)
            assert np.array_equal(got, ctx.lombscargle(ser, freq, y_batch=Y[None], weighted=weighted), equal_nan=True)
    finally:
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
def test_device_group_matches_single_device(pb, ctx, series, devices):
    if len(devices) > _ndev():
        pytest.skip("needs %d GPUs" % len(devices))
    t, s2, ser, rows = series[len(T)]
    freq = lm.frequency_grid(t, 1000)
    grp = pb.Context(devices)
    sg = grp.upload_series(t, np.zeros_like(t), s2)
    try:
        one = ctx.lombscargle(ser, freq, y_batch=rows[:301])
        assert np.array_equal(grp.lombscargle(sg, freq, y_batch=rows[:301]), one, equal_nan=True)
        grp.set_lsp_workspace(1 << 20)
        assert np.array_equal(grp.lombscargle(sg, freq, y_batch=rows[:301]), one, equal_nan=True)
    finally:
        sg.free()
        grp.close()


def test_invariances(ctx, series):
    t, s2, ser, rows = series[len(T)]
    freq = lm.frequency_grid(t, 1000)
    Yb = rows[:64]
    base = ctx.lombscargle(ser, freq, y_batch=Yb)
    for what, tt, ss, yy in (("t + 1e6", t + 1e6, s2, Yb), ("σ² × 7.3", t, 7.3 * s2, Yb), ("y + 100", t, s2, Yb + 100.0)):
        s = ctx.upload_series(tt, np.zeros_like(tt), ss)
        try:
            got = ctx.lombscargle(s, freq, y_batch=yy)
        finally:
            s.free()
        assert np.array_equal(np.isnan(got), np.isnan(base)), what
        assert np.nanmax(np.abs(got - base)) <= TOL, what


def test_degenerate_values(ctx):
    t = np.arange(40.0) + 3.0
    y = np.random.default_rng(5).normal(size=(2, 40))
    y[1] = 0.0
    freq = np.array([0.1, 0.5, 0.37])
    ser = ctx.upload_series(t, np.zeros(40), np.ones(40))
    one = ctx.upload_series(t[:1], np.ones(1), np.ones(1))
    try:
        p = ctx.lombscargle(ser, freq, y_batch=y)
        assert np.all(np.isfinite(p[0, [0, 2]])) and np.isnan(p[0, 1])   # integer times at f = 0.5
        assert np.all(np.isnan(p[1]))                                     # an all-zero row
        assert np.all(np.isnan(ctx.lombscargle(one, freq)))              # N = 1
        assert np.all(np.isnan(ctx.lombscargle(one, freq, weighted=False)))
    finally:
        ser.free(); one.free()


def test_launches_grow_with_chunks_not_rows(ctx, series):
    t, s2, ser, rows = series[2000]
    freq = lm.frequency_grid(t, 1000)
    counts = []
    for B in (1, 7, 64, 1000):
        n0 = ctx.launch_count
        ctx.lombscargle(ser, freq, y_batch=rows[:B])
        counts.append(ctx.launch_count - n0)
    assert counts == [3, 3, 3, 3]   # basis, rows, product
    try:
        ctx.set_lsp_workspace(5 << 20)   # 64 frequencies per chunk: 16 chunks
        n0 = ctx.launch_count
        ctx.lombscargle(ser, freq, y_batch=rows[:7])
        assert ctx.launch_count - n0 == 1 + 16 * 2
    finally:
        ctx.set_lsp_workspace(0)


def test_argument_checks(ctx):
    lib = ctx.lib
    dp = C.POINTER(C.c_double)
    p = lambda x: x.ctypes.data_as(dp) if x is not None else None
    freq = np.array([0.1, 0.2, 0.3])
    y = np.random.default_rng(1).normal(size=(2, len(T)))
    out = np.empty((2, 3))
    ser = ctx.upload_series(T, Y, S2)
    bad_s2 = {}
    for name, v in (("zero", 0.0), ("negative", -1.0), ("inf", np.inf), ("nan", np.nan)):
        s = S2.copy(); s[17] = v
        bad_s2[name] = ctx.upload_series(T, Y, s)
    call = lambda h, sid, B, yb, wt, F, fq, o: lib.pioran_lombscargle(h, sid, B, yb, wt, F, fq, o)
    try:
        assert call(ctx.h, ser.id, 2, p(y), 1, 3, p(freq), p(out)) == 0
        assert call(None, ser.id, 2, p(y), 1, 3, p(freq), p(out)) == -1           # NULL ctx
        assert call(ctx.h, ser.id, 2, p(y), 1, 3, None, p(out)) == -1             # NULL freq
        assert call(ctx.h, ser.id, 2, p(y), 1, 3, p(freq), None) == -1            # NULL power_out
        assert call(ctx.h, ser.id, 0, p(y), 1, 3, p(freq), p(out)) == -1          # B < 1
        assert call(ctx.h, ser.id, 2, p(y), 1, 0, p(freq), p(out)) == -1          # F < 1
        assert call(ctx.h, ser.id, 2, None, 1, 3, p(freq), p(out)) == -1          # resident y with B > 1
        for v in (0.0, -0.1, np.inf, np.nan):                                     # frequencies
            fq = freq.copy(); fq[1] = v
            assert call(ctx.h, ser.id, 2, p(y), 1, 3, p(fq), p(out)) == -1
        assert call(ctx.h, ser.id + 1000, 2, p(y), 1, 3, p(freq), p(out)) == -1   # unknown series
        for name, s in bad_s2.items():                                            # weights of a bad σ²
            assert call(ctx.h, s.id, 2, p(y), 1, 3, p(freq), p(out)) == -1, name
            assert "s2[17]" in lib.pioran_last_error().decode()
            assert call(ctx.h, s.id, 2, p(y), 0, 3, p(freq), p(out)) == 0, name
        assert lib.pioran_ctx_set_lsp_workspace(ctx.h, -1) == -1
        assert call(ctx.h, ser.id, 1, None, 1, 3, p(freq), p(out)) == 0
    finally:
        ser.free()
        for s in bad_s2.values():
            s.free()


def test_python_interface(pb, series):
    t, s2, ser, rows = series[len(T)]
    freq = np.geomspace(1 / (t[-1] - t[0]), 0.999 * 0.5 / np.min(np.diff(t)), 1000)   # below the degenerate 1/(2·min Δt)
    dy = np.sqrt(s2)
    scipy = lambda y, w: signal.lombscargle(t, y, 2 * np.pi * freq, weights=w, floating_mean=True, normalize="normalize")
    one = pb.lombscargle(t, Y, dy, frequencies=freq)
    assert one.shape == (1000,) and np.max(np.abs(one - scipy(Y, 1 / s2))) <= TOL
    many = pb.lombscargle(t, rows[:20], frequencies=freq)
    assert many.shape == (20, 1000)
    assert max(np.max(np.abs(many[i] - scipy(rows[i], None))) for i in range(20)) <= TOL
    # the points may come in any order
    perm = np.random.default_rng(2).permutation(len(t))
    assert np.array_equal(pb.lombscargle(t[perm], Y[perm], dy[perm], frequencies=freq), one)
