"""The Lomb–Scargle restatement K9 is tested against (tests/tools/proto/lsp_math.py): agreement with scipy's generalised
periodogram with a floating mean, weighted and unweighted, invariance to a time offset, and agreement with its own 80-bit
evaluation."""
import os
import sys

import numpy as np
import pytest
from scipy import signal

from conftest import GOLDEN

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "tools", "proto"))
import lsp_math as lm  # noqa: E402

TS = np.loadtxt(os.path.join(GOLDEN, "simu_single_subset_time_series.txt"))


def _series(N, seed):
    rng = np.random.default_rng(seed)
    t = np.cumsum(0.05 + rng.exponential(1.0, N))
    y = np.sin(2 * np.pi * t / 17.0) + rng.normal(0, 0.5, N) + 3.0
    s2 = rng.uniform(0.01, 0.3, N) ** 2
    return t, y, s2


def _degenerate(t, freq):
    """Frequencies at which sin πx vanishes at every time: there the definition divides 0 by 0 (NaN), while scipy returns
    whatever its rounding of sin gives.  The golden series lies on a 0.25-day grid, so its 1/(2·min Δt) is one of them."""
    sn, _ = lm.sincospi((2 * freq)[:, None] * (t - t[0])[None, :])
    return np.all(sn == 0, axis=1)


def _scipy(t, y, freq, s2=None):
    w = None if s2 is None else 1 / s2
    return signal.lombscargle(t, y, 2 * np.pi * freq, weights=w, floating_mean=True, normalize="normalize")


CASES = {"irregular-300": _series(300, 1), "irregular-57": _series(57, 2),
         "simu_single": (TS[:, 0], np.log(TS[:, 1]), TS[:, 2] ** 2 / TS[:, 1] ** 2)}


@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("weighted", [True, False])
def test_matches_scipy(case, weighted):
    t, y, s2 = CASES[case]
    freq = lm.frequency_grid(t, 500)
    got = lm.lombscargle(t, y, freq, s2 if weighted else None)
    want = _scipy(t, y, freq, s2 if weighted else None)
    deg = _degenerate(t, freq)
    assert np.array_equal(np.isnan(got), deg) and deg.sum() == (case == "simu_single")
    assert np.max(np.abs(got - want)[~deg]) <= 1e-11


def test_batch_rows_are_single_calls():
    t, y, s2 = CASES["irregular-300"]
    Y = np.stack([y, 2 * y - 1, np.cos(t)])
    freq = lm.frequency_grid(t, 64)
    P = lm.lombscargle(t, Y, freq, s2)
    for i in range(3):
        assert np.max(np.abs(P[i] - lm.lombscargle(t, Y[i], freq, s2))) <= 1e-14


@pytest.mark.parametrize("weighted", [True, False])
def test_time_offset(weighted):
    t, y, s2 = CASES["irregular-300"]
    freq = lm.frequency_grid(t, 500)
    s = s2 if weighted else None
    assert np.max(np.abs(lm.lombscargle(t + 1e6, y, freq, s) - lm.lombscargle(t, y, freq, s))) <= 1e-9


@pytest.mark.parametrize("case", sorted(CASES))
def test_longdouble(case):
    t, y, s2 = CASES[case]
    freq = lm.frequency_grid(t, 200)
    got = lm.lombscargle(t, y, freq, s2)
    ld = lm.lombscargle(t, y, freq, s2, dtype=np.longdouble).astype(np.float64)
    assert np.array_equal(np.isnan(got), np.isnan(ld))
    assert np.nanmax(np.abs(got - ld)) <= 1e-11


def test_sincospi_exact_at_integers():
    s, c = lm.sincospi(np.arange(-8.0, 9.0))
    assert np.all(s == 0) and np.all(np.abs(c) == 1)
    x = np.random.default_rng(3).uniform(-1e3, 1e3, 1000)
    s, c = lm.sincospi(x)
    assert np.max(np.abs(s - np.sin(np.pi * x))) <= 1e-12 and np.max(np.abs(c - np.cos(np.pi * x))) <= 1e-12


def test_degenerate_values_are_nan():
    t = np.arange(20.0)
    y = np.random.default_rng(4).normal(size=20)
    p = lm.lombscargle(t, y, np.array([0.1, 0.5]))
    assert np.isfinite(p[0]) and np.isnan(p[1])
    assert np.all(np.isnan(lm.lombscargle(t, np.zeros(20), np.array([0.1, 0.2]))))
    assert np.all(np.isnan(lm.lombscargle(t[:1], y[:1], np.array([0.1, 0.2]))))
