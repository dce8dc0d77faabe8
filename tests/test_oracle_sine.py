"""The sinusoidal-mean oracle (tests/tools/oracle_sine.c) on the CPU: its values against the shipped pairs of the reference's
periodicity run, its constant-mean limit against the gradient oracle it is built on, and its mean partials against central
differences of its own values."""
import os
import sys

import numpy as np

from conftest import rel_err
from oracle import oracle as orc

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "tools"))
import oracle_sine as osn  # noqa: E402


def test_values_are_the_golden_pairs(golden_periodic):
    g = golden_periodic
    rows = g.chain[::500]
    val, _ = osn.approx_logl_sine_grad_batch("SBPL", rows[:, 2:11], g.f_min, g.f_max, 20, g.t, g.y, g.s2)
    assert rel_err(val, rows[:, 1]).max() <= 1e-9


def test_amplitude_zero_is_the_gradient_oracle(golden_periodic):
    g = golden_periodic
    th = np.ascontiguousarray(g.chain[::900, 2:11])
    th[:, 6] = 0.0
    val, grad = osn.approx_logl_sine_grad_batch("SBPL", th, g.f_min, g.f_max, 20, g.t, g.y, g.s2)
    pv, pg = orc.approx_logl_grad_batch("SBPL", th[:, :6], g.f_min, g.f_max, 20, g.t, g.y, g.s2)
    assert np.array_equal(val, pv) and np.array_equal(grad[:, :6], pg)
    assert np.all(grad[:, 7:] == 0.0)


def test_mean_partials_against_central_differences(golden_periodic):
    g = golden_periodic
    th = np.ascontiguousarray(g.chain[::1000, 2:11])
    _, grad = osn.approx_logl_sine_grad_batch("SBPL", th, g.f_min, g.f_max, 20, g.t, g.y, g.s2)
    for k in (5, 6, 7, 8):
        h = 1e-6 * np.maximum(np.abs(th[:, k]), 1e-3)
        tp, tm = th.copy(), th.copy()
        tp[:, k] += h
        tm[:, k] -= h
        fd = (osn.approx_logl_sine_grad_batch("SBPL", tp, g.f_min, g.f_max, 20, g.t, g.y, g.s2)[0] -
              osn.approx_logl_sine_grad_batch("SBPL", tm, g.f_min, g.f_max, 20, g.t, g.y, g.s2)[0]) / (2 * h)
        assert np.all(np.abs(grad[:, k] - fd) <= 1e-5 * np.maximum(1.0, np.abs(fd))), k
    ld, lgrad = osn.approx_logl_sine_grad_batch("SBPL", th, g.f_min, g.f_max, 20, g.t, g.y, g.s2, long_double=True)
    assert np.all(np.abs(lgrad - grad) <= 1e-8 * np.maximum(1.0, np.abs(grad)).max(axis=0))
