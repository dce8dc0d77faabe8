import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run with -m gpu on the GPU box)")


def rel_err(x, ref):
    """|Δ| / max(1, |ref|): relative error that stays meaningful near logL ≈ 0 (SURVEY §7)."""
    x, ref = np.asarray(x, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    return np.abs(x - ref) / np.maximum(1.0, np.abs(ref))


EXEMPTIONS = []   # (test id, rows checked, rows that used the conditioning exemption, worst |gpu − ref| among them)
MAX_EXEMPT_FRACTION = 0.02


def assert_parity(got, want, theta, ld_fn, tol=1e-9, slack=4.0, label=None):
    """Parity bar of BASELINE.json (≤ 1e-9 relative on logL, FP64) made conditioning-aware: a row may exceed `tol`
    only if the reference algorithm's own FP64 answer `want` is itself farther than tol/slack from the 80-bit
    evaluation of the same recursion (ld_fn(row) → long double twin in the oracle), and then the GPU value must lie
    within slack × that distance of the 80-bit value.  SURVEY §7 "parity on ill-conditioned θ": at steep PSD slopes
    the cancellation D_n = Σa + σ²_n − UᵀSU (src/celerite_solver.jl:92) loses ~7 digits in any operation order.
    The exemption is this repo's rule, not BASELINE's: every use is counted, capped at MAX_EXEMPT_FRACTION of the rows of the
    call, and listed in the terminal summary of the run (pytest_terminal_summary below)."""
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    r = rel_err(got, want)
    bad = np.flatnonzero(~(r <= tol))
    report = []
    for i in bad:
        if not np.isfinite(want[i]):
            assert not np.isfinite(got[i]), f"row {i}: reference non-finite, GPU {got[i]}"
            continue
        ld = float(ld_fn(theta[i]))
        e_ref, e_gpu = float(rel_err(want[i], ld)), float(rel_err(got[i], ld))
        report.append((int(i), float(r[i]), e_ref, e_gpu))
        assert e_ref > tol / slack and e_gpu <= slack * e_ref, (
            f"row {i}: |gpu-ref| {r[i]:.3e} > {tol:g}; vs 80-bit: ref {e_ref:.3e}, gpu {e_gpu:.3e}")
    name = label or os.environ.get("PYTEST_CURRENT_TEST", "?").split(" ")[0]
    EXEMPTIONS.append((name, int(got.size), len(report), max((x[1] for x in report), default=0.0)))
    assert len(report) <= max(1, int(MAX_EXEMPT_FRACTION * got.size)), (
        f"{len(report)} of {got.size} rows needed the conditioning exemption (cap {MAX_EXEMPT_FRACTION:.0%})")
    return report


def pytest_terminal_summary(terminalreporter):
    if not EXEMPTIONS:
        return
    tr = terminalreporter
    rows, used = sum(e[1] for e in EXEMPTIONS), sum(e[2] for e in EXEMPTIONS)
    tr.write_line(f"parity exemptions (conftest.assert_parity): {used} of {rows} rows over {len(EXEMPTIONS)} checks")
    for name, n, k, worst in EXEMPTIONS:
        if k:
            tr.write_line(f"  {name}: {k}/{n} rows beyond 1e-9 where the FP64 reference itself is off the 80-bit value; worst |gpu-ref| {worst:.2e}")


class GoldenRun:
    """One shipped ultranest run of the reference: the series it used and the (θ, logL) pairs it produced."""

    def __init__(self, stem, model, n_psd_par, log_transform, chains_file="chains.npz"):
        ts = np.loadtxt(os.path.join(GOLDEN, f"{stem}_subset_time_series.txt"))
        self.t, self.y_raw, self.yerr = (np.ascontiguousarray(c) for c in ts.T)
        chains = np.load(os.path.join(GOLDEN, chains_file))
        self.chain = chains[stem]
        self.columns = [str(c) for c in chains[stem + "_columns"]]
        self.model, self.n_psd_par = model, n_psd_par
        # examples/ultranest/single_pl.jl:48: f_min, f_max = 1/(t[end]-t[1]), 1/minimum(diff(t))/2
        self.f_min = 1.0 / (self.t[-1] - self.t[0])
        self.f_max = 1.0 / np.min(np.diff(self.t)) / 2.0
        if log_transform:  # single_pl.jl:70-73: σ² = ν σ²/y², yn = log y
            self.y = np.log(self.y_raw)
            self.s2 = self.yerr ** 2 / self.y_raw ** 2
        else:              # single_pl_periodicity.jl: σ² = ν σ²
            self.y = self.y_raw.copy()
            self.s2 = self.yerr ** 2
        self.logl = self.chain[:, 1]
        self.theta = self.chain[:, 2:2 + n_psd_par + 3]  # psd parameters…, variance, ν, μ


@pytest.fixture(scope="session")
def golden_single():
    return GoldenRun("simu_single", "SingleBendingPowerLaw", 3, True)


@pytest.fixture(scope="session")
def golden_double():
    return GoldenRun("simu_double", "DoubleBendingPowerLaw", 5, True)


@pytest.fixture(scope="session")
def golden_periodic():
    g = GoldenRun("simu_periodic_rednoise", "SingleBendingPowerLaw", 3, False, "simu_periodic_rednoise_chains.npz")
    return g


def periodic_mean(t, row):
    """examples/ultranest/single_pl_periodicity.jl: A·sin(2πt/T₀ + ϕ) + μ ; columns … μ A ϕ T₀."""
    mu, A, phi, T0 = row[7], row[8], row[9], row[10]
    return A * np.sin(2 * np.pi * t / T0 + phi) + mu


sys.path.insert(0, os.path.join(ROOT, "tools"))
import workloads as _wl  # noqa: E402


def synthetic_series(N, seed, theta0=(0.82, 0.01, 3.3), variance=1.0, basis="SHO", J=20):
    """SURVEY §8d generator (tools/workloads.py — the same inputs bench.py uses): gaps 0.05+Exp(1), σ~U(0.01,0.05),
    y = celerite GP draw at θ₀ + N(0,σ²).  → t, y, σ², f_min, f_max"""
    return _wl.make_series(N, seed, theta0, variance, J)


def prior_theta(B, f_min, f_max, ybar, ysd, seed, alpha2_max=4.0):
    """Prior transform of examples/ultranest/single_pl.jl:96-104 on a seeded unit cube (SURVEY §8d, config C2)."""
    return _wl.prior_theta(B, f_min, f_max, ybar, ysd, seed, alpha2_max)
