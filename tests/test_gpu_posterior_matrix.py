"""Posterior matrix: every kernel instantiation the posterior mean, variance, covariance, posterior draws and prior draws of
csrc/api.cu can reach, one cell each, at the rank, term-layout and size edges.

A cell is one call through pioran_b200.Context.  It asserts:
  1. Context.last_kernel_name() is the last kernel expected() predicts.  The ABI names only the last kernel of a call; the
     kernels before it (the STEP_STORE factor, the covariance pass of the variance kernel) are pinned by the restatement and
     by the CPU ledger test;
  2. every set of the call against a dense CPU reference: the mean against a dense solve (orc.direct_predict), the variance
     and the covariance against postcov_math.dense_cov (1e-9·Σa), the posterior draws against the oracle composition of
     test_gpu_postdraw (1e-9·√Σa), the prior draws against the dense Cholesky factor of K + diag(νσ²) times q;
  3. the identities of the entries: the mean of predict_var and predict_cov is predict's bit for bit, diag(cov) is var within
     1e-9·Σa, cov is exactly symmetric, and each set equals its single-set call: bit for bit where the set's own rank is the
     batch rank, within the tolerance where it is lower (a term real in some sets and complex in others).

Inputs are well-conditioned sets (COND of the sweep matrix: the FP64 log-likelihood of the set within 1e-12 of its 80-bit
twin), so that an error of 1e-7 in one row stands out.  Where the FP64 dense reference is itself off, the 80-bit route decides
(postcov_math.dense_cov_ld, an 80-bit Cholesky factor, the dense-draw rule of test_gpu_postdraw); every such use is counted
and capped per cell at the fraction conftest.assert_parity allows.

The module uses its own context."""
import os
import sys
import zlib

import numpy as np
import pytest
from scipy.linalg import cholesky

from conftest import MAX_EXEMPT_FRACTION, rel_err
from oracle import oracle as orc
from test_gpu_postdraw import _check_oracle, oracle_draws
from test_gpu_sweep_matrix import COND, Unsupported, bs_for_rank, nw_for_bs
from test_postdraw_proto import _chol_ld, _kernel_ld

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "tools", "proto"))
import postcov_math as cm  # noqa: E402
import postvar_math as pm  # noqa: E402

TOL = 1e-9
B200_SMS = 148
MAX_RANK = 128
ENTRIES = ("predict", "var", "cov", "draws", "simulate")


# ------------------------------------------------------------------------------------------------ the dispatch, restated
def _cdiv(a, b):
    return -(-a // b)


def _factor(R, mode):
    """launch_wide<MODE> (ranks 65 … 128: one CTA per set) or dispatch_generic_mode<MODE> (one warp per set)."""
    BS = bs_for_rank(R)
    if BS > 8:
        return f"wide_reg_{mode}<{max(5, _cdiv(R, 16))}>"
    return f"generic_{mode}<{BS},{nw_for_bs(BS)}>"


def expected(entry, R, Jt):
    """Every templated kernel one call launches, in launch order; the last is the one last_kernel_name() reports.
    predict<PT> stands for the backsolve and predict kernels of launch_posterior_mean (PT by the term count Jt); var and cov
    are called with the mean.  The draws factor the data covariance and the covariance on the merged grid of t and τ."""
    if R > MAX_RANK:
        raise Unsupported(R)
    store = _factor(R, "store")
    mean = f"predict<{2 if Jt <= 64 else 4}>"
    TS = _cdiv(R, 16)                       # launch_postvar
    PT = 1 if R <= 32 else 2 if R <= 64 else 4
    return {
        "predict": [store, mean],
        "var": [store, mean, f"postvar<{TS}>"],
        "cov": [store, mean, f"postvar_cov<{TS}>", f"postcov<{PT}>"],
        "draws": [store, store, f"postdraw<{PT}>"],
        "simulate": [_factor(R, "sim")],
    }[entry]


# ------------------------------------------------------------------------------------------------ coverage ledger
LEDGER = (
    {"generic_store<4,12>", "generic_store<5,12>", "generic_store<6,10>", "generic_store<7,8>", "generic_store<8,8>"}
    | {"wide_reg_store<5>", "wide_reg_store<6>", "wide_reg_store<7>", "wide_reg_store<8>"}
    | {"generic_sim<4,12>", "generic_sim<5,12>", "generic_sim<6,10>", "generic_sim<7,8>", "generic_sim<8,8>"}
    | {"wide_reg_sim<5>", "wide_reg_sim<6>", "wide_reg_sim<7>", "wide_reg_sim<8>"}
    | {"predict<2>", "predict<4>"}
    | {f"postvar<{ts}>" for ts in range(1, 9)} | {f"postvar_cov<{ts}>" for ts in range(1, 9)}
    | {"postdraw<1>", "postdraw<2>", "postdraw<4>", "postcov<1>", "postcov<2>", "postcov<4>"}
)


# ------------------------------------------------------------------------------------------------ cells
class Cell:
    """One call: ncx complex and nre real terms in a term layout, N data points, M prediction points, S draws, B = k·SMs + c
    sets (bk = (k, c)).  mixed: one more column, real (b = d = 0) in the even sets and complex in the odd ones."""

    def __init__(self, name, entry, ncx, nre, layout="cx-first", N=61, M=24, S=3, bk=(0, 3), mixed=False):
        self.name, self.entry, self.ncx, self.nre, self.layout = name, entry, ncx, nre, layout
        self.N, self.M, self.S, self.bk, self.mixed = N, M, S, bk, mixed
        self.Jt = ncx + nre + mixed
        self.R = 2 * (ncx + mixed) + nre

    def B(self, num_sms):
        return self.bk[0] * num_sms + self.bk[1]

    def expected(self):
        return expected(self.entry, self.R, self.Jt)

    def __repr__(self):
        return self.name


def _split(R):
    """(complex, real) terms of rank R: one real term at odd ranks, two at even ones (rank 2: two real terms)."""
    nre = 1 if R % 2 else 2
    return (R - nre) // 2, nre


RANKS = (1, 2, 16, 17, 32, 33, 40, 41, 48, 49, 56, 57, 64, 65, 80, 81, 96, 97, 112, 113, 127, 128)
BOUNDARY = (16, 17, 32, 33, 64, 65, 96, 97, 128)   # postvar TS 1|2, PT 1|2, BS 8 | TS 5, TS 6|7, the limit

RANK_CELLS = [Cell(f"{e}-r{R}", e, *_split(R)) for e in ENTRIES for R in RANKS]
LAYOUT_CELLS = [Cell(f"{e}-r{R}-{lay}", e, *_split(R), layout=lay) for e in ENTRIES for R in BOUNDARY
                for lay in ("re-first", "interleaved")]
# many real terms: the term count of the mean kernels (predict<2> up to 64 terms) at rank = term count
TERM_CELLS = [Cell(f"{e}-jt{jt}-real", e, 0, jt) for e in ENTRIES for jt in (64, 65, 128)]
# the mixed column makes the batch rank 33 (PT 2, postvar<3>); the even sets alone are rank 32 (PT 1, postvar<2>)
MIXED_CELLS = [Cell(f"{e}-mixed-r33", e, 15, 1, bk=(0, 4), mixed=True) for e in ENTRIES]

# sizes around the staging chunks: the factor's 4 steps (GCH, WIDE_CH), the 8 steps of K6 … K8 over t or the merged grid
# (M = 8 keeps N + M at the residues of N), 16 warps per CTA of K7 and K8, 4 sets per CTA of predict
EDGE_N = (1, 2, 3, 4, 5, 7, 8, 9, 16, 17)
EDGE_CELLS = [Cell(f"{e}-r{R}-N{N}", e, *_split(R), N=N, M=8, S=2) for R in (41, 97) for e in ENTRIES for N in EDGE_N]
EDGE_CELLS += [Cell(f"{e}-r{R}-M{M}", e, *_split(R), M=M) for R in (49, 113) for e in ENTRIES[:4] for M in (1, 15, 16, 17, 33)]
EDGE_CELLS += [Cell(f"draws-r{R}-S{S}", "draws", *_split(R), N=40, M=16, S=S) for R in (33, 113) for S in (1, 15, 16, 17)]
EDGE_CELLS += [Cell(f"{e}-r{R}-B{B}", e, *_split(R), N=30, M=12, bk=(0, B)) for R in (20, 41) for e in ENTRIES
               for B in sorted({1, 3, 4, 5, nw_for_bs(bs_for_rank(R)) - 1, nw_for_bs(bs_for_rank(R)) + 1})]
# whole waves of work items of the factor: nw_for_bs(BS) sets per CTA, and one set more or less
FULL_CELLS = [Cell(f"{e}-r{R}-full-items{tag}", e, *_split(R), N=17, M=9, S=1, bk=(nw_for_bs(bs_for_rank(R)), c))
              for R in (20, 41) for e in ("predict", "simulate") for tag, c in (("-1", -1), ("+1", 1))]

ALL_CELLS = RANK_CELLS + LAYOUT_CELLS + TERM_CELLS + MIXED_CELLS + EDGE_CELLS + FULL_CELLS


def test_ledger_is_exactly_what_the_cells_reach():
    """CPU: the cells launch every ledger entry and nothing else; no cell is refused; names are unique."""
    reached = set().union(*(c.expected() for c in ALL_CELLS))
    assert reached - LEDGER == set(), f"cells reach kernels missing from the ledger: {sorted(reached - LEDGER)}"
    assert LEDGER - reached == set(), f"ledger entries no cell reaches: {sorted(LEDGER - reached)}"
    assert len(LEDGER) == 42
    assert len({c.name for c in ALL_CELLS}) == len(ALL_CELLS)
    assert all(c.R <= MAX_RANK for c in ALL_CELLS)


def test_expected_restates_known_dispatch_points():
    """CPU: fixed points of the dispatch that the posterior tests and DESIGN.md rely on."""
    assert expected("predict", 40, 20) == ["generic_store<5,12>", "predict<2>"]
    assert expected("var", 40, 20)[-1] == "postvar<3>" and expected("var", 60, 40)[-1] == "postvar<4>"
    assert expected("var", 128, 68)[-1] == "postvar<8>" and expected("cov", 128, 68)[-2:] == ["postvar_cov<8>", "postcov<4>"]
    assert expected("draws", 40, 20) == ["generic_store<5,12>", "generic_store<5,12>", "postdraw<2>"]
    assert expected("draws", 60, 40)[-1] == "postdraw<2>" and expected("cov", 80, 40)[-1] == "postcov<4>"
    assert expected("simulate", 40, 20) == ["generic_sim<5,12>"] and expected("simulate", 90, 60) == ["wide_reg_sim<6>"]
    assert expected("predict", 120, 80) == ["wide_reg_store<8>", "predict<4>"]
    assert expected("predict", 64, 64)[-1] == "predict<2>" and expected("predict", 65, 65)[-1] == "predict<4>"
    assert expected("var", 1, 1) == ["generic_store<4,12>", "predict<2>", "postvar<1>"]
    for e in ENTRIES:
        with pytest.raises(Unsupported):
            expected(e, 129, 65)


def test_cells_cover_the_grid():
    """CPU: every entry at every rank of RANKS, and each layout edge of the issue's table at least once per entry."""
    for e in ENTRIES:
        assert {c.R for c in RANK_CELLS if c.entry == e} == set(RANKS)
        assert {c.Jt for c in TERM_CELLS if c.entry == e} == {64, 65, 128}
    assert {c.N for c in EDGE_CELLS} >= set(EDGE_N)
    assert {c.S for c in EDGE_CELLS if c.entry == "draws"} >= {1, 15, 16, 17}
    assert {c.M for c in EDGE_CELLS} >= {1, 15, 16, 17, 33}


# ------------------------------------------------------------------------------------------------ inputs
def _seed(name):
    return zlib.crc32(name.encode())


def _series(N, rng):
    """A short random series that does not start at t = 0: gaps 0.05 + Exp(1), σ² ~ U(0.01, 0.05)."""
    t = rng.uniform(-40.0, 40.0) + np.cumsum(0.05 + rng.exponential(1.0, N))
    return t, rng.normal(0.0, 0.7, N), rng.uniform(0.01, 0.05, N)


def _kinds(cell):
    """'c' (complex) or 'r' (real) per column; 'm' marks the mixed column."""
    ncx, nre = cell.ncx, cell.nre
    if cell.layout == "cx-first":
        k = ["c"] * ncx + ["r"] * nre
    elif cell.layout == "re-first":
        k = ["r"] * nre + ["c"] * ncx
    else:   # interleaved: a real term after each of the first complex terms, so complex rows start at odd offsets
        k = []
        for j in range(max(ncx, nre)):
            k += (["c"] if j < ncx else []) + (["r"] if j < nre else [])
    if cell.mixed:
        k.insert(len(k) // 2, "m")
    return k


def _candidates(cell, n, rng):
    """n coefficient sets of the cell's layout (|b d| < a c per complex term) with per-set μ and ν."""
    kinds = np.array(_kinds(cell))
    Jt = len(kinds)
    a = rng.uniform(0.2, 1.0, (n, Jt)) / Jt
    c = np.exp(rng.uniform(np.log(0.02), np.log(3.0), (n, Jt)))
    d = rng.choice([-1.0, 1.0], (n, Jt)) * np.exp(rng.uniform(np.log(0.05), np.log(5.0), (n, Jt)))
    b = rng.uniform(-0.9, 0.9, (n, Jt)) * a * c / np.abs(d)
    re = kinds == "r"
    b[:, re] = 0.0
    d[:, re] = 0.0
    c[:, re] = np.exp(rng.uniform(np.log(0.05), np.log(2.0), (n, int(re.sum()))))
    return [a, b, c, d, rng.normal(0.0, 0.3, n), rng.uniform(0.5, 2.0, n)]


def _inputs(cell, B):
    """Series, B well-conditioned sets (mixed column real in the even sets), τ and q of a cell."""
    rng = np.random.default_rng(_seed(cell.name))
    t, y, s2 = _series(cell.N, rng)
    x = None
    for _ in range(64):
        cand = _candidates(cell, B + B // 4 + 8, rng)
        ok = []
        for i in range(len(cand[0])):
            a, b, c, d, mu, nu = (v[i] for v in cand)
            args = (a, b, c, d, t, y - mu, nu * s2)
            ok.append(rel_err(orc.celerite_logl(*args), orc.celerite_logl(*args, long_double=True)) <= COND)
        good = [v[np.flatnonzero(ok)] for v in cand]
        x = good if x is None else [np.concatenate([u, v]) for u, v in zip(x, good)]
        if len(x[0]) >= B:
            break
    assert len(x[0]) >= B, f"{cell.name}: fewer than {B} well-conditioned sets"
    x = [v[:B].copy() for v in x]
    if cell.mixed:
        j = _kinds(cell).index("m")
        x[1][0::2, j] = 0.0
        x[3][0::2, j] = 0.0
    tau = _tau(t, cell.M, rng)
    NQ = cell.N + cell.M if cell.entry == "draws" else cell.N
    q = rng.standard_normal((B, cell.S, NQ) if cell.entry == "draws" else (B, NQ))
    return t, y, s2, x, tau, q


def _tau(t, M, rng):
    """M ascending prediction times: before t₁ and after t_N, equal to a data time, a tie, the rest random over the span."""
    lo, hi = t[0] - 3.0, t[-1] + 3.0
    special = [t[0] - 1.3, t[-1] + 2.1, t[len(t) // 2]] + [0.5 * (t[0] + t[-1]) + 0.37] * 2
    if M < len(special):
        return np.sort(rng.uniform(lo, hi, M))
    return np.sort(np.concatenate([special, rng.uniform(lo, hi, M - len(special))]))


def _rank(b, d):
    """The rank make_term_rows gives a batch: a column is one row if real in every set, two otherwise."""
    real = np.all((np.atleast_2d(b) == 0.0) & (np.atleast_2d(d) == 0.0), axis=0)
    return int(np.sum(np.where(real, 1, 2)))


def _s2tau(a):
    return 1e-5 * float(np.min(a.sum(axis=1)))   # τ ties need σ²_τ > 0 in the draws


# ------------------------------------------------------------------------------------------------ references
class Tally:
    """Worst error against the reference (in the tolerance unit of each quantity), and the checks of the quantities with an
    80-bit route: how many, and how many needed it."""

    def __init__(self):
        self.worst, self.exempt, self.sets = 0.0, 0, 0

    def add(self, err, exempt=None):
        self.worst = max(self.worst, float(err) / TOL)
        if exempt is not None:
            self.exempt += bool(exempt)
            self.sets += 1


def _mean_ref(x, i, t, y, s2, tau):
    a, b, c, d, mu, nu = (v[i] for v in x)
    return orc.direct_predict(a, b, c, d, tau, t, y - mu, nu * s2) + mu


def _check_mean(got, x, t, y, s2, tau, tally):
    for i in range(len(got)):
        want = _mean_ref(x, i, t, y, s2, tau)
        err = np.max(np.abs(got[i] - want)) / max(1.0, np.max(np.abs(want)))
        assert err <= TOL, f"set {i}: mean {err:.2e} from the dense solve"
        tally.add(err)


def _check_var(got, x, t, s2, tau, tally):
    for i in range(len(got)):
        a, b, c, d, mu, nu = (v[i] for v in x)
        want = np.diag(cm.dense_cov(a, b, c, d, t, nu * s2, tau))
        err = np.max(np.abs(got[i] - want)) / np.sum(a)
        if err > TOL:   # the conditioning rule of test_gpu_postcov, on the diagonal
            ld = np.diag(cm.dense_cov_ld(a, b, c, d, t, nu * s2, tau))
            e_got, e_ref = (float(np.max(np.abs(v - ld))) / np.sum(a) for v in (got[i], want))
            assert e_got <= max(TOL, e_ref), f"set {i}: var {err:.2e}; 80-bit: {e_got:.2e} against {e_ref:.2e}"
        tally.add(err, err > TOL)


def _check_cov(got, x, t, s2, tau, tally):
    for i in range(len(got)):
        a, b, c, d, mu, nu = (v[i] for v in x)
        assert np.array_equal(got[i], got[i].T), f"set {i}: cov not exactly symmetric"
        err, ld = cm.conditioned_error(got[i], a, b, c, d, t, nu * s2, tau, TOL)
        if ld is not None:
            assert ld[0] <= max(TOL, ld[1]), f"set {i}: cov {err:.2e}; 80-bit: {ld[0]:.2e} against {ld[1]:.2e}"
        tally.add(err, ld is not None)


def _check_draws(got, x, t, y, s2, tau, q, s2t, tally):
    for i in range(len(got)):
        a, b, c, d, mu, nu = (v[i] for v in x)
        want = oracle_draws(a, b, c, d, t, y, nu * s2, tau, q[i], mu, s2t)
        err = np.max(np.abs(got[i] - want)) / np.sqrt(np.sum(a))
        if err > TOL:   # the dense-draw rule
            one = slice(i, i + 1)
            _check_oracle(got[one], *(v[one] for v in x), tau, q[one], f"set {i}", sigma2_tau=s2t, t=t, y=y, s2=s2)
        tally.add(err, err > TOL)


def _check_simulate(got, x, t, s2, q, tally):
    for i in range(len(got)):
        a, b, c, d, mu, nu = (v[i] for v in x)
        K = pm.kernel(a, b, c, d, t[:, None] - t[None, :]) + np.diag(nu * s2)
        want = cholesky(K, lower=True) @ q[i]
        scale = max(1.0, np.max(np.abs(want)))
        err = np.max(np.abs(got[i] - want)) / scale
        if err > TOL:   # the 80-bit factor decides: the GPU at least as close to it as the FP64 factor
            Kld = _kernel_ld(a, b, c, d, t[:, None] - t[None, :]) + np.diag((nu * s2).astype(np.longdouble))
            ld = _chol_ld(Kld) @ q[i].astype(np.longdouble)
            e_got, e_ref = (float(np.max(np.abs(v - ld))) / scale for v in (got[i], want))
            assert e_got <= max(TOL, e_ref), f"set {i}: sim {err:.2e}; 80-bit: {e_got:.2e} against {e_ref:.2e}"
        tally.add(err, err > TOL)


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def pb():
    import pioran_b200
    return pioran_b200


@pytest.fixture(scope="module")
def ctx(pb):
    c = pb.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def num_sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


OBSERVED = {}   # cell name → kernel name the library reported


def _call(ctx, entry, ser, x, tau, q, s2t):
    """The cell's entry on sets x; its outputs as a tuple (mean and var / cov with the mean)."""
    a, b, c, d, mu, nu = x
    if entry == "predict":
        return (ctx.celerite_predict(ser, a, b, c, d, tau, mu=mu, nu=nu),)
    if entry == "var":
        return ctx.celerite_predict_var(ser, a, b, c, d, tau, mu=mu, nu=nu)
    if entry == "cov":
        return ctx.celerite_predict_cov(ser, a, b, c, d, tau, mu=mu, nu=nu)
    if entry == "draws":
        return (ctx.celerite_posterior_draws(ser, a, b, c, d, tau, q, mu=mu, nu=nu, sigma2_tau=s2t),)
    return (ctx.celerite_simulate(ser, a, b, c, d, q, nu=nu),)


def _unit(entry, k, out, x, i):
    """The tolerance unit of output k of one set: Σa (var, cov), √Σa (draws), max(1, ‖out‖∞) (mean, prior draws)."""
    sa = float(np.sum(x[0][i]))
    if entry in ("var", "cov") and k == 1:
        return sa
    if entry == "draws":
        return np.sqrt(sa)
    return max(1.0, float(np.max(np.abs(out))))


def _invariance_sets(B):
    return sorted({0, 1, B // 2, B - 1} & set(range(B)))


@pytest.mark.gpu
@pytest.mark.parametrize("cell", ALL_CELLS, ids=repr)
def test_posterior_cell(pb, ctx, num_sms, cell, record_property):
    B = cell.B(num_sms)
    t, y, s2, x, tau, q = _inputs(cell, B)
    s2t = _s2tau(x[0])
    assert _rank(x[1], x[3]) == cell.R
    ser = ctx.upload_series(t, y, s2)
    try:
        out = _call(ctx, cell.entry, ser, x, tau, q, s2t)
        name = ctx.last_kernel_name()
        OBSERVED[cell.name] = name
        assert name == cell.expected()[-1], f"{cell.name}: ran {name}, dispatch restatement says {cell.expected()}"
        # identities with the other entries
        if cell.entry in ("var", "cov"):
            assert np.array_equal(out[0], ctx.celerite_predict(ser, *x[:4], tau, mu=x[4], nu=x[5])), "mean is not predict's"
        if cell.entry == "cov":
            var = ctx.celerite_predict_var(ser, *x[:4], tau, mu=x[4], nu=x[5], return_mean=False)
            diag = np.diagonal(out[1], axis1=1, axis2=2)
            assert np.all(np.abs(diag - var) <= TOL * x[0].sum(axis=1)[:, None]), "diag(cov) is not var"
        # batch invariance: each set against its single-set call
        for i in _invariance_sets(B):
            one = slice(i, i + 1)
            single = _call(ctx, cell.entry, ser, [v[one] for v in x], tau, q[one], s2t)
            same_rank = _rank(x[1][one], x[3][one]) == cell.R
            for k, (got, ref) in enumerate(zip(single, out)):
                if same_rank:
                    assert np.array_equal(got[0], ref[i]), f"set {i} differs from its single-set call"
                else:
                    err = np.max(np.abs(got[0] - ref[i])) / _unit(cell.entry, k, ref[i], x, i)
                    assert err <= TOL, f"set {i}: {err:.2e} from its single-set call at rank {_rank(x[1][one], x[3][one])}"
    finally:
        ser.free()
    # every set against the dense reference
    tally = Tally()
    if cell.entry in ("predict", "var", "cov"):
        _check_mean(out[0], x, t, y, s2, tau, tally)
    if cell.entry == "var":
        _check_var(out[1], x, t, s2, tau, tally)
    if cell.entry == "cov":
        _check_cov(out[1], x, t, s2, tau, tally)
    if cell.entry == "draws":
        _check_draws(out[0], x, t, y, s2, tau, q, s2t, tally)
    if cell.entry == "simulate":
        _check_simulate(out[0], x, t, s2, q, tally)
    record_property("kernel", name)
    record_property("worst_error", tally.worst)
    print(f"{cell.name}: ran {name}, worst error {tally.worst:.3f} of the bar over {B} sets, "
          f"{tally.exempt} of {tally.sets} checks on the 80-bit route")
    assert tally.exempt <= max(1, int(MAX_EXEMPT_FRACTION * tally.sets)), (
        f"{tally.exempt} of {tally.sets} sets needed the 80-bit route (cap {MAX_EXEMPT_FRACTION:.0%})")


@pytest.mark.gpu
def test_rank_129_is_refused_by_every_entry(pb, ctx):
    cell = Cell("refused-r129", "draws", 64, 1, N=20, M=6, S=1)
    rng = np.random.default_rng(129)
    t, y, s2 = _series(cell.N, rng)
    a, b, c, d, mu, nu = _candidates(cell, 2, rng)
    assert _rank(b, d) == 129
    tau = _tau(t, cell.M, rng)
    ser = ctx.upload_series(t, y, s2)
    try:
        for e in ENTRIES:
            with pytest.raises(Unsupported):
                expected(e, 129, 65)
            q = rng.standard_normal((2, 1, cell.N + cell.M) if e == "draws" else (2, cell.N))
            with pytest.raises(pb.PioranError) as err:
                _call(ctx, e, ser, [a, b, c, d, mu, nu], tau, q, 1e-6)
            assert err.value.code == -5, e                                            # PIORAN_EUNSUPPORTED
    finally:
        ser.free()


@pytest.mark.gpu
def test_observed_kernels_are_the_ledger():
    """After a run of the whole matrix: the last kernels the library reported are exactly the ledger's consumer entries
    (the last kernel of some cell's restatement)."""
    if len(OBSERVED) < len(ALL_CELLS):
        pytest.skip(f"only {len(OBSERVED)} of {len(ALL_CELLS)} cells ran")
    consumers = {c.expected()[-1] for c in ALL_CELLS}
    assert consumers <= LEDGER and len(consumers) == 25
    assert set(OBSERVED.values()) == consumers
