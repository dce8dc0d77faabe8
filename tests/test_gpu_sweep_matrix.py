"""Sweep matrix: every likelihood and gradient kernel instantiation the dispatch of csrc/api.cu can reach, one cell each.

A cell is one call through the public API.  It asserts two things:
  1. Context.last_kernel_name() is the kernel expected_kernel() predicts, so a dispatch change that moves a cell to another
     kernel fails here instead of silently testing a kernel that is already tested;
  2. parity of every row of the call with the CPU oracle: values through conftest.assert_parity (1e-9 relative, 80-bit twin
     for the conditioning exemption), gradients through the column-scaled 1e-8 check of test_gpu_grad.py.  The inputs are
     well-conditioned rows (see COND), so that a kernel error of 1e-7 in one amplitude or pivot stands out.

expected_kernel() restates the dispatch of csrc/api.cu in plain Python.  LEDGER lists by hand every instantiation the default
build can reach; UNREACHABLE names the compiled ones it cannot, with the reason.  The CPU test at the top checks that the cells
reach exactly the ledger on a 148-SM B200, so the matrix cannot lose a cell without a failing test on a machine with no GPU.
Batch sizes are derived from the SM count of the device, so the cells keep their kernels on a part with another SM count.

The module uses its own context: the sweep mode it switches must never leak into the shared get_context(0)."""
import zlib

import numpy as np
import pytest

from conftest import assert_parity, prior_theta, rel_err, synthetic_series
from oracle import oracle as orc
from test_gpu_grad import _check as check_grad
from test_gpu_parity import _ld_twin

TOL = 1e-9
B200_SMS = 148


# ------------------------------------------------------------------------------------------------ the dispatch, restated
def _cdiv(a, b):
    return -(-a // b)


def blk_nt(R):
    return (R + 7) // 8


def blk_ntr(R):
    return (R + 8) // 8


def blk_half(R):
    return 1 <= R % 8 <= 4


def bs_for_rank(R):
    return max(4, _cdiv(R, 8))


def blocked_enabled(R, mode):
    return mode == "auto" and R >= 1 and blk_ntr(R) <= 8


def blocked_wide_enabled(R, mode):
    return mode == "auto" and 64 < R <= 128


def blocked_nw(NT):
    return 8 if NT >= 7 else 12 if NT >= 5 else 16


def nw_for_bs(BS):
    return 12 if BS <= 5 else 10 if BS == 6 else 8


def theta_per_item(BS):       # the θ-paired kernel takes two parameter vectors per warp at block sizes <= 5
    return 16 if BS <= 5 else nw_for_bs(BS)


def plan_items(S, B, NW, num_sms, tail_items=False):
    """csrc/api.cu plan_items for one series length: (θ per item, [(first row, count), …])."""
    E = S * B
    if tail_items and S == 1 and E > NW * num_sms:
        per_wave = NW * num_sms
        full = E // per_wave * per_wave
        rem = E - full
        items = [(b, NW) for b in range(0, full, NW)]
        nit = min(num_sms, rem)
        items += [(full + rem * k // nit, rem * (k + 1) // nit - rem * k // nit) for k in range(nit)]
        return NW, items
    tpi = min(NW, max(1, _cdiv(E, num_sms)))
    items = S * _cdiv(B, tpi)
    target = _cdiv(items, num_sms) * num_sms
    tpi = min(NW, max(1, _cdiv(E, target)))
    nit = _cdiv(B, tpi)
    return tpi, [(s * B + B * k // nit, B * (k + 1) // nit - B * k // nit) for s in range(S) for k in range(nit)]


def auto_scan(N, B, R, mode, explicit):
    min_steps = 2048 if R <= 32 else 4096
    if explicit:
        min_steps //= 2
    if 25 <= R <= 63 and mode != "scalar":
        min_steps = 4096 if R <= 32 else 8192
    if R > 64:
        return N >= (4096 if mode == "scalar" else 20480) and B <= 4 and R <= 96
    return N >= min_steps and B <= 4


class Unsupported(Exception):
    """The library refuses the shape (PIORAN_EUNSUPPORTED)."""


def _blocked(R, NW):
    NT, own = blk_nt(R), R % 8 == 0
    if NT == 8 and own:
        raise Unsupported(R)
    return f"blocked<{NT},{NT + 1 if own else NT},{'true' if blk_half(R) else 'false'},{NW}>"


def _blocked_tier(R, tpi):       # launch_blocked
    return _blocked(R, 4 if tpi <= 4 else 8 if tpi <= 8 else blocked_nw(blk_nt(R)))


def _blocked_wide(R):            # dispatch_blocked_wide
    NT = blk_nt(R)
    if not 4 <= NT <= 16:
        raise Unsupported(R)
    W = 4 if NT <= 12 else 8
    if R % 8 == 0:
        return f"blocked_wide<{NT},{NT + 1},{8 if NT + 1 > 12 else W}>"
    return f"blocked_wide<{NT},{NT},{W}>"


def _shared(BS, tpi):            # dispatch_shared
    if tpi <= 4:
        return f"shared<{BS},4>"
    if tpi <= 8 and BS <= 6:
        return f"shared<{BS},8>"
    if BS <= 5:
        return f"shared_pair<{BS},8>"
    return f"shared<{BS},{nw_for_bs(BS)}>"


def _generic(BS, tpi):           # dispatch_generic
    return f"generic<{BS},{4 if tpi <= 4 else nw_for_bs(BS)}>"


def _wide(R):                    # launch_wide
    if R > 160:
        raise Unsupported(R)
    return f"wide_reg<{max(5, _cdiv(R, 16))}>" if R <= 128 else "wide"


def _blocked_grad(R, NTAN):      # dispatch_blocked_grad on the gradient's row layout (R ≡ 7 mod 8 gets its own data-row tile)
    NT = blk_nt(R)
    own = R % 8 in (0, 7)
    return f"blocked_grad<{NT},{NT + 1 if own else NT},{'true' if blk_half(R) and not own else 'false'},{NTAN}>"


def expected_kernel(entry, R, S, B, mode, num_sms, N):
    """Kernel name csrc/api.cu launches for one call.  entry: "approx" (approx_logl and its device-pointer entry), "celerite"
    (explicit coefficients), "grad_sbpl", "grad_dbpl", "grad_logshift" (approx_logl_grad, … on DoubleBendingPowerLaw, the
    log-normal model).  mode: "auto" or "scalar" (Context.set_sweep_kernel)."""
    BS = bs_for_rank(R)
    if entry == "approx":                                   # approx_logl_dev_locked
        if S == 1 and auto_scan(N, B, R, mode, False):
            return "scan_finish"
        if BS > 8:
            return _blocked_wide(R) if blocked_wide_enabled(R, mode) else _wide(R)
        if blocked_enabled(R, mode):
            if blk_nt(R) >= 4 and S * B <= 2 * num_sms:    # one CTA per evaluation
                return _blocked_wide(R)
            tpi, _ = plan_items(S, B, blocked_nw(blk_nt(R)), num_sms, tail_items=True)
            return _blocked_tier(R, tpi)
        tpi, _ = plan_items(S, B, theta_per_item(BS), num_sms)
        return _shared(BS, tpi)
    if entry == "celerite":                                 # generic_logl_locked
        if auto_scan(N, B, R, mode, True):
            return "scan_finish"
        NT, NTR = blk_nt(R), (blk_ntr(R) if R % 8 == 0 else blk_nt(R))
        tbytes = 8 * _cdiv(N, 8) * (64 * NT + 72 * NTR + 256 * NT + 32)
        if (blocked_enabled(R, mode) or blocked_wide_enabled(R, mode)) and B <= 4 * num_sms and tbytes * B <= 2 << 30:
            return _blocked_wide(R) if R > 64 or NT >= 4 else _blocked(R, 4)
        if BS > 8:
            return _wide(R)
        tpi, _ = plan_items(1, B, nw_for_bs(BS), num_sms)
        return _generic(BS, tpi)
    ND = {"grad_sbpl": 3, "grad_dbpl": 5, "grad_logshift": 3}[entry]   # approx_logl_grad_dev_locked
    logshift = entry == "grad_logshift"
    if BS > 8:
        if R > 96 or logshift:
            raise Unsupported(R)
        return f"wide_grad<{max(5, _cdiv(R, 16))}>"
    blkg = blocked_enabled(R, mode) and (blk_nt(R) + (1 if R % 8 in (0, 7) else 0)) <= 8
    if logshift and not blkg:
        raise Unsupported(R)
    if blkg:
        return _blocked_grad(R, 5 if logshift else 4 if ND == 3 else 6)
    if BS >= 6:
        return f"grad_pipe<{BS},{ND + 2}>"
    tpi, _ = plan_items(1, B * (ND + 1), 8, num_sms)
    return f"grad<{BS},{4 if tpi <= 4 else 8}>"


# ------------------------------------------------------------------------------------------------ coverage ledger
# The 23 row layouts (NT, NTR, HALF) of a block table: the data row in a row tile of its own (R ≡ 0 mod 8; for the gradient
# also R ≡ 7), HALF mode (R ≡ 1 … 4 mod 8: the last column tile carries at most 4 rows) and the plain layout.  NT = 8 has no
# own-tile layout: rank 64 is served by the scalar-pipe kernels.
LAYOUTS = ([(nt, nt + 1, "false") for nt in range(1, 8)] + [(nt, nt, "true") for nt in range(1, 9)]
           + [(nt, nt, "false") for nt in range(1, 9)])
# warps per CTA of the blocked kernel: 4 (≤ 4 θ per item), 8 (≤ 8), and the full-size CTA (16 / 12 / 8 by register budget)
BLOCKED_NW = {1: (4, 8, 16), 2: (4, 8, 16), 3: (4, 8, 16), 4: (4, 8, 16), 5: (4, 8, 12), 6: (4, 8, 12), 7: (4, 8), 8: (4, 8)}

LEDGER = (
    {f"blocked<{nt},{ntr},{half},{nw}>" for nt, ntr, half in LAYOUTS for nw in BLOCKED_NW[nt]}
    | {f"blocked_wide<{nt},{nt},4>" for nt in range(4, 13)} | {f"blocked_wide<{nt},{nt},8>" for nt in range(13, 17)}
    | {"blocked_wide<4,5,4>", "blocked_wide<5,6,4>", "blocked_wide<6,7,4>", "blocked_wide<7,8,4>",
       "blocked_wide<9,10,4>", "blocked_wide<10,11,4>", "blocked_wide<11,12,4>", "blocked_wide<12,13,8>",
       "blocked_wide<13,14,8>", "blocked_wide<14,15,8>", "blocked_wide<15,16,8>", "blocked_wide<16,17,8>"}
    | {"shared<4,4>", "shared<5,4>", "shared<6,4>", "shared<7,4>", "shared<8,4>", "shared<4,8>", "shared<5,8>", "shared<6,8>",
       "shared<6,10>", "shared<7,8>", "shared<8,8>", "shared_pair<4,8>", "shared_pair<5,8>"}
    | {"generic<4,4>", "generic<5,4>", "generic<6,4>", "generic<7,4>", "generic<8,4>",
       "generic<4,12>", "generic<5,12>", "generic<6,10>", "generic<7,8>", "generic<8,8>"}
    | {"wide_reg<5>", "wide_reg<6>", "wide_reg<7>", "wide_reg<8>", "wide"}
    | {f"blocked_grad<{nt},{ntr},{half},{ntan}>" for nt, ntr, half in LAYOUTS for ntan in (4, 5, 6)}
    | {"grad<4,4>", "grad<4,8>", "grad<5,4>", "grad<5,8>", "grad_pipe<6,5>", "grad_pipe<7,5>", "grad_pipe<8,5>",
       "grad_pipe<6,7>", "grad_pipe<7,7>", "grad_pipe<8,7>", "wide_grad<5>", "wide_grad<6>"}
)
# compiled, not reachable through the public API with default environment
UNREACHABLE = {
    "shared<4,12>": "needs PIORAN_PAIR=0 (the θ-paired kernel serves block sizes <= 5); read once per process",
    "shared<5,12>": "needs PIORAN_PAIR=0, as shared<4,12>",
    "blocked_wide<8,9,4>": "rank 64 (the only 8-tile rank with its own data-row tile) goes to the scalar-pipe kernels",
}
# reachable, covered by their own rank grids elsewhere: K3 scan (test_gpu_scan.py), dense K4 (test_gpu_dense.py), posterior
# mean and draws (test_posterior.py), JVP (test_gpu_jvp.py)
OUT_OF_SCOPE = ("scan_finish", "scan_partial", "dense_finish", "predict<·>", "generic_sim<·,·>", "wide_reg_store<·>",
                "wide_reg_sim<·>", "jvp<·>")


# ------------------------------------------------------------------------------------------------ cells
class Cell:
    """One call.  B = k·SMs + c (bk = (k, c)); R from basis and J (fused and gradient entries) or given (explicit)."""

    def __init__(self, name, entry, R, bk, mode="auto", N=101, basis="SHO", J=None):
        self.name, self.entry, self.R, self.bk, self.mode, self.N, self.basis, self.J = name, entry, R, bk, mode, N, basis, J

    def B(self, num_sms):
        return self.bk[0] * num_sms + self.bk[1]

    def expected(self, num_sms):
        return expected_kernel(self.entry, self.R, 1, self.B(num_sms), self.mode, num_sms, self.N)

    def __repr__(self):
        return self.name


def _fused(name, basis, J, bk, mode="auto", N=101, entry="approx"):
    return Cell(name, entry, 2 * J if basis == "SHO" else 3 * J, bk, mode, N, basis, J)


def _sho_j_for_layout(nt, cls):
    """SHO J whose rank 2J has the layout class cls of column tile count nt: own (R ≡ 0 mod 8), half (R ≡ 2 or 4), plain (R ≡ 6)."""
    R = {"own": 8 * nt, "half": 8 * nt - (4 if nt % 2 else 6), "plain": 8 * nt - 2}[cls]
    return R // 2


LAYOUT_CLASSES = [(nt, cls) for nt in range(1, 9) for cls in ("own", "half", "plain") if not (nt == 8 and cls == "own")]

FUSED_CELLS = []
for nt, cls in LAYOUT_CLASSES:
    J = _sho_j_for_layout(nt, cls)
    FUSED_CELLS += [_fused(f"blocked-nt{nt}-{cls}-nw4", "SHO", J, (3, 1) if nt >= 4 else (1, 37)),
                    _fused(f"blocked-nt{nt}-{cls}-nw8", "SHO", J, (6, 5))]
    if nt <= 6:
        FUSED_CELLS.append(_fused(f"blocked-nt{nt}-{cls}-nwfull", "SHO", J, (10, 3)))
    if nt >= 4:
        FUSED_CELLS.append(_fused(f"blocked_wide-nt{nt}-{cls}-small-batch", "SHO", J, (0, 5)))
FUSED_CELLS += [
    _fused("blocked-nt8-plain-drw-r63", "DRWCelerite", 21, (6, 5)),
    _fused("blocked-nt8-plain-drw-r63-nw4", "DRWCelerite", 21, (3, 1)),
]
# tail-wave plan (one series, more than one wave of full items) at each full CTA size: 16 (NT 3), 12 (NT 5), 8 (NT 8)
for nw, J in ((16, 10), (12, 19), (8, 30)):
    for tag, bk in (("+1", (nw, 1)), ("+sms-1", (nw + 1, -1)), ("+sms+1", (nw + 1, 1))):
        FUSED_CELLS.append(_fused(f"blocked-tail-nw{nw}{tag}", "SHO", J, bk))
# ranks 65 … 128 on the tensor pipe (one CTA per evaluation), with and without the data row's own tile
for nt in range(9, 17):
    FUSED_CELLS += [_fused(f"blocked_wide-nt{nt}-own", "SHO", 4 * nt, (0, 7)),
                    _fused(f"blocked_wide-nt{nt}-{'half' if nt % 2 else 'plain'}", "SHO", 4 * nt - (3 if nt % 2 else 1), (0, 7))]
FUSED_CELLS += [_fused("shared-r64-4w", "SHO", 32, (3, 1)), _fused("shared-r64-8w", "SHO", 32, (6, 5)),
                _fused("shared-r64-full", "SHO", 32, (10, 3)), _fused("wide-r150-drw", "DRWCelerite", 50, (0, 5))]

# scalar-pipe selection (PIORAN_SWEEP_SCALAR): one rank per block size 4 … 8
SCALAR_J = {4: 15, 5: 19, 6: 23, 7: 27, 8: 31}
SCALAR_CELLS = [_fused(f"shared-bs{bs}-4w", "SHO", J, (3, 1), "scalar") for bs, J in SCALAR_J.items()]
SCALAR_CELLS += [_fused(f"shared-bs{bs}-8w", "SHO", SCALAR_J[bs], (6, 5), "scalar") for bs in (4, 5, 6)]
SCALAR_CELLS += [_fused("shared-bs6-10w", "SHO", 23, (9, 5), "scalar"),
                 _fused("shared-bs7-full", "SHO", 27, (10, 3), "scalar"),
                 _fused("shared-bs8-full-drw-r63", "DRWCelerite", 21, (10, 3), "scalar"),
                 _fused("shared_pair-bs4", "SHO", 15, (10, 3), "scalar"),
                 _fused("shared_pair-bs5-drw", "DRWCelerite", 13, (12, 7), "scalar")]
SCALAR_CELLS += [_fused(f"wide_reg-ts{ts}", "SHO", J, (0, 9), "scalar") for ts, J in ((5, 37), (6, 45), (7, 55), (8, 63))]

# explicit coefficients: mixed complex and real terms, odd ranks
GENERIC_RANKS = {4: 29, 5: 37, 6: 45, 7: 53, 8: 63}
EXPLICIT_CELLS = [Cell(f"generic-bs{bs}-full", "celerite", R, (4, 1)) for bs, R in GENERIC_RANKS.items()]
EXPLICIT_CELLS += [Cell(f"generic-bs{bs}-4w-scalar", "celerite", R, (3, 1), "scalar") for bs, R in GENERIC_RANKS.items()]
EXPLICIT_CELLS += [Cell("generic-r64-4w", "celerite", 64, (2, 9))]
EXPLICIT_CELLS += [Cell(f"wide_reg-ts{ts}-explicit", "celerite", R, (4, 1)) for ts, R in ((5, 75), (6, 89), (7, 105), (8, 121))]
EXPLICIT_CELLS += [Cell(f"per-theta-table-r{R}", "celerite", R, (0, 37)) for R in (5, 7, 8, 11, 13, 16, 19, 23, 24, 32, 45, 75)]
EXPLICIT_CELLS += [Cell("wide-r141-explicit", "celerite", 141, (0, 5))]
NAN_CELLS = [Cell("generic-bs5-nan-first-pivot", "celerite", 37, (4, 1)), Cell("wide_reg-nan-first-pivot", "celerite", 89, (4, 1))]

# gradients: every layout for each tangent count (4: SingleBendingPowerLaw, 6: DoubleBendingPowerLaw, 5: the log-normal model)
GRAD_CELLS = []
for nt, cls in LAYOUT_CLASSES:
    J = _sho_j_for_layout(nt, cls)
    for entry in ("grad_sbpl", "grad_dbpl", "grad_logshift"):
        GRAD_CELLS.append(_fused(f"blocked_grad-nt{nt}-{cls}-{entry}", "SHO", J, (0, 37), entry=entry))
GRAD_CELLS += [_fused("blocked_grad-own-r15-drw", "DRWCelerite", 5, (0, 37), entry="grad_sbpl"),
               _fused("blocked_grad-own-r39-drw", "DRWCelerite", 13, (0, 37), entry="grad_sbpl"),
               _fused("grad_pipe-r63-drw", "DRWCelerite", 21, (0, 37), entry="grad_sbpl"),
               _fused("grad_pipe-r64", "SHO", 32, (0, 37), entry="grad_sbpl"),
               _fused("grad_pipe-r64-dbpl", "SHO", 32, (0, 37), entry="grad_dbpl"),
               _fused("grad_pipe-r63-drw-dbpl", "DRWCelerite", 21, (0, 37), entry="grad_dbpl"),
               _fused("wide_grad-ts5", "SHO", 40, (0, 12), entry="grad_sbpl"),
               _fused("wide_grad-ts6-drw", "DRWCelerite", 30, (0, 12), entry="grad_sbpl")]
for bs, J in ((6, 23), (7, 27)):
    for entry in ("grad_sbpl", "grad_dbpl"):
        GRAD_CELLS.append(_fused(f"grad_pipe-bs{bs}-{entry}-scalar", "SHO", J, (0, 37), "scalar", entry=entry))
for bs, J in ((4, 10), (5, 19)):
    GRAD_CELLS += [_fused(f"grad-bs{bs}-4w-scalar", "SHO", J, (0, 101), "scalar", entry="grad_sbpl"),
                   _fused(f"grad-bs{bs}-8w-scalar", "SHO", J, (2, 5), "scalar", entry="grad_sbpl")]

# series lengths around the 8-step block and 3 TMA stages (blocked), the 16-step chunk (shared), the 4-step chunk (generic)
EDGE_N = (1, 2, 7, 8, 9, 16, 17, 24, 25, 33)
EDGE_FAMILIES = {
    "blocked": lambda N: _fused(f"edge-blocked-N{N}", "SHO", 10, (10, 3), N=N),
    "blocked_wide": lambda N: _fused(f"edge-blocked_wide-N{N}", "SHO", 45, (0, 7), N=N),
    "shared_pair": lambda N: _fused(f"edge-shared_pair-N{N}", "SHO", 10, (10, 3), "scalar", N=N),
    "shared": lambda N: _fused(f"edge-shared-N{N}", "SHO", 27, (10, 3), "scalar", N=N),
    "wide_reg": lambda N: _fused(f"edge-wide_reg-N{N}", "SHO", 45, (0, 7), "scalar", N=N),
    "generic": lambda N: Cell(f"edge-generic-N{N}", "celerite", 29, (4, 1), N=N),
    "blocked_grad": lambda N: _fused(f"edge-blocked_grad-N{N}", "SHO", 10, (0, 37), N=N, entry="grad_sbpl"),
}
EDGE_CELLS = [make(N) for make in EDGE_FAMILIES.values() for N in EDGE_N]

HEADLINE = _fused("dev-headline", "DRWCelerite", 20, (0, 65536), N=1000)   # bench.py's timed step

ALL_CELLS = FUSED_CELLS + SCALAR_CELLS + EXPLICIT_CELLS + NAN_CELLS + GRAD_CELLS + EDGE_CELLS + [HEADLINE]


def test_ledger_is_exactly_what_the_cells_reach():
    """CPU: at 148 SMs the cells reach every ledger entry and nothing else; no cell is refused."""
    reached = {c.expected(B200_SMS) for c in ALL_CELLS}
    assert reached - LEDGER == set(), f"cells reach kernels missing from the ledger: {sorted(reached - LEDGER)}"
    assert LEDGER - reached == set(), f"ledger entries no cell reaches: {sorted(LEDGER - reached)}"
    assert not LEDGER & set(UNREACHABLE)
    assert len({c.name for c in ALL_CELLS}) == len(ALL_CELLS)


def test_expected_kernel_restates_known_dispatch_points():
    """CPU: fixed points of the dispatch that other files and DESIGN.md rely on."""
    assert expected_kernel("approx", 60, 1, 65536, "auto", 148, 1000) == "blocked<8,8,true,8>"      # bench.py's step
    assert expected_kernel("approx", 40, 1, 67, "scalar", 148, 485) == "shared<5,4>"
    assert expected_kernel("approx", 64, 1, 67, "auto", 148, 485) == "shared<8,4>"
    assert expected_kernel("approx", 60, 1, 296, "auto", 148, 485) == "blocked_wide<8,8,4>"
    assert expected_kernel("approx", 60, 1, 297, "auto", 148, 485) == "blocked<8,8,true,4>"
    assert expected_kernel("grad_sbpl", 63, 1, 8, "auto", 148, 485) == "grad_pipe<8,5>"
    assert expected_kernel("grad_sbpl", 39, 1, 8, "auto", 148, 485) == "blocked_grad<5,6,false,4>"
    assert expected_kernel("celerite", 20, 1, 6475, "auto", 148, 485) == "generic<4,12>"
    assert expected_kernel("approx", 40, 1, 1, "auto", 148, 8192) == "scan_finish"
    with pytest.raises(Unsupported):
        expected_kernel("grad_logshift", 40, 1, 8, "scalar", 148, 101)
    # the tail-wave plan: whole waves of full items, then the remainder over every SM
    tpi, items = plan_items(1, 8 * 148 + 149, 8, 148, tail_items=True)
    assert tpi == 8 and len(items) == 148 + 148 and sum(n for _, n in items) == 8 * 148 + 149
    assert [n for _, n in items[148:]].count(2) == 1
    tpi, items = plan_items(1, 3 * 148 + 1, 16, 148)
    assert tpi == 4 and sum(n for _, n in items) == 3 * 148 + 1 and {n for _, n in items} == {3, 4}


# ------------------------------------------------------------------------------------------------ GPU fixtures and inputs
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


def _run_on(ctx, cell, num_sms, fn):
    """Runs fn() in the cell's sweep mode and checks the kernel it launched."""
    ctx.set_sweep_kernel(cell.mode)
    out = fn()
    name = ctx.last_kernel_name()
    OBSERVED[cell.name] = name
    assert name == cell.expected(num_sms), f"{cell.name}: ran {name}, dispatch restatement says {cell.expected(num_sms)}"
    return out


def _seed(cell):
    return zlib.crc32(cell.name.encode())


# Inputs are well-conditioned rows: the FP64 reference value lies within COND of its 80-bit twin.  The parity bar then measures
# the kernel, not the rounding amplification of an ill-conditioned covariance (steep PSD slopes, where any two FP64 operation
# orders differ by 1e-9 … 1e-7: bench.py's parity triage, test_gpu_parity.py with conftest's exemption).  A perturbation of a
# kernel by 1e-7 in one amplitude or pivot still moves these rows far beyond the bar.
COND = 1e-12
_POOLS = {}


def _cond(model, th, f_min, f_max, J, basis, t, y, s2, logshift=False):
    """|FP64 reference − 80-bit twin| / max(1, |twin|) per row (threaded oracle)."""
    if logshift:
        want = orc.approx_logl_logshift_grad_batch(model, th, f_min, f_max, J, t, y, s2, basis=basis, nthreads=0)[0]
        ld = orc.approx_logl_logshift_grad_batch(model, th, f_min, f_max, J, t, y, s2, basis=basis, nthreads=0, long_double=True)[0]
    else:
        want = orc.approx_logl_batch(model, th, f_min, f_max, J, t, y, s2, basis=basis, nthreads=0)
        ld = orc.approx_logl_grad_batch(model, th, f_min, f_max, J, t, y, s2, basis=basis, nthreads=0, long_double=True)[0]
    return rel_err(want, ld)


def _pick(key, B, candidates, cond):
    """The first B rows of the candidate stream whose conditioning is below COND (cached per key, grown on demand)."""
    pool = _POOLS.get(key)
    k = 0
    while pool is None or len(pool) < B:
        cand = candidates(k)
        good = cand[cond(cand) <= COND]
        pool = good if pool is None else np.concatenate([pool, good])
        k += 1
        assert k <= 64, f"{key}: fewer than {B} well-conditioned rows in {k} candidate batches"
    _POOLS[key] = pool
    return pool[:B].copy()


def _theta(g, B, basis, J, N, f_min=None, f_max=None, series=None):
    """Distinct, well-conditioned parameter vectors: golden_single rows and prior draws, alternating in batches of 256.
    DRWCelerite shifts α₂ by 1 as the other GPU tests do (its basis allows steeper slopes)."""
    t, y, s2 = series if series is not None else _prefix(g, N)
    f_min = g.f_min if f_min is None else f_min
    f_max = g.f_max if f_max is None else f_max
    order = np.random.default_rng(J).permutation(len(g.theta))

    def candidates(k):
        gold = g.theta[order[(k // 2) * 256 % len(order):][:256]].copy()
        if basis == "DRWCelerite":
            gold[:, 2] += 1.0
        if k % 2 == 0:
            return gold
        return prior_theta(256, f_min, f_max, y.mean(), max(y.std(), 0.1), seed=1000 * J + k,
                           alpha2_max=6.0 if basis == "DRWCelerite" else 4.0)

    def cond(th):
        return _cond("SBPL", th, f_min, f_max, J, basis, t, y, s2)
    return _pick(("SBPL", basis, J, N, len(t), float(f_min)), B, candidates, cond)


def _prefix(g, N):
    return g.t[:N].copy(), g.y[:N].copy(), g.s2[:N].copy()


def _fused_value(pb, ctx, g, cell, num_sms):
    B = cell.B(num_sms)
    t, y, s2 = _prefix(g, cell.N)
    th = _theta(g, B, cell.basis, cell.J, cell.N)
    spec = pb.make_spec(g.model, g.f_min, g.f_max, cell.J, basis_function=cell.basis)
    ser = ctx.upload_series(t, y, s2)
    got = _run_on(ctx, cell, num_sms, lambda: ctx.approx_logl(ser, spec, th)[0])
    want = orc.approx_logl_batch("SBPL", th, g.f_min, g.f_max, cell.J, t, y, s2, basis=cell.basis, nthreads=0)
    assert got.shape == (B,)
    report = assert_parity(got, want, th, _ld_twin("SBPL", g.f_min, g.f_max, cell.J, cell.basis, t, y, s2), TOL, label=cell.name)
    return ser, spec, th, got, report


@pytest.mark.gpu
@pytest.mark.parametrize("cell", FUSED_CELLS, ids=repr)
def test_fused_value(pb, ctx, num_sms, golden_single, cell):
    ser, *_ = _fused_value(pb, ctx, golden_single, cell, num_sms)
    ser.free()


@pytest.mark.gpu
@pytest.mark.parametrize("cell", SCALAR_CELLS, ids=repr)
def test_fused_value_scalar_pipe(pb, ctx, num_sms, golden_single, cell, record_property):
    """The scalar-pipe kernels, and their agreement with the default kernel on the same rows.  Both are held to the oracle;
    their difference is reported (record_property / stdout), bounded only by twice the parity bar outside exempted rows."""
    ser, spec, th, got, report = _fused_value(pb, ctx, golden_single, cell, num_sms)
    g = golden_single
    t, y, s2 = _prefix(g, cell.N)
    ctx.set_sweep_kernel("auto")
    dflt = ctx.approx_logl(ser, spec, th)[0]
    ctx.set_sweep_kernel("scalar")
    ser.free()
    want = orc.approx_logl_batch("SBPL", th, g.f_min, g.f_max, cell.J, t, y, s2, basis=cell.basis, nthreads=0)
    report += assert_parity(dflt, want, th, _ld_twin("SBPL", g.f_min, g.f_max, cell.J, cell.basis, t, y, s2), TOL,
                            label=cell.name + " (default kernel)")
    diff = rel_err(got, dflt)
    keep = np.isfinite(dflt)
    keep[[r[0] for r in report]] = False
    assert np.array_equal(np.isfinite(got), np.isfinite(dflt))
    worst = float(diff[keep].max()) if keep.any() else 0.0
    record_property("scalar_vs_default_max_rel", worst)
    print(f"{cell.name}: scalar vs default kernel, largest relative difference {worst:.3e} over {int(keep.sum())} rows")
    assert worst <= 2 * TOL


def _explicit_batch(R, B, N, seed, t, y, s2):
    """B coefficient sets of rank R: complex terms (random-sign b and d, |b d| < a c) and one or two real terms (b = d = 0,
    one with a negative amplitude), interleaved; per-set μ, ν, y and σ²."""
    rng = np.random.default_rng(seed)
    nreal = 1 if R % 2 else 2
    ncx = (R - nreal) // 2
    Jt = ncx + nreal
    a = np.empty((B, Jt)); b = np.zeros((B, Jt)); c = np.empty((B, Jt)); d = np.zeros((B, Jt))
    order = rng.permutation(Jt)
    cx, re = order[:ncx], order[ncx:]
    a[:, cx] = rng.uniform(0.2, 1.0, (B, ncx)) / Jt
    c[:, cx] = np.exp(rng.uniform(np.log(0.02), np.log(3.0), (B, ncx)))
    d[:, cx] = rng.choice([-1.0, 1.0], (B, ncx)) * np.exp(rng.uniform(np.log(0.05), np.log(5.0), (B, ncx)))
    b[:, cx] = rng.uniform(-0.9, 0.9, (B, ncx)) * a[:, cx] * c[:, cx] / np.abs(d[:, cx])
    a[:, re] = rng.uniform(0.2, 1.0, (B, nreal)) / Jt
    a[:, re[0]] *= -0.1
    c[:, re] = np.exp(rng.uniform(np.log(0.05), np.log(2.0), (B, nreal)))
    mu = rng.normal(0.0, 0.3, B)
    nu = rng.uniform(0.5, 2.0, B)
    yb = y[None, :] + rng.normal(0.0, 0.05, (B, N))
    sb = s2[None, :] * rng.uniform(0.5, 2.0, (B, N))
    return [a, b, c, d, mu, nu, yb, sb]


def _explicit_cell(pb, ctx, num_sms, golden_single, cell, nan_rows=()):
    """nan_rows: all amplitudes of these sets negative, so the first pivot Σa + νσ²₀ is negative and log L is NaN (log
    without abs, celerite_solver.jl:126)."""
    g = golden_single
    B = cell.B(num_sms)
    t, y, s2 = _prefix(g, cell.N)
    cand = _explicit_batch(cell.R, B + B // 2 + 16, cell.N, _seed(cell), t, y, s2)

    def ref(arrs, i, long_double=False):
        a, b, c, d, mu, nu, yb, sb = arrs
        return orc.celerite_logl(a[i], b[i], c[i], d[i], t, yb[i] - mu[i], nu[i] * sb[i], long_double=long_double)
    fp = np.array([ref(cand, i) for i in range(len(cand[0]))])
    ld = np.array([ref(cand, i, True) for i in range(len(cand[0]))])
    keep = np.flatnonzero(rel_err(fp, ld) <= COND)[:B]          # well-conditioned sets (see COND)
    assert len(keep) == B, f"{cell.name}: {len(keep)} of {len(fp)} candidate sets are well-conditioned"
    arrs = [x[keep].copy() for x in cand]
    want = fp[keep]
    for i in nan_rows:
        arrs[0][i] = -np.abs(arrs[0][i]) * 10
        want[i] = ref(arrs, i)
    a, b, c, d, mu, nu, yb, sb = arrs
    ser = ctx.upload_series(t, y, s2)
    got = _run_on(ctx, cell, num_sms, lambda: ctx.celerite_logl(ser, a, b, c, d, mu=mu, nu=nu, y_batch=yb, s2_batch=sb))
    ser.free()
    assert_parity(got, want, np.arange(B), lambda i: ref(arrs, int(i), True), TOL, label=cell.name)
    return got, want


@pytest.mark.gpu
@pytest.mark.parametrize("cell", EXPLICIT_CELLS, ids=repr)
def test_explicit_coefficients(pb, ctx, num_sms, golden_single, cell):
    got, want = _explicit_cell(pb, ctx, num_sms, golden_single, cell)
    assert np.isfinite(want).all()


@pytest.mark.gpu
@pytest.mark.parametrize("cell", NAN_CELLS, ids=repr)
def test_explicit_nan_first_pivot(pb, ctx, num_sms, golden_single, cell):
    """Negative first pivot → NaN in exactly the rows where the reference gives NaN (test_nonfinite_semantics_match_reference),
    on rows spread over the items of the call; the other rows stay at parity."""
    B = cell.B(num_sms)
    bad = (0, 5, B // 2, B - 1)
    got, want = _explicit_cell(pb, ctx, num_sms, golden_single, cell, nan_rows=bad)
    assert np.isnan(want[list(bad)]).all() and np.isnan(got[list(bad)]).all()
    assert np.array_equal(np.isnan(got), np.isnan(want))


def _grad_inputs(cell, B, golden_single, golden_double, seed):
    """(theta, t, y, s2, g, model) of a gradient cell: well-conditioned golden rows only (the gradient check has no
    conditioning exemption)."""
    if cell.entry == "grad_dbpl":
        g, model = golden_double, "DBPL"
    else:
        g, model = golden_single, "SBPL"
    N = cell.N
    logshift = cell.entry == "grad_logshift"
    if logshift:
        t, y, s2 = g.t[:N].copy(), g.y_raw[:N].copy(), (g.yerr ** 2)[:N].copy()
    else:
        t, y, s2 = _prefix(g, N)
    order = np.random.default_rng(seed).permutation(len(g.theta))

    def candidates(k):
        th = g.theta[order[k * 128:(k + 1) * 128]].copy()
        if cell.basis == "DRWCelerite":
            th[:, 2] += 1.0
        if logshift:
            th = np.column_stack([th, np.random.default_rng(seed + k).uniform(-0.5, 0.9, len(th)) * y.min()])
        return th

    def cond(th):
        return _cond(model, th, g.f_min, g.f_max, cell.J, cell.basis, t, y, s2, logshift)
    th = _pick((cell.name,), B, candidates, cond)
    return th, t, y, s2, g, model


def _grad_cell(pb, ctx, num_sms, golden_single, golden_double, cell):
    th, t, y, s2, g, model = _grad_inputs(cell, cell.B(num_sms), golden_single, golden_double, _seed(cell))
    spec = pb.make_spec(g.model, g.f_min, g.f_max, cell.J, basis_function=cell.basis)
    ser = ctx.upload_series(t, y, s2)
    if cell.entry == "grad_logshift":
        val, grad = _run_on(ctx, cell, num_sms, lambda: ctx.approx_logl_logshift_grad(ser, spec, th))
        plain = ctx.approx_logl_logshift(ser, spec, th)
        oval, ograd = orc.approx_logl_logshift_grad_batch(model, th, g.f_min, g.f_max, cell.J, t, y, s2, basis=cell.basis, nthreads=0)
    else:
        val, grad = _run_on(ctx, cell, num_sms, lambda: ctx.approx_logl_grad(ser, spec, th))
        plain = ctx.approx_logl(ser, spec, th)[0]
        oval, ograd = orc.approx_logl_grad_batch(model, th, g.f_min, g.f_max, cell.J, t, y, s2, basis=cell.basis, nthreads=0)
    ser.free()
    assert grad.shape == th.shape
    verr = rel_err(val, oval)
    assert verr.max() <= TOL, f"value parity {verr.max():.3e}"
    assert rel_err(val, plain).max() <= TOL, "value column differs from the likelihood entry"
    check_grad(grad, ograd)


@pytest.mark.gpu
@pytest.mark.parametrize("cell", GRAD_CELLS, ids=repr)
def test_gradient(pb, ctx, num_sms, golden_single, golden_double, cell):
    _grad_cell(pb, ctx, num_sms, golden_single, golden_double, cell)


@pytest.mark.gpu
def test_logshift_gradient_refused_under_scalar_pipe(pb, ctx, golden_single):
    """The log-shift gradient exists only on the tensor-pipe kernel: the scalar selection refuses it rather than computing it
    on another path."""
    g = golden_single
    ser = ctx.upload_series(g.t[:101], g.y_raw[:101], (g.yerr ** 2)[:101])
    spec = pb.make_spec(g.model, g.f_min, g.f_max, 20)
    th = np.column_stack([g.theta[:4], np.full(4, 0.5 * g.y_raw[:101].min())])
    ctx.set_sweep_kernel("scalar")
    try:
        with pytest.raises(pb.PioranError):
            ctx.approx_logl_logshift_grad(ser, spec, th)
    finally:
        ctx.set_sweep_kernel("auto")
    ctx.approx_logl_logshift_grad(ser, spec, th)      # and the default selection computes it
    assert ctx.last_kernel_name() == expected_kernel("grad_logshift", 40, 1, 4, "auto", 148, 101) == "blocked_grad<5,6,false,5>"
    ser.free()


@pytest.mark.gpu
@pytest.mark.parametrize("cell", EDGE_CELLS, ids=repr)
def test_series_length_edges(pb, ctx, num_sms, golden_single, golden_double, cell):
    if cell.entry == "approx":
        ser, *_ = _fused_value(pb, ctx, golden_single, cell, num_sms)
        ser.free()
    elif cell.entry == "celerite":
        _explicit_cell(pb, ctx, num_sms, golden_single, cell)
    else:
        _grad_cell(pb, ctx, num_sms, golden_single, golden_double, cell)


@pytest.mark.gpu
def test_device_pointer_entries_at_the_benchmark_shape(pb, ctx, num_sms, golden_single):
    """bench.py's timed step (DRWCelerite J = 20, N = 1 000, B = 65 536) through approx_logl_dev on torch buffers: bit for bit
    the host entry; against the oracle on the first and last row of every item of the first and last full wave, every row
    of the tail wave and 256 seeded rows (well-conditioned parameter vectors are placed there, prior draws elsewhere).
    approx_logl_grad_dev likewise on a small batch."""
    import torch
    cell = HEADLINE
    B = cell.B(num_sms)
    t, y, s2, f_min, f_max = synthetic_series(cell.N, seed=1234, basis="DRWCelerite")
    nw = blocked_nw(blk_nt(cell.R))
    _, items = plan_items(1, B, nw, num_sms, tail_items=True)
    nfull = B // (nw * num_sms) * num_sms
    rows = set()
    for beg, n in items[:num_sms] + items[nfull - num_sms:nfull]:
        rows |= {beg, beg + n - 1}
    for beg, n in items[nfull:]:
        rows |= set(range(beg, beg + n))
    rows |= set(np.random.default_rng(7).choice(B, 256, replace=False).tolist())
    rows = np.array(sorted(rows))
    assert len(items) - nfull > 0 and rows.max() == B - 1
    Bg = 37
    good = _theta(golden_single, len(rows) + Bg, "DRWCelerite", cell.J, cell.N, f_min, f_max, (t, y, s2))
    th = prior_theta(B, f_min, f_max, y.mean(), y.std(), seed=42, alpha2_max=6.0)
    th[rows] = good[:len(rows)]
    spec = pb.make_spec("SingleBendingPowerLaw", f_min, f_max, cell.J, basis_function="DRWCelerite")
    ser = ctx.upload_series(t, y, s2)
    th_d = torch.from_numpy(th).cuda()
    out_d = torch.full((B,), float("nan"), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    _run_on(ctx, cell, num_sms, lambda: ctx.approx_logl_dev([ser], [spec], B, th_d.data_ptr(), out_d.data_ptr()))
    ctx.synchronize()
    got = out_d.cpu().numpy()
    host = ctx.approx_logl(ser, spec, th)[0]
    assert np.array_equal(got, host, equal_nan=True)
    want = orc.approx_logl_batch("SBPL", th[rows], f_min, f_max, cell.J, t, y, s2, basis="DRWCelerite", nthreads=0)
    assert_parity(got[rows], want, th[rows], _ld_twin("SBPL", f_min, f_max, cell.J, "DRWCelerite", t, y, s2), TOL,
                  label="dev-headline")
    # gradient: device pointers against the host entry and the oracle
    thg = good[len(rows):]
    thg_d = torch.from_numpy(thg).cuda()
    logl_d = torch.empty(Bg, dtype=torch.float64, device="cuda")
    grad_d = torch.empty((Bg, thg.shape[1]), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    ctx.approx_logl_grad_dev(ser, spec, Bg, thg_d.data_ptr(), logl_d.data_ptr(), grad_d.data_ptr())
    ctx.synchronize()
    assert ctx.last_kernel_name() == expected_kernel("grad_sbpl", cell.R, 1, Bg, "auto", num_sms, cell.N)
    val, grad = ctx.approx_logl_grad(ser, spec, thg)
    assert np.array_equal(logl_d.cpu().numpy(), val, equal_nan=True) and np.array_equal(grad_d.cpu().numpy(), grad, equal_nan=True)
    oval, ograd = orc.approx_logl_grad_batch("SBPL", thg, f_min, f_max, cell.J, t, y, s2, basis="DRWCelerite", nthreads=0)
    assert rel_err(val, oval).max() <= TOL
    check_grad(grad, ograd)
    ser.free()


@pytest.mark.gpu
def test_kernel_name_probe(pb, num_sms, golden_single):
    """Empty before the first launch, the size check of the buffer, and PIORAN_EUNSUPPORTED on a device group."""
    import ctypes as C
    from pioran_b200._lib import PioranError
    g = golden_single
    fresh = pb.Context(0)
    try:
        assert fresh.last_kernel_name() == ""
        ser = fresh.upload_series(g.t, g.y, g.s2)
        fresh.approx_logl(ser, pb.make_spec(g.model, g.f_min, g.f_max, 20), g.theta[:3])
        name = fresh.last_kernel_name()
        assert name == expected_kernel("approx", 40, 1, 3, "auto", num_sms, len(g.t))
        buf = C.create_string_buffer(len(name) + 1)
        assert fresh.lib.pioran_ctx_last_kernel_name(fresh.h, buf, len(name) + 1) == 0 and buf.value.decode() == name
        assert fresh.lib.pioran_ctx_last_kernel_name(fresh.h, buf, len(name)) == -1     # PIORAN_EINVAL: no room for the NUL
    finally:
        fresh.close()
    group = pb.Context([0])
    try:
        with pytest.raises(PioranError) as e:
            group.last_kernel_name()
        assert e.value.code == -5                                                          # PIORAN_EUNSUPPORTED
    finally:
        group.close()


@pytest.mark.gpu
def test_observed_kernels_are_the_ledger():
    """After a run of the whole matrix: the kernels the library reported are exactly the ledger."""
    if len(OBSERVED) < len(ALL_CELLS):
        pytest.skip(f"only {len(OBSERVED)} of {len(ALL_CELLS)} cells ran")
    assert set(OBSERVED.values()) == LEDGER
