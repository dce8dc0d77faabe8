"""Cost of the Lomb–Scargle periodograms K9 (csrc/lsp.cuh, pioran_lombscargle) at two shapes:

  1. the posterior predictive check: P = 1 000 draws from pioran_celerite_simulate on the simu_single series (N = 485), one per
     posterior sample of the shipped chain (SingleBendingPowerLaw + SHO J = 20, the sample's ν and μ), weighted by 1/σ², on
     F = 1 000 log-spaced frequencies from 1/T to 1/(2·min Δt);
  2. a large shape: B = 1 000 rows, N = 2 000 irregular times, F = 25 000 (LombScargle.jl's automatic grid size, ≈ 12.5·N).
Host clock around calls that end in a device synchronise (every host entry of the C ABI does); the median of `--reps` timed
calls after `--warmup` untimed ones.  The device time between the events around the launches (output copies included) is
reported beside it, and the kernels' own device time from torch.profiler in a separate call.  Achieved rate:
F_lsp = 4·B·N·F FLOP (the product [B × N] · [N × 2F] as multiply-adds) over each time, next to the measured FP64 peak of BASELINE.md (36.97 TFLOP/s DFMA, 37.1 DMMA).  The CPU figure is scipy.signal.lombscargle
on a few rows, one row at a time, extrapolated to B.  The card name, power limit and max SM clock are read in the same run.
A spot check against the numpy restatement runs on a few rows of each shape (on every F/1000-th frequency).

    python tools/lsp_bench.py [--out FILE.json]
"""
import argparse
import json
import os
import sys
import time

import numpy as np
from scipy import signal

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests", "tools", "proto"))
import lsp_math as lm  # noqa: E402
import pioran_b200 as pb  # noqa: E402
import workloads as wl  # noqa: E402
from postvar_bench import card, timed  # noqa: E402

PEAK_TFLOPS = 36.97


def kernel_seconds(fn):
    """Device time of the K9 kernels of one call (torch.profiler, CUDA activity), by kernel; None when it cannot be read."""
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.init()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
        out = {}
        for row in prof.key_averages():
            if "lsp_" in row.key:
                us = getattr(row, "device_time_total", None)
                out[row.key] = (us if us is not None else row.cuda_time_total) * 1e-6
        return out or None
    except Exception as e:   # noqa: BLE001 — the number is then reported as not measured
        print("kernel times not measured:", e, flush=True)
        return None


def measure(ctx, ser, t, s2, Y, freq, warmup, reps, cpu_rows):
    B, N, F = Y.shape[0], len(t), len(freq)
    weighted = s2 is not None
    P = ctx.lombscargle(ser, freq, y_batch=Y, weighted=weighted)
    k, sel = min(4, B), slice(None, None, max(1, F // 1000))
    want = lm.lombscargle(t, Y[:k], freq[sel], s2)
    check = float(np.nanmax(np.abs(P[:k, sel] - want)))
    call = timed(lambda: ctx.lombscargle(ser, freq, y_batch=Y, weighted=weighted), warmup, reps)
    dev = ctx.last_kernel_ms() * 1e-3
    w = None if s2 is None else 1 / s2
    t0 = time.perf_counter()
    for i in range(cpu_rows):
        signal.lombscargle(t, Y[i], 2 * np.pi * freq, weights=w, floating_mean=True, normalize="normalize")
    cpu_row = (time.perf_counter() - t0) / cpu_rows
    flop = 4.0 * B * N * F
    kern = kernel_seconds(lambda: ctx.lombscargle(ser, freq, y_batch=Y, weighted=weighted))
    prod = sum(v for k, v in kern.items() if "product" in k) if kern else None
    return {"kernels_s": kern if kern else "not measured", "product_kernel_s": prod if prod else "not measured",
            "tflops_product_kernel": flop / prod * 1e-12 if prod else "not measured",
            "share_of_peak_product_kernel": flop / prod * 1e-12 / PEAK_TFLOPS if prod else "not measured",
            "B": B, "N": N, "F": F, "weighted": weighted, "kernel": ctx.last_kernel_name(), "call_s": call,
            "device_events_s": dev, "flop": flop, "tflops_call": flop / call * 1e-12, "tflops_device": flop / dev * 1e-12,
            "peak_tflops_fp64": PEAK_TFLOPS, "share_of_peak_device": flop / dev * 1e-12 / PEAK_TFLOPS,
            "cpu_scipy_row_s": cpu_row, "cpu_rows_timed": cpu_rows, "cpu_scipy_extrapolated_s": cpu_row * B,
            "check_vs_lsp_math": check}


def report(name, r):
    print(f"{name}: B={r['B']} N={r['N']} F={r['F']} [{r['kernel']}]: call {r['call_s'] * 1e3:.2f} ms "
          f"({r['tflops_call']:.2f} TFLOP/s), device {r['device_events_s'] * 1e3:.2f} ms ({r['tflops_device']:.2f} TFLOP/s, "
          f"{r['share_of_peak_device']:.1%} of {PEAK_TFLOPS} FP64); scipy {r['cpu_scipy_row_s'] * 1e3:.2f} ms per row, "
          f"{r['cpu_scipy_extrapolated_s']:.1f} s extrapolated to B; vs lsp_math {r['check_vs_lsp_math']:.1e}", flush=True)
    if isinstance(r["product_kernel_s"], float):
        print(f"  product kernel {r['product_kernel_s'] * 1e3:.3f} ms: {r['tflops_product_kernel']:.2f} TFLOP/s, "
              f"{r['share_of_peak_product_kernel']:.1%} of the FP64 peak; all K9 kernels: "
              + ", ".join(f"{k.split('(')[0]} {v * 1e3:.3f} ms" for k, v in r["kernels_s"].items()), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    ctx = pb.get_context(0)
    res = {"card": card()}
    print("card (name, power limit, max SM clock):", res["card"], flush=True)

    # 1. the check: one draw per posterior sample on the data times, then their periodograms
    ts = np.loadtxt(os.path.join(ROOT, "tests", "golden", "simu_single_subset_time_series.txt"))
    t, y_raw, yerr = (np.ascontiguousarray(c) for c in ts.T)
    y, s2 = np.log(y_raw), yerr ** 2 / y_raw ** 2
    f_min, f_max = 1 / (t[-1] - t[0]), 0.5 / np.min(np.diff(t))
    theta = np.load(os.path.join(ROOT, "tests", "golden", "chains.npz"))["simu_single"][:1000, 2:8]
    P = theta.shape[0]
    spec = pb.make_spec("SingleBendingPowerLaw", f_min, f_max, 20, basis_function="SHO")
    a, b, c, d = ctx.approx_coeffs(spec, theta[:, :4])
    ser = ctx.upload_series(t, y, s2)
    q = np.random.default_rng(0).standard_normal((P, len(t)))
    draws = ctx.celerite_simulate(ser, a, b, c, d, q, nu=theta[:, 4]) + theta[:, 5:6]
    sim_s = timed(lambda: ctx.celerite_simulate(ser, a, b, c, d, q, nu=theta[:, 4]), args.warmup, args.reps)
    freq = np.geomspace(f_min, f_max, 1000)
    res["check"] = {"simulate_s": sim_s, **measure(ctx, ser, t, s2, draws, freq, args.warmup, args.reps, 8)}
    report("posterior predictive check", res["check"])
    print(f"  the {P} draws (pioran_celerite_simulate): {sim_s * 1e3:.2f} ms", flush=True)
    ser.free()

    # 2. the large shape
    N, B, F = 2000, 1000, 25_000
    t, y, s2, f_min, f_max = wl.make_series(N, 7)
    Y = y + np.random.default_rng(1).normal(0, 0.3, (B, N))
    ser = ctx.upload_series(t, y, s2)
    freq = np.geomspace(1 / (t[-1] - t[0]), 0.5 / np.min(np.diff(t)), F)
    res["large"] = measure(ctx, ser, t, s2, Y, freq, 1, max(3, args.reps // 2), 2)
    report("large", res["large"])
    ser.free()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
