"""Cost of the sinusoidal-mean likelihood (pioran_approx_logl_sine) and its gradient (pioran_approx_logl_sine_grad), the model of
the reference's periodicity run (examples/ultranest/single_pl_periodicity.jl): SingleBendingPowerLaw + SHO J = 20 red noise plus
m(t) = μ + A·sin(2πt/T₀ + ϕ).

Value, at B ∈ {400, 4 096, 65 536} on the golden series of that run (N = 485) and on the synthetic N = 1 000 series of bench.py:
  - the fused entry: y − A·sin(…) formed on the device in front of K1 + K2;
  - the route without it: the rows y − m_θ(t) built on the host with numpy (timed on its own), then pioran_approx_coeffs and
    pioran_celerite_logl with y_batch (μ folded into the rows; the upload of the rows is part of that call).
Gradient, at B = 4 096 on both series: gradients per second of pioran_approx_logl_sine_grad against pioran_approx_logl_grad at the
same shape; the difference is the cost of the mean warp and of the per-θ data row.
Host clock around calls that end in a device synchronise; the median of `--reps` timed calls after `--warmup` untimed ones.
The parameter vectors are the golden chain's rows (repeated to B) on the golden series and prior draws on the synthetic one.
Each shape also reports the largest relative difference between the two routes' values.  The card name, power limit and max
SM clock are read in the same run.

    python tools/sine_bench.py [--out FILE.json]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import pioran_b200 as pb  # noqa: E402
import workloads as wl  # noqa: E402
from postvar_bench import card, timed  # noqa: E402


def host_rows(t, y, theta):
    """Today's host-side data: y − (μ + A·sin(2πt/T₀ + ϕ)) for every θ and every time."""
    return y[None] - (theta[:, 5:6] + theta[:, 6:7] * np.sin(2 * np.pi * t[None] / theta[:, 8:9] + theta[:, 7:8]))


def theta_rows(name, B, t, y, f_min, f_max):
    if name == "golden":
        chain = np.load(os.path.join(ROOT, "tests", "golden", "simu_periodic_rednoise_chains.npz"))["simu_periodic_rednoise"]
        th = chain[:, 2:11]
        return np.ascontiguousarray(np.resize(th, (B, th.shape[1])))
    rng = np.random.default_rng(B)
    base = wl.prior_theta(B, f_min, f_max, y.mean(), y.std(), 5)
    mean = np.column_stack([rng.uniform(0, 2 * y.std(), B), rng.uniform(0, 2 * np.pi, B),
                            np.exp(rng.uniform(np.log(10 * np.min(np.diff(t))), np.log(t[-1] - t[0]), B))])
    return np.ascontiguousarray(np.column_stack([base, mean]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    ctx = pb.get_context(0)
    res = {"card": card(), "value": {}, "gradient": {}}
    print("card (name, power limit, max SM clock):", res["card"], flush=True)

    ts = np.loadtxt(os.path.join(ROOT, "tests", "golden", "simu_periodic_rednoise_subset_time_series.txt"))
    tg, yg, eg = (np.ascontiguousarray(c) for c in ts.T)
    ts_, ys_, s2s, fmn, fmx = wl.make_series(1000, 0)
    series = {"golden_N485": ("golden", tg, yg, eg ** 2, 1 / (tg[-1] - tg[0]), 0.5 / np.min(np.diff(tg))),
              "synthetic_N1000": ("synthetic", ts_, ys_, s2s, fmn, fmx)}
    for label, (kind, t, y, s2, f_min, f_max) in series.items():
        spec = pb.make_spec("SingleBendingPowerLaw", f_min, f_max, 20)
        ser = ctx.upload_series(t, y, s2)
        for B in (400, 4096, 65536):
            th = theta_rows(kind, B, t, y, f_min, f_max)
            fused = ctx.approx_logl_sine(ser, spec, th)
            fused_s = timed(lambda: ctx.approx_logl_sine(ser, spec, th), args.warmup, args.reps)
            rows_s = timed(lambda: host_rows(t, y, th), 1, max(3, args.reps // 2))
            yb = host_rows(t, y, th)

            def old_route():
                a, b, c, d = ctx.approx_coeffs(spec, th[:, :4])
                return ctx.celerite_logl(ser, a, b, c, d, nu=th[:, 4], y_batch=yb)
            old = old_route()
            old_kernel = ctx.last_kernel_name()
            old_s = timed(old_route, args.warmup, args.reps)
            ok = np.isfinite(fused) & np.isfinite(old)
            diff = float(np.max(np.abs(fused[ok] - old[ok]) / np.maximum(1.0, np.abs(old[ok])))) if ok.any() else float("nan")
            r = {"B": B, "N": len(t), "fused_s": fused_s, "host_rows_s": rows_s, "generic_with_upload_s": old_s,
                 "old_route_total_s": rows_s + old_s, "speedup_vs_old_route": (rows_s + old_s) / fused_s,
                 "rows_bytes": 8 * B * len(t), "generic_kernel": old_kernel, "max_rel_diff_vs_old_route": diff,
                 "nonfinite_rows": int((~np.isfinite(fused)).sum())}
            res["value"][f"{label}_B{B}"] = r
            print(f"value {label} B={B}: fused {fused_s * 1e3:.2f} ms; host rows {rows_s * 1e3:.2f} ms + generic "
                  f"{old_s * 1e3:.2f} ms [{old_kernel}] = {(rows_s + old_s) * 1e3:.2f} ms ({r['speedup_vs_old_route']:.1f}x); "
                  f"max rel diff {diff:.1e}", flush=True)
        B = 4096
        th = theta_rows(kind, B, t, y, f_min, f_max)
        ctx.approx_logl_sine_grad(ser, spec, th)
        sine_kernel = ctx.last_kernel_name()
        sine_s = timed(lambda: ctx.approx_logl_sine_grad(ser, spec, th), args.warmup, args.reps)
        ctx.approx_logl_grad(ser, spec, th[:, :6])
        plain_kernel = ctx.last_kernel_name()
        plain_s = timed(lambda: ctx.approx_logl_grad(ser, spec, th[:, :6]), args.warmup, args.reps)
        r = {"B": B, "N": len(t), "sine_grad_s": sine_s, "sine_gradients_per_s": B / sine_s, "sine_kernel": sine_kernel,
             "plain_grad_s": plain_s, "plain_gradients_per_s": B / plain_s, "plain_kernel": plain_kernel,
             "mean_warp_cost": sine_s / plain_s - 1.0}
        res["gradient"][f"{label}_B{B}"] = r
        print(f"gradient {label} B={B}: sine {B / sine_s:.0f}/s ({sine_s * 1e3:.2f} ms, {sine_kernel}); plain {B / plain_s:.0f}/s "
              f"({plain_s * 1e3:.2f} ms, {plain_kernel}); mean warp +{r['mean_warp_cost']:.1%}", flush=True)
        ser.free()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    t0 = time.perf_counter()
    main()
    print(f"total {time.perf_counter() - t0:.1f} s", flush=True)
