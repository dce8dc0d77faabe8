"""Throughput of the K5g paths (csrc/jvp.cuh): the gradient with one QPO feature (SingleBendingPowerLaw + SHO, J = 20, N = 1 000)
against the value of the same batch, and the explicit-coefficient JVP with P = 12 directions at ranks 16 … 96 (B = 64, N = 1 000).
Host clock around calls that end in a device synchronise (every host entry of the C ABI does); the median of `--reps` timed calls
after `--warmup` untimed ones.  The working set (series, coefficients, tangents) is well inside the 126 MB L2.
The card name and power limit are read in the same run and printed with the numbers.

    python tools/jvp_bench.py [--out FILE.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import pioran_b200 as pb  # noqa: E402
import workloads as wl  # noqa: E402


def timed(fn, warmup, reps):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts))


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    ctx = pb.get_context(0)
    res = {"card": card(), "features": [], "jvp": []}
    N = 1000
    t, y, s2, f_min, f_max = wl.make_series(N, 7, (0.82, 0.01, 3.3), 1.0, 20)
    rng = np.random.default_rng(3)
    like = pb.BatchedLikelihood(t, y, s2, "SingleBendingPowerLaw", 20, "SHO", f_min=f_min, f_max=f_max, ctx=ctx, n_features=1)
    for B in (16, 1024):
        th = wl.prior_theta(B, f_min, f_max, y.mean(), y.std(), 5)
        qpo = np.column_stack([rng.uniform(0.5, 3, B), np.exp(rng.uniform(np.log(2 * f_min), np.log(f_max / 2), B)),
                               rng.uniform(1.0, 15, B)])
        th = np.column_stack([th, qpo])
        tg = timed(lambda: like.value_and_gradient(th), args.warmup, args.reps)
        tv = timed(lambda: like(th), args.warmup, args.reps)
        row = {"B": B, "grad_s": tg, "value_s": tv, "gradients_per_s": B / tg, "grad_over_value": tg / tv}
        res["features"].append(row)
        print(f"features SBPL+SHO J=20 + 1 QPO, N={N}, B={B}: gradient {tg * 1e3:.3f} ms ({B / tg:,.0f}/s), "
              f"value {tv * 1e3:.3f} ms, ratio {tg / tv:.2f}", flush=True)
    like.close()
    ser = ctx.upload_series(t, y, s2)
    B, P = 64, 12
    for R in (16, 42, 64, 96):
        Jt = R // 2
        a = rng.uniform(0.1, 1.0, (B, Jt)) / Jt
        c = np.exp(rng.uniform(np.log(0.05), np.log(5.0), (B, Jt)))
        tan = {n: rng.normal(size=(B, P, Jt)) for n in ("da", "db", "dc", "dd")}
        tj = timed(lambda: ctx.celerite_logl_jvp(ser, a, a, c, c, **tan), args.warmup, args.reps)
        tv = timed(lambda: ctx.celerite_logl(ser, a, a, c, c), args.warmup, args.reps)
        row = {"R": R, "B": B, "P": P, "N": N, "jvp_s": tj, "value_s": tv, "directional_derivatives_per_s": B * P / tj}
        res["jvp"].append(row)
        print(f"jvp R={R} B={B} P={P} N={N}: {tj * 1e3:.3f} ms ({B * P / tj:,.0f} directional derivatives/s), "
              f"value {tv * 1e3:.3f} ms", flush=True)
    ser.free()
    print("card:", res["card"])
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
