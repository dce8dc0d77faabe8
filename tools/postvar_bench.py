"""Cost of the posterior variance K6 (csrc/postvar.cuh, pioran_celerite_predict_var) against the posterior mean alone
(pioran_celerite_predict) on the same batch.

  1. B = 256, N = M = 1 000: SingleBendingPowerLaw + SHO J = 20 (rank 40), + DRWCelerite J = 20 (rank 60), and explicit
     coefficients of rank 128 (56 complex + 16 real terms): predict, predict_var with the mean, predict_var without it;
  2. B = 148 (one set per SM), SHO J = 20, N = M = 1e3, 1e4, 1e5: the same three calls, to show the cost grows linearly in
     N + M (an O(N·M) method would grow 100× per decade).
Host clock around calls that end in a device synchronise (every host entry of the C ABI does); the median of `--reps` timed calls
after `--warmup` untimed ones.  The card name, power limit and max SM clock are read in the same run and printed with the
numbers.  A spot check of var against a dense Cholesky solve runs on the first workload.

    python tools/postvar_bench.py [--out FILE.json]
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
sys.path.insert(0, os.path.join(ROOT, "tests", "tools", "proto"))
import pioran_b200 as pb  # noqa: E402
import postvar_math as pm  # noqa: E402
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


def approx_coefs(ctx, basis, B, f_min, f_max, y, seed):
    spec = pb.make_spec("SingleBendingPowerLaw", f_min, f_max, 20, basis_function=basis)
    th = wl.prior_theta(B, f_min, f_max, y.mean(), y.std(), seed)[:, :4]
    return ctx.approx_coeffs(spec, th)


def explicit_coefs(B, n_complex, n_real, seed):
    rng = np.random.default_rng(seed)
    Jt = n_complex + n_real
    a = rng.uniform(0.2, 1.0, (B, Jt)) / Jt
    b = rng.uniform(-0.1, 0.1, (B, Jt)) / Jt
    c = np.exp(rng.uniform(np.log(0.01), np.log(2.0), (B, Jt)))
    d = c * rng.uniform(0.0, 1.5, (B, Jt))
    b[:, n_complex:] = 0.0
    d[:, n_complex:] = 0.0
    return a, b, c, d


def measure(ctx, ser, co, tau, warmup, reps):
    a, b, c, d = co
    tp = timed(lambda: ctx.celerite_predict(ser, a, b, c, d, tau), warmup, reps)
    tmv = timed(lambda: ctx.celerite_predict_var(ser, a, b, c, d, tau), warmup, reps)
    tv = timed(lambda: ctx.celerite_predict_var(ser, a, b, c, d, tau, return_mean=False), warmup, reps)
    return {"predict_s": tp, "predict_var_s": tmv, "var_only_s": tv, "kernel": ctx.last_kernel_name(),
            "ratio": tmv / tp}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    ctx = pb.get_context(0)
    res = {"card": card(), "rank": [], "length": []}
    print("card (name, power limit, max SM clock):", res["card"], flush=True)

    N = 1000
    t, y, s2, f_min, f_max = wl.make_series(N, 7)
    tau = np.sort(np.random.default_rng(1).uniform(t[0] - 5, t[-1] + 5, N))
    ser = ctx.upload_series(t, y, s2)
    B = 256
    cases = [("SHO J=20", approx_coefs(ctx, "SHO", B, f_min, f_max, y, 3)),
             ("DRWCelerite J=20", approx_coefs(ctx, "DRWCelerite", B, f_min, f_max, y, 4)),
             ("explicit rank 128", explicit_coefs(B, 56, 16, 5))]
    for name, co in cases:
        a, b, c, d = co
        var = ctx.celerite_predict_var(ser, a[:2], b[:2], c[:2], d[:2], tau, return_mean=False)
        want = pm.predict_var(a[0], b[0], c[0], d[0], t, s2, tau[::10])
        err = float(np.max(np.abs(var[0][::10] - want)) / np.sum(a[0]))
        row = {"case": name, "B": B, "N": N, "M": N, "check_vs_proto": err, **measure(ctx, ser, co, tau, args.warmup, args.reps)}
        res["rank"].append(row)
        print(f"{name}, B={B}, N=M={N} [{row['kernel']}]: predict {row['predict_s'] * 1e3:.3f} ms, predict_var "
              f"{row['predict_var_s'] * 1e3:.3f} ms ({row['ratio']:.2f}x), var only {row['var_only_s'] * 1e3:.3f} ms; "
              f"var vs prototype {err:.1e} of sum(a)", flush=True)
    ser.free()

    B = 148
    for N in (1000, 10_000, 100_000):
        t, y, s2, f_min, f_max = wl.make_series_fast(N, 11)
        tau = np.sort(np.random.default_rng(2).uniform(t[0] - 5, t[-1] + 5, N))
        ser = ctx.upload_series(t, y, s2)
        co = approx_coefs(ctx, "SHO", B, f_min, f_max, y, 6)
        reps = args.reps if N < 100_000 else max(3, args.reps // 2)
        row = {"case": "SHO J=20", "B": B, "N": N, "M": N, **measure(ctx, ser, co, tau, 1, reps)}
        res["length"].append(row)
        print(f"SHO J=20, B={B}, N=M={N} [{row['kernel']}]: predict {row['predict_s'] * 1e3:.3f} ms, predict_var "
              f"{row['predict_var_s'] * 1e3:.3f} ms ({row['ratio']:.2f}x), var only {row['var_only_s'] * 1e3:.3f} ms", flush=True)
        ser.free()
    L = res["length"]
    for k in range(1, len(L)):
        print(f"N {L[k - 1]['N']} -> {L[k]['N']}: predict_var x{L[k]['predict_var_s'] / L[k - 1]['predict_var_s']:.1f}, "
              f"var only x{L[k]['var_only_s'] / L[k - 1]['var_only_s']:.1f}", flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
