"""Cost of the posterior draws K7 (csrc/postdraw.cuh, pioran_celerite_posterior_draws), and of the posterior variance
(pioran_celerite_predict_var) on the same sets beside it.

  1. B = 256, N = M = 1 000: SingleBendingPowerLaw + SHO J = 20 (rank 40), + DRWCelerite J = 20 (rank 60), and explicit
     coefficients of rank 128 (56 complex + 16 real terms): draws at S = 1, 8, 64, and predict_var;
  2. B = 148 (one set per SM), SHO J = 20, N = M = 1e4, S = 8, and predict_var.
The figure of merit is the marginal cost of one more draw, (t(S = 64) − t(S = 8)) / 56, against t(S = 1), which holds the
two O((N + M)·R²) factorisations.  Host clock around calls that end in a device synchronise (every host entry of the C ABI
does); the median of `--reps` timed calls after `--warmup` untimed ones.  The card name, power limit and max SM clock are
read in the same run and printed with the numbers.  A spot check against the numpy prototype runs on the first set of each
rank.

    python tools/postdraw_bench.py [--out FILE.json]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests", "tools", "proto"))
import pioran_b200 as pb  # noqa: E402
import postdraw_math as dm  # noqa: E402
import workloads as wl  # noqa: E402
from postvar_bench import approx_coefs, card, explicit_coefs, timed  # noqa: E402


def measure(ctx, ser, co, tau, Ss, warmup, reps):
    a, b, c, d = co
    B, NG = a.shape[0], ser.N + len(tau)
    row = {}
    for S in Ss:
        q = np.random.default_rng(S).standard_normal((B, S, NG))
        row[f"draws_S{S}_s"] = timed(lambda: ctx.celerite_posterior_draws(ser, a, b, c, d, tau, q), warmup, reps)
    row["kernel"] = ctx.last_kernel_name()
    row["predict_var_s"] = timed(lambda: ctx.celerite_predict_var(ser, a, b, c, d, tau, return_mean=False), warmup, reps)
    if 8 in Ss and 64 in Ss:
        row["marginal_draw_s"] = (row["draws_S64_s"] - row["draws_S8_s"]) / 56
        row["marginal_over_S1"] = row["marginal_draw_s"] / row["draws_S1_s"]
    return row


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
        q = np.random.default_rng(9).standard_normal((1, 2, N + N))
        got = ctx.celerite_posterior_draws(ser, a[:1], b[:1], c[:1], d[:1], tau, q, sigma2_tau=1e-10)[0]
        want = dm.posterior_draws(a[0], b[0], c[0], d[0], t, y, s2, tau, q[0], 0.0, 1e-10)
        err = float(np.max(np.abs(got - want)) / np.sqrt(np.sum(a[0])))
        row = {"case": name, "B": B, "N": N, "M": N, "check_vs_proto": err,
               **measure(ctx, ser, co, tau, (1, 8, 64), args.warmup, args.reps)}
        res["rank"].append(row)
        print(f"{name}, B={B}, N=M={N} [{row['kernel']}]: draws S=1 {row['draws_S1_s'] * 1e3:.3f} ms, S=8 "
              f"{row['draws_S8_s'] * 1e3:.3f} ms, S=64 {row['draws_S64_s'] * 1e3:.3f} ms; one more draw "
              f"{row['marginal_draw_s'] * 1e3:.4f} ms ({row['marginal_over_S1']:.3f} of S=1); predict_var "
              f"{row['predict_var_s'] * 1e3:.3f} ms; vs prototype {err:.1e} of sqrt(sum(a))", flush=True)
    ser.free()

    B, N = 148, 10_000
    t, y, s2, f_min, f_max = wl.make_series_fast(N, 11)
    tau = np.sort(np.random.default_rng(2).uniform(t[0] - 5, t[-1] + 5, N))
    ser = ctx.upload_series(t, y, s2)
    co = approx_coefs(ctx, "SHO", B, f_min, f_max, y, 6)
    row = {"case": "SHO J=20", "B": B, "N": N, "M": N, **measure(ctx, ser, co, tau, (8,), 1, max(3, args.reps // 2))}
    res["length"].append(row)
    print(f"SHO J=20, B={B}, N=M={N} [{row['kernel']}]: draws S=8 {row['draws_S8_s'] * 1e3:.3f} ms; predict_var "
          f"{row['predict_var_s'] * 1e3:.3f} ms", flush=True)
    ser.free()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
