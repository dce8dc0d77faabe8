"""Cost of the K5r reverse-mode gradient (csrc/vjp.cuh) against the value and against the same gradient in forward mode (K5g).

  1. explicit coefficients, N = 1 000, B = 64, ranks 16 / 42 / 64 / 96: K5r with and without the data gradients, the value
     (pioran_celerite_logl) on the same batch, and K5g with P = 4·Jt + 2 unit directions (the same full gradient);
  2. the DESIGN table workload with features, SingleBendingPowerLaw + SHO J = 20 + 1 QPO, N = 1 000, B = 16 and 1 024: forward
     and reverse gradients and the value;
  3. CARMA(5, 2) with the log shift, N = 1 000, B = 256: gradient rate against value rate.
Host clock around calls that end in a device synchronise (every host entry of the C ABI does); the median of `--reps` timed calls
after `--warmup` untimed ones.  The card name and power limit are read in the same run and printed with the numbers.

    python tools/vjp_bench.py [--out FILE.json]
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
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    ctx = pb.get_context(0)
    res = {"card": card(), "explicit": [], "features": [], "carma": []}
    print("card:", res["card"], flush=True)
    N = 1000
    t, y, s2, f_min, f_max = wl.make_series(N, 7, (0.82, 0.01, 3.3), 1.0, 20)
    rng = np.random.default_rng(3)

    ser = ctx.upload_series(t, y, s2)
    B = 64
    for R in (16, 42, 64, 96):
        Jt = R // 2
        a = rng.uniform(0.1, 1.0, (B, Jt)) / Jt
        c = np.exp(rng.uniform(np.log(0.05), np.log(5.0), (B, Jt)))
        P = 4 * Jt + 2
        tan = {k: np.zeros((B, P, Jt)) for k in ("da", "db", "dc", "dd")}
        for q, k in enumerate(("da", "db", "dc", "dd")):
            tan[k][:, q * Jt:(q + 1) * Jt, :] = np.eye(Jt)[None]
        dmu, dnu = np.zeros((B, P)), np.zeros((B, P))
        dmu[:, 4 * Jt], dnu[:, 4 * Jt + 1] = 1.0, 1.0
        tr = timed(lambda: ctx.celerite_logl_vjp(ser, a, a, c, c), args.warmup, args.reps)
        trd = timed(lambda: ctx.celerite_logl_vjp(ser, a, a, c, c, data_grad=True), args.warmup, args.reps)
        tv = timed(lambda: ctx.celerite_logl(ser, a, a, c, c), args.warmup, args.reps)
        tf = timed(lambda: ctx.celerite_logl_jvp(ser, a, a, c, c, dmu=dmu, dnu=dnu, **tan), 1, max(2, args.reps // 4))
        row = {"R": R, "B": B, "N": N, "P_forward": P, "vjp_s": tr, "vjp_data_s": trd, "value_s": tv, "jvp_full_s": tf,
               "vjp_over_value": tr / tv, "jvp_over_vjp": tf / tr}
        res["explicit"].append(row)
        print(f"explicit R={R} B={B} N={N}: vjp {tr * 1e3:.3f} ms, vjp+data {trd * 1e3:.3f} ms, value {tv * 1e3:.3f} ms "
              f"(vjp/value {tr / tv:.2f}), jvp P={P} {tf * 1e3:.3f} ms (jvp/vjp {tf / tr:.1f})", flush=True)
    ser.free()

    kw = dict(f_min=f_min, f_max=f_max, ctx=ctx, n_features=1)
    fwd = pb.BatchedLikelihood(t, y, s2, "SingleBendingPowerLaw", 20, "SHO", **kw)
    rev = pb.BatchedLikelihood(t, y, s2, "SingleBendingPowerLaw", 20, "SHO", gradient="reverse", **kw)
    for B in (16, 1024):
        th = wl.prior_theta(B, f_min, f_max, y.mean(), y.std(), 5)
        qpo = np.column_stack([rng.uniform(0.5, 3, B), np.exp(rng.uniform(np.log(2 * f_min), np.log(f_max / 2), B)),
                               rng.uniform(1.0, 15, B)])
        th = np.column_stack([th, qpo])
        gf, gr = fwd.value_and_gradient(th)[1], rev.value_and_gradient(th)[1]
        scale = np.maximum(np.abs(gf), np.abs(gf).max(axis=0, keepdims=True))
        diff = float(np.max(np.abs(gr - gf) / np.where(scale > 0, scale, 1.0)))
        tf = timed(lambda: fwd.value_and_gradient(th), args.warmup, args.reps)
        tr = timed(lambda: rev.value_and_gradient(th), args.warmup, args.reps)
        tv = timed(lambda: fwd(th), args.warmup, args.reps)
        row = {"B": B, "N": N, "forward_s": tf, "reverse_s": tr, "value_s": tv, "forward_over_reverse": tf / tr,
               "reverse_over_value": tr / tv, "max_rel_diff": diff}
        res["features"].append(row)
        print(f"features SBPL+SHO J=20 + 1 QPO, N={N}, B={B}: forward {tf * 1e3:.3f} ms, reverse {tr * 1e3:.3f} ms "
              f"(speed-up {tf / tr:.2f}), value {tv * 1e3:.3f} ms (reverse/value {tr / tv:.2f}), max rel diff {diff:.1e}", flush=True)
    fwd.close(); rev.close()

    yp = np.exp(0.3 * (y - y.mean()) / y.std()) + 1.0
    like = pb.BatchedCARMALikelihood(t, yp, (0.05 * yp) ** 2, 5, 2, f_min, f_max, log_shift=True, ctx=ctx)
    B = 256
    th = np.concatenate([rng.uniform(0.4, 1.8, (B, 5)), rng.uniform(0.4, 1.8, (B, 2)),
                         rng.uniform(0.5, 2.0, (B, 1)), rng.uniform(0.8, 1.3, (B, 1)), rng.normal(0, 0.2, (B, 1)),
                         rng.uniform(0.0, 0.8 * yp.min(), (B, 1))], axis=1)
    ok = int(np.isfinite(like(th)).sum())
    tg = timed(lambda: like.value_and_gradient(th), args.warmup, args.reps)
    tv = timed(lambda: like(th), args.warmup, args.reps)
    res["carma"].append({"p": 5, "q": 2, "B": B, "N": N, "rows_in_bounds": ok, "grad_s": tg, "value_s": tv,
                         "gradients_per_s": B / tg, "values_per_s": B / tv})
    print(f"CARMA(5,2) log shift, N={N}, B={B} ({ok} in bounds): gradient {tg * 1e3:.3f} ms ({B / tg:,.0f}/s), "
          f"value {tv * 1e3:.3f} ms ({B / tv:,.0f}/s)", flush=True)
    like.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
