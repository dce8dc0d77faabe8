"""Cost of the posterior covariance K8 (csrc/postcov.cuh, pioran_celerite_predict_cov), against the posterior variance
(pioran_celerite_predict_var) on the same sets and against a one-set dense solve on the CPU (scipy: the Cholesky factor of
K̃, then K_ττ − K_τt K̃⁻¹ K_tτ, the route of the reference's predict_cov).

  1. B = 64, N = M = 1 000: SingleBendingPowerLaw + SHO J = 20 (rank 40), + DRWCelerite J = 20 (rank 60), and explicit
     coefficients of rank 128 (56 complex + 16 real terms);
  2. B = 16, SHO J = 20, N = M = 1e4 (12.8 GB of output: θ-chunks of one set each under the 1 GiB cap).
Host clock around calls that end in a device synchronise (every host entry of the C ABI does), so a predict_cov time includes
the copy of the B·M² output into host memory; the device time of the same call (CUDA events around its launches and copies)
is printed beside it, and one more call runs under the CUDA activity trace of torch.profiler, which splits the device time
into the kernels (by name, in the JSON) and the copies.  The median of `--reps` timed calls after `--warmup` untimed ones.  The card name, power limit and max SM
clock are read in the same run and printed with the numbers.  A spot check against the dense FP64 covariance runs on the first
set of each rank.

    python tools/postcov_bench.py [--out FILE.json]
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
sys.path.insert(0, os.path.join(ROOT, "tests", "tools", "proto"))
import pioran_b200 as pb  # noqa: E402
import postcov_math as cm  # noqa: E402
import workloads as wl  # noqa: E402
from postvar_bench import approx_coefs, card, explicit_coefs, timed  # noqa: E402


def measure(ctx, ser, co, tau, warmup, reps):
    a, b, c, d = co
    row = {}
    ms = []

    def call():
        ctx.celerite_predict_cov(ser, a, b, c, d, tau, return_mean=False)
        ms.append(ctx.last_kernel_ms())
    row["predict_cov_s"] = timed(call, warmup, reps)
    row["predict_cov_device_s"] = float(np.median(ms[warmup:])) * 1e-3
    row["kernel"] = ctx.last_kernel_name()
    row["trace_ms"] = trace(call)
    row["predict_var_s"] = timed(lambda: ctx.celerite_predict_var(ser, a, b, c, d, tau, return_mean=False), warmup, reps)
    return row


def trace(fn):
    """Device time of one call by what ran: the CUDA activity trace of torch.profiler (CUPTI), summed per kernel name and
    for the copies.  Returns {name: [ms, count]}, or {"error": text} when the trace is not available."""
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.init()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        return {e.key: [e.self_device_time_total * 1e-3, e.count] for e in prof.key_averages() if e.self_device_time_total > 0}
    except Exception as e:  # noqa: BLE001
        return {"error": repr(e)}


def split(tr):
    """(kernels, copies) in ms from a trace."""
    if "error" in tr:
        return float("nan"), float("nan")
    cp = sum(v[0] for k, v in tr.items() if k.startswith(("Memcpy", "Memset")))
    return sum(v[0] for v in tr.values()) - cp, cp


def dense_one_set(co, t, s2, tau, reps=3):
    a, b, c, d = (x[0] for x in co)
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        cm.dense_cov(a, b, c, d, t, s2, tau)
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    ctx = pb.get_context(0)
    res = {"card": card(), "rank": [], "length": []}
    print("card (name, power limit, max SM clock):", res["card"], flush=True)

    N = 1000
    t, y, s2, f_min, f_max = wl.make_series(N, 7)
    tau = np.sort(np.random.default_rng(1).uniform(t[0] - 5, t[-1] + 5, N))
    ser = ctx.upload_series(t, y, s2)
    B = 64
    cases = [("SHO J=20", approx_coefs(ctx, "SHO", B, f_min, f_max, y, 3)),
             ("DRWCelerite J=20", approx_coefs(ctx, "DRWCelerite", B, f_min, f_max, y, 4)),
             ("explicit rank 128", explicit_coefs(B, 56, 16, 5))]
    for name, co in cases:
        a, b, c, d = co
        got = ctx.celerite_predict_cov(ser, a[:1], b[:1], c[:1], d[:1], tau, return_mean=False)[0]
        err = float(np.max(np.abs(got - cm.dense_cov(a[0], b[0], c[0], d[0], t, s2, tau))) / np.sum(a[0]))
        row = {"case": name, "B": B, "N": N, "M": N, "check_vs_dense": err, **measure(ctx, ser, co, tau, args.warmup, args.reps),
               "dense_cpu_one_set_s": dense_one_set(co, t, s2, tau)}
        res["rank"].append(row)
        print(f"{name}, B={B}, N=M={N} [{row['kernel']}]: predict_cov {row['predict_cov_s'] * 1e3:.3f} ms "
              f"(device {row['predict_cov_device_s'] * 1e3:.3f} ms: kernels {split(row['trace_ms'])[0]:.3f} ms, "
              f"copies {split(row['trace_ms'])[1]:.3f} ms); "
              f"predict_var {row['predict_var_s'] * 1e3:.3f} ms; dense CPU, one set {row['dense_cpu_one_set_s'] * 1e3:.1f} ms; vs dense {err:.1e} of sum(a)", flush=True)
    ser.free()

    B, N = 16, 10_000
    t, y, s2, f_min, f_max = wl.make_series_fast(N, 11)
    tau = np.sort(np.random.default_rng(2).uniform(t[0] - 5, t[-1] + 5, N))
    ser = ctx.upload_series(t, y, s2)
    co = approx_coefs(ctx, "SHO", B, f_min, f_max, y, 6)
    row = {"case": "SHO J=20", "B": B, "N": N, "M": N, **measure(ctx, ser, co, tau, 1, 2)}
    res["length"].append(row)
    print(f"SHO J=20, B={B}, N=M={N} [{row['kernel']}]: predict_cov {row['predict_cov_s'] * 1e3:.3f} ms "
          f"(device {row['predict_cov_device_s'] * 1e3:.3f} ms: kernels {split(row['trace_ms'])[0]:.3f} ms, "
          f"copies {split(row['trace_ms'])[1]:.3f} ms); predict_var {row['predict_var_s'] * 1e3:.3f} ms", flush=True)
    ser.free()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
