"""Grassmann-average iteration rates for the three averages of rpca_ga (mu_mean, entrywise_trimmed_mean,
entrywise_median) on shapes whose X exceeds the 126 MB L2, plus the two sides of the 16 384-observation boundary
where rpca_ga switches from the per-row sort to the per-row selection kernels.

    python tools/bench_ga_robust.py [--out results.json]

Per-iteration time = (t(K2 iterations) - t(K1 iterations)) / (K2 - K1) of whole rpca_ga(X, 1) solves on CUDA tensors
with tol = 0 (so every solve runs exactly its iteration count); the difference removes the copy of X, the column norms
and the once-per-component trimmed-mean selection.  Bytes per iteration count the reads of X only (d N 8 per pass):
  mu_mean          1 pass  (the fused average + next dot products sweep)
  trimmed mean     2 passes (the kept-range sweep, then the dot products sweep)
  median          10 passes (8 radix passes, the tie pass, the dot products sweep)
The per-column vectors (norms, signs) add 16 bytes per column and pass on top, which matters at small d.
The building-block column times the selection kernels alone (10 passes of X for either average: 8 radix passes and the
tie pass, plus the kept-range sweep for the trimmed mean or the sign lookup for the median).
"""
import argparse
import json
import os
import subprocess
import sys
import time
import warnings

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import tlsq_b200 as T  # noqa: E402

PASSES = {"mu_mean": 1, "entrywise_trimmed_mean": 2, "entrywise_median": 10}
MUS = {"mu_mean": T.mu_mean, "entrywise_trimmed_mean": T.entrywise_trimmed_mean,
       "entrywise_median": T.entrywise_median}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def solve_time(X, q0, mu, iters):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        T.rpca_ga(X, 1, mu=mu, q0=q0, tol=0.0, iters=iters)
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def per_iteration(X, q0, mu, k1, k2, reps=3):
    solve_time(X, q0, mu, k1)                                             # warm-up of this shape
    best = []
    for _ in range(reps):
        a = solve_time(X, q0, mu, k1)
        b = solve_time(X, q0, mu, k2)
        best.append((b - a) / (k2 - k1))
    best.sort()
    return best[len(best) // 2], best


def make(d, N, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    X = torch.randn((N, d), dtype=torch.float64, device="cuda", generator=g).t()            # column-major d x N
    X += 1000.0 * torch.randn((N, d), dtype=torch.float64, device="cuda", generator=g).t() * \
        (torch.rand((N, d), dtype=torch.float64, device="cuda", generator=g).t() < 0.01)
    q0 = torch.randn((1, d), dtype=torch.float64, device="cuda", generator=g).t()
    return X, q0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_ga_robust: needs a CUDA device (no CPU fallback)")
    res = {"card": card(), "rows": []}
    print(f"card: {res['card']}", flush=True)
    for d, N, k1, k2 in [(256, 1_000_000, 3, 13), (8, 4_000_000, 3, 13)]:
        X, q0 = make(d, N, seed=d)
        for name, mu in MUS.items():
            t, all_t = per_iteration(X, q0, mu, k1, k2)
            byts = PASSES[name] * d * N * 8
            row = {"d": d, "N": N, "mu": name, "it_per_s": 1.0 / t, "ms_per_it": 1e3 * t, "passes": PASSES[name],
                   "bytes_per_it": byts, "TB_per_s": byts / t / 1e12, "spread_ms": [1e3 * v for v in all_t]}
            if name != "mu_mean":
                # the selection kernels alone (building block): median = 8 radix passes + tie pass; trimmed mean =
                # 8 radix passes + tie pass (its once-per-component part) + the kept-range sweep
                w = torch.ones(N, dtype=torch.float64, device="cuda")
                T.robust_average(X, w, mu)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(5):
                    T.robust_average(X, w, mu)
                torch.cuda.synchronize()
                tb = (time.perf_counter() - t0) / 5
                row["building_block_ms"] = 1e3 * tb
                row["building_block_TB_per_s"] = 10 * d * N * 8 / tb / 1e12
            res["rows"].append(row)
            extra = (f"  | building block {row['building_block_ms']:7.3f} ms = "
                     f"{row['building_block_TB_per_s']:5.2f} TB/s over 10 passes" if "building_block_ms" in row else "")
            print(f"d={d:4d} N={N:8d} {name:24s} {row['it_per_s']:9.1f} it/s  {row['ms_per_it']:8.3f} ms/it  "
                  f"{PASSES[name]:2d} passes  {byts / 1e9:6.2f} GB/it  {row['TB_per_s']:5.2f} TB/s{extra}", flush=True)
        del X, q0
        torch.cuda.empty_cache()
    # the boundary: per-row sort (N = 16 384) and per-row selection (N = 16 385), through rpca_ga and the building block
    for d in (256,):
        for N in (16_384, 16_385):
            X, q0 = make(d, N, seed=N)
            for name in ("entrywise_trimmed_mean", "entrywise_median"):
                t, _ = per_iteration(X, q0, MUS[name], 3, 23)
                w = torch.ones(N, dtype=torch.float64, device="cuda")
                T.robust_average(X, w, MUS[name])
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(20):
                    T.robust_average(X, w, MUS[name])
                torch.cuda.synchronize()
                tb = (time.perf_counter() - t0) / 20
                row = {"d": d, "N": N, "mu": name, "rpca_ga_ms_per_it": 1e3 * t,
                       "rpca_ga_path": "sort" if N <= 16_384 else "select", "building_block_ms": 1e3 * tb}
                res["rows"].append(row)
                print(f"d={d:4d} N={N:8d} {name:24s} rpca_ga ({row['rpca_ga_path']:6s}) {1e3 * t:8.3f} ms/it   "
                      f"building block (select) {1e3 * tb:8.3f} ms", flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
