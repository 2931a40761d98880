#!/usr/bin/env python
"""lowrankfilter with a lag on one GPU.  Prints ONE JSON line.

    python tools/bench_lag.py [--rows 1000000] [--lags 1 2 4 16] [--c5-lags 2 3] [--compare-tree DIR --c5-reps 2]

1. Per-pass time of the one-pass kernel (fused.cu) on a Hankel matrix of --rows rows x 256 at each lag of --lags:
   lowrankfilter(y, 256; lag) with TLSQ_FUSED=1 on a 6-sinusoid signal of (rows - 1) lag + 256 samples (rank estimate
   about 12).  Two solves with a fixed iteration count (tol = 0), a and b iterations; the `fused` phase (CUDA events) of
   the second minus that of the first, over the difference in passes, is the time of one pass.
2. A C5-sized signal (bench.py's c5_signal: 50 000 000 samples, three sinusoids, 10 % of the samples shifted by +100)
   filtered with lowrankfilter(y, 256; lag) for every lag of --c5-lags on the default route: wall time of two solves
   (the second with the per-phase timing on), ALM iterations, normalised MSE against the clean signal, the phases that
   ran (the route) and the peak device memory.
3. --compare-tree DIR: `bench.py --workload c5` (lag 1) alternated between DIR (another built checkout) and this tree,
   --c5-reps times each, first, in processes of their own; the parity digests and rates of every run.
The card's name, power limit and maximum SM clock are read in the same run.
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
N_EMB = 256


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                              "-i", "0"], capture_output=True, text=True, timeout=60).stdout.strip()
        name, power, clk = [v.strip() for v in out.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as e:                                    # the numbers below are then unattributed: say so
        return {"name": None, "power_limit": None, "error": repr(e)}


def per_pass(T, torch, rows, lags, a, b):
    out = []
    os.environ["TLSQ_FUSED"] = "1"
    for lag in lags:
        Ns = (rows - 1) * lag + N_EMB
        _, y = T.synth.sinusoids_np(Ns, 6, seed=5)
        yd = torch.from_numpy(y).cuda()
        del y
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            T.lowrankfilter(yd, N_EMB, lag=lag, iters=3, tol=0.0)            # warm-up: module load, every shape
        res = {}
        for its in (a, b):
            T.set_profiling(True)
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                _, info = T.lowrankfilter(yd, N_EMB, lag=lag, iters=its, tol=0.0, return_info=True)
            torch.cuda.synchronize()
            res[its] = (T.get_profile(), info)
            T.set_profiling(False)
        (pa, _), (pb, ib) = res[a], res[b]
        dms, dn = pb["fused"][0] - pa["fused"][0], pb["fused"][1] - pa["fused"][1]
        out.append({"lag": lag, "rows": rows, "samples": Ns, "ranks": [int(v) for v in ib["hist"][a:b, 1]],
                    "passes": dn, "ms_per_pass": dms / dn if dn else None, "handover": pb["epilogue"][1] > 0})
        del yd
    del os.environ["TLSQ_FUSED"]
    return out


def c5_lag(T, torch, lag, Ns=50_000_000, reps=2):
    from bench import c5_signal
    dev = torch.device("cuda", 0)
    y0, yn = c5_signal(Ns, dev, 5)
    runs = []
    for rep in range(reps):
        prof_on = rep == reps - 1
        T.set_profiling(prof_on)
        torch.cuda.reset_peak_memory_stats()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        yf, info = T.lowrankfilter(yn, N_EMB, lag=lag, return_info=True)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        mse = (torch.mean((yf - y0) ** 2) / torch.mean(y0 ** 2)).item()
        r = {"seconds": dt, "profiling": prof_on, "iters": int(info["iters"]), "converged": bool(info["converged"]),
             "sv": int(info["sv"]), "normalised_mse_out": mse, "peak_torch_GB": torch.cuda.max_memory_allocated() / 1e9}
        if prof_on:
            r["phase_ms_spans"] = {k: [round(v[0], 2), v[1]] for k, v in T.get_profile().items() if v[1]}
            T.set_profiling(False)
        runs.append(r)
        del yf
    K = (Ns - N_EMB) // lag + 1
    del y0, yn
    return {"Ns": Ns, "n": N_EMB, "lag": lag, "K": K, "S_GB": K * N_EMB * 8 / 1e9, "runs": runs}


def bench_c5(tree, steps, warmup):
    tree = os.path.abspath(tree)
    out = subprocess.run([sys.executable, os.path.join(tree, "bench.py"), "--workload", "c5", "--gpus", "1", "--no-cpu",
                          "--steps", str(steps), "--warmup", str(warmup)], capture_output=True, text=True, cwd=tree,
                         timeout=3000)
    line = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    if out.returncode != 0 or not line:
        return {"tree": tree, "error": out.stderr[-1500:]}
    r = json.loads(line[-1])
    return {"tree": tree, "value": r["value"], "ms_per_step": r["ms_per_step"], "iters_per_step": r["iters_per_step"],
            "parity": r["parity"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=1_000_000)
    ap.add_argument("--lags", type=int, nargs="*", default=[1, 2, 4, 16])
    ap.add_argument("--iters", type=int, nargs=2, default=[6, 12], metavar=("A", "B"))
    ap.add_argument("--c5-lags", type=int, nargs="*", default=[2, 3])
    ap.add_argument("--compare-tree")
    ap.add_argument("--c5-reps", type=int, default=2)
    ap.add_argument("--c5-steps", type=int, default=2)
    args = ap.parse_args()
    res = {"card": card()}
    if args.compare_tree:                  # first, in processes of their own: nothing else holds device memory
        seq = []
        for _ in range(args.c5_reps):
            seq.append(bench_c5(args.compare_tree, args.c5_steps, 1))
            seq.append(bench_c5(ROOT, args.c5_steps, 1))
        res["bench_c5_alternated"] = seq
    import torch
    import tlsq_b200 as T
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device")
    if args.lags:
        res["per_pass"] = per_pass(T, torch, args.rows, args.lags, *args.iters)
    res["c5_lag"] = [c5_lag(T, torch, lag) for lag in args.c5_lags]
    res["card_after"] = card()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
