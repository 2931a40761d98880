#!/usr/bin/env python
"""The one-pass kernel (fused.cu) at rank estimates from 6 to 32 on one GPU.  Prints ONE JSON line.

    python tools/bench_fused_rank.py [--rows 1000000] [--c5] [--compare-tree DIR --c5-reps 2]

1. Per-pass time.  lowrankfilter(y, 256) with TLSQ_FUSED=1 on a signal of k sinusoids (synth.sinusoids_np, rank
   estimate about 2k) whose Hankel matrix has --rows rows (2 GB per M x 256 matrix at 10^6 rows: larger than the L2).
   Two solves with a fixed iteration count (tol = 0), a and b iterations; the `fused` phase (CUDA events) of the second
   minus that of the first, over the difference in passes, is the time of one pass at the ranks of iterations a+1..b,
   which are reported with it.
2. --c5: a C5-sized solve (50 000 000 samples, n = 256, implicit Hankel matrix 49 999 745 x 256) of a 12-sinusoid
   signal on the default route (odd row count: one-pass kernel, Y in place): wall time of two solves, ALM iterations,
   rank history and normalised MSE against the clean signal.
3. --compare-tree DIR: `bench.py --workload c5` alternated between this tree and DIR (another built checkout), --c5-reps
   times each; the parity digests and times of every run.
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


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                              "-i", "0"], capture_output=True, text=True, timeout=60).stdout.strip()
        name, power, clk = [v.strip() for v in out.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as e:                                    # the numbers below are then unattributed: say so
        return {"name": None, "power_limit": None, "error": repr(e)}


def rank_pad(r):
    return 4 if r <= 4 else (((r + 3) // 4) * 4 if r <= 16 else (24 if r <= 24 else 32))


def per_pass(T, torch, rows, ks, a, b):
    n = 256
    out = []
    os.environ["TLSQ_FUSED"] = "1"
    for k in ks:
        _, y = T.synth.sinusoids_np(rows + n - 1, k, seed=5)
        yd = torch.from_numpy(y).cuda()
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            T.lowrankfilter(yd, n, iters=3, tol=0.0)                          # warm-up: module load, every shape
        res = {}
        for its in (a, b):
            T.set_profiling(True)
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                _, info = T.lowrankfilter(yd, n, iters=its, tol=0.0, return_info=True)
            torch.cuda.synchronize()
            res[its] = (T.get_profile(), info)
            T.set_profiling(False)
        (pa, _), (pb, ib) = res[a], res[b]
        ranks = [int(v) for v in ib["hist"][a:b, 1]]
        dms, dn = pb["fused"][0] - pa["fused"][0], pb["fused"][1] - pa["fused"][1]
        out.append({"k": k, "rows": rows, "ranks": ranks, "rank_pads": sorted({rank_pad(r) for r in ranks}),
                    "passes": dn, "ms_per_pass": dms / dn if dn else None,
                    "handover": pb["epilogue"][1] > 0})
        del yd
    del os.environ["TLSQ_FUSED"]
    return out


def c5_high_rank(T, torch, k=12, Ns=50_000_000, reps=2):
    import numpy as np
    y0, y = T.synth.sinusoids_np(Ns, k, seed=5)
    y0d, yd = torch.from_numpy(y0).cuda(), torch.from_numpy(y).cuda()
    del y0, y
    runs = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        yf, info = T.lowrankfilter(yd, 256, return_info=True)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        mse = (torch.mean((yf - y0d) ** 2) / torch.mean(y0d ** 2)).item()
        runs.append({"seconds": dt, "iters": int(info["iters"]), "converged": bool(info["converged"]),
                     "sv": int(info["sv"]), "ranks": [int(v) for v in np.asarray(info["hist"])[:, 1]],
                     "normalised_mse_out": mse})
        del yf
    return {"Ns": Ns, "k": k, "runs": runs}


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
    ap.add_argument("--ks", type=int, nargs="*", default=[3, 6, 8, 12, 15])
    ap.add_argument("--iters", type=int, nargs=2, default=[8, 14], metavar=("A", "B"))
    ap.add_argument("--c5", action="store_true")
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
    res["per_pass"] = per_pass(T, torch, args.rows, args.ks, *args.iters)
    if args.c5:
        res["c5_high_rank"] = c5_high_rank(T, torch)
    res["card_after"] = card()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
