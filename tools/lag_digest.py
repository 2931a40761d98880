#!/usr/bin/env python
"""SHA-256 of lowrankfilter's filtered signal for a fixed list of lag > 1 solves that take the two-kernel pipeline
(even Hankel row count, n >= 65, memory to spare).  Prints ONE JSON line.

    python tools/lag_digest.py [--tree DIR] [--compare-tree DIR]

--tree DIR: import the library from another built checkout (default: this one).
--compare-tree DIR: run the list in a process of its own for DIR and for this tree, one after the other, and report
whether every digest, iteration count and rank history agrees.
The inputs are sums of k sinusoids (synth.sinusoids_np, seed 5) of (K - 1) lag + n samples.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# (n, lag, Hankel rows K, sinusoids k)
CASES = [(256, 2, 20_000, 6), (256, 3, 20_000, 6), (256, 7, 20_000, 5), (256, 2, 20_000, 13), (128, 4, 20_000, 5),
         (600, 3, 6_000, 6), (256, 256, 8_192, 5), (256, 2, 1_000_000, 6)]


def run(tree):
    sys.path.insert(0, tree)
    import numpy as np
    import torch
    import tlsq_b200 as T
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device")
    out = []
    for n, lag, K, k in CASES:
        Ns = (K - 1) * lag + n
        _, y = T.synth.sinusoids_np(Ns, k, seed=5)
        T.set_profiling(True)
        yf, info = T.lowrankfilter(y, n, lag=lag, return_info=True)
        prof = T.get_profile()
        T.set_profiling(False)
        yf = np.ascontiguousarray(yf, dtype=np.float64)
        out.append({"n": n, "lag": lag, "K": K, "k": k, "sha256": hashlib.sha256(yf.tobytes()).hexdigest(),
                    "iters": int(info["iters"]), "ranks": [int(v) for v in np.asarray(info["hist"])[:, 1]],
                    "fused_spans": prof["fused"][1], "epilogue_spans": prof["epilogue"][1]})
    return {"tree": os.path.abspath(tree), "lib": os.path.abspath(T.__file__), "cases": out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tree", default=ROOT)
    ap.add_argument("--compare-tree")
    args = ap.parse_args()
    if not args.compare_tree:
        print(json.dumps(run(args.tree)))
        return
    res = {}
    for name, tree in (("other", args.compare_tree), ("this", ROOT)):
        p = subprocess.run([sys.executable, os.path.abspath(__file__), "--tree", os.path.abspath(tree)],
                           capture_output=True, text=True, timeout=3000)
        line = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
        if p.returncode != 0 or not line:
            raise SystemExit(f"{tree}: {p.stderr[-2000:]}")
        res[name] = json.loads(line[-1])
    keys = ("sha256", "iters", "ranks")
    same = [all(a[key] == b[key] for key in keys) for a, b in zip(res["other"]["cases"], res["this"]["cases"])]
    res["identical"] = same
    res["all_identical"] = all(same)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
