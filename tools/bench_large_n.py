#!/usr/bin/env python
"""rpca above 2048 columns on one GPU: 100 000 x N FP64, rank 10 + 5 % sparse, fixed seed, solved to the reference's
tolerance, for N = 4096 and N = 2048 beside it.  Prints ONE JSON line.

    python tools/bench_large_n.py [--rows 100000] [--cols 4096 2048]

Per N, three solves of the same matrix, all with the input resident in HBM:
  1. timed with CUDA events, profiling off: ALM iterations per second over the whole solve (returned SVD included);
  2. profiled (set_profiling / get_profile): per-phase device ms; SYRK rate from the `gram` phase and M N (N + 1) flop
     per Gram against the measured 37.1 TFLOP/s FP64 DMMA peak;
  3. profiled without the returned SVD: its `finalize` phase subtracted from solve 2's is the time of the returned-SVD
     refinement (full Jacobi of G, Cholesky, Jacobi of K, GEMMs).
The iterations whose eigen step fell back from the certified subspace iteration to the full Jacobi are counted from
the library's TLSQ_DEBUG_EIG lines (two 4-byte copies per iteration).  The card's name and power limit are read in the
same run.
"""
import argparse
import json
import math
import os
import re
import subprocess
import sys
import tempfile
import warnings

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ["TLSQ_DEBUG_EIG"] = "1"

FP64_TENSOR_PEAK_TFLOPS = 37.1      # measured FP64 DMMA peak of a B200 (profiles/r01_microbench_fp64_hbm.log)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                              "-i", "0"], capture_output=True, text=True, timeout=60).stdout.strip()
        name, power, clk = [v.strip() for v in out.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as e:                                    # the numbers below are then unattributed: say so
        return {"name": None, "power_limit": None, "error": repr(e)}


class StderrCapture:
    """Collects what the library writes to file descriptor 2 (its TLSQ_DEBUG_EIG lines)."""

    def __enter__(self):
        sys.stderr.flush()
        self.f = tempfile.TemporaryFile(mode="w+b")
        self.saved = os.dup(2)
        os.dup2(self.f.fileno(), 2)
        return self

    def __exit__(self, *a):
        sys.stderr.flush()
        os.dup2(self.saved, 2)
        os.close(self.saved)
        self.f.seek(0)
        self.text = self.f.read().decode("utf-8", "replace")
        self.f.close()


def run(M, N, seed):
    import torch

    import tlsq_b200 as T

    dev = torch.device("cuda", 0)
    D = T.synth.lowrank_sparse_cuda(0, M, N, dev, 10, 0.05, seed=seed, nonneg=False)
    lam = 1.0 / math.sqrt(max(M, N))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        Dw = T.synth.lowrank_sparse_cuda(0, N + 64, N, dev, 10, 0.05, seed=seed, nonneg=False)
        T.rpca(Dw, iters=2, tol=0.0)                              # loads the modules at this N (not timed)
        del Dw
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with StderrCapture() as cap:
            e0.record()
            A, E, s, sv, info = T.rpca(D, lam=lam, return_info=True)
            e1.record()
            torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        iters = info["iters"]
        fallbacks = len(re.findall(r"need_full 1", cap.text))
        T.set_profiling(True, 0)
        A, E, s, sv, info2 = T.rpca(D, lam=lam, return_info=True)
        prof = T.get_profile(0)
        T.set_profiling(False, 0)
        T.set_profiling(True, 0)
        T.rpca(D, lam=lam, want_svd=False)
        prof_nosvd = T.get_profile(0)
        T.set_profiling(False, 0)
    gram_ms, gram_calls = prof["gram"]
    syrk_ms = gram_ms / max(gram_calls, 1)
    flop = float(M) * N * (N + 1)
    tflops = flop / (syrk_ms * 1e-3) / 1e12
    return {
        "M": M, "N": N, "iters": iters, "converged": bool(info["converged"]), "sv": int(sv),
        "solve_ms": round(ms, 1), "alm_it_per_s": round(iters / (ms * 1e-3), 3),
        "phase_ms": {k: round(prof[k][0], 2) for k in ("gram", "eig", "epilogue", "exact_cost", "init", "finalize")},
        "phase_calls": {k: prof[k][1] for k in ("gram", "eig", "epilogue", "exact_cost", "init", "finalize")},
        "syrk_ms_per_gram": round(syrk_ms, 3), "syrk_tflops": round(tflops, 2),
        "syrk_share_of_dmma_peak": round(tflops / FP64_TENSOR_PEAK_TFLOPS, 3),
        "full_jacobi_fallback_iters": fallbacks,
        "svd_refinement_ms": round(prof["finalize"][0] - prof_nosvd["finalize"][0], 1),
        "finalize_ms_without_svd": round(prof_nosvd["finalize"][0], 1),
        "profiled_iters": info2["iters"],
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=100_000)
    ap.add_argument("--cols", type=int, nargs="+", default=[4096, 2048])
    ap.add_argument("--seed", type=int, default=41)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_large_n: needs a CUDA device")
    info = card()
    res = []
    for n in args.cols:
        res.append(run(args.rows, n, args.seed))
        print(json.dumps(res[-1]), file=sys.stderr, flush=True)     # progress: one line per finished N
    print(json.dumps({"workload": f"rpca {args.rows}xN FP64 rank10+5%sparse seed {args.seed}, tol sqrt(eps)",
                      "device": info, "dmma_peak_tflops": FP64_TENSOR_PEAK_TFLOPS,
                      "flop_per_gram": "M*N*(N+1)", "results": res}))


if __name__ == "__main__":
    main()
