#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 robust-PCA hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload c4|c2|c3|c5]
                    [--dump-outputs DIR]

One "step" = one full `rpca` solve to the reference's tolerance (sqrt(eps)) on the workload:
    c4 (default, the configuration the metric is quoted on): 1 000 000 x 256 FP64, rank 10 + 5 % sparse,
        nonnegA=true; rows sharded over the N GPUs (strong scaling: the global matrix is fixed)
    c2: 100 000 x 512 FP64, rank 10 + 5 % sparse (single GPU)
    c3: rpca_ga(X, 10) on 2 000 000 x 256 (rows sharded); metric = Grassmann iterations/s
    c5: lowrankfilter(y, 256) on a 50 000 000-sample sinusoid sum with 10 % missing values (implicit Hankel matrix
        49 999 745 x 256, never materialised; Hankel rows sharded); one step = one full filter run (tol 1e-3)
Metric: ALM iterations per second (whole job).  `value` is measured with the input resident in HBM, `e2e` through
the public host-buffer API (pinned host memory, H2D of D and D2H of A and E inside the timed region).
`--impl reference` times the CPU restatement of the reference (oracle/, same LAPACK routines the Julia reference
reaches through OpenBLAS; Julia itself is not installed in this image) on a bounded row sample.
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

def measured_traffic(kernel: str, rows: int, cols: int):
    """dram read+write GB per launch from a committed `ncu --set full` capture (profiles/traffic.json, keyed by kernel
    and "<rows per GPU>x<cols>"); None for shapes that were never profiled."""
    try:
        tab = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        return tab.get(kernel, {}).get(f"{rows}x{cols}")
    except Exception:
        return None


FP64_TENSOR_PEAK_TFLOPS = 37.1      # measured on this pool's B200 (tools/microbench.cu -> profiles/r01_microbench_fp64_hbm.log)

WORKLOADS = {
    "c4": dict(kind="rpca", M=1_000_000, N=256, rank=10, frac=0.05, seed=4, nonneg=True,
               name="rpca 1Mx256 FP64 rank10+5%sparse nonnegA=true (BASELINE configs[3])"),
    "c2": dict(kind="rpca", M=100_000, N=512, rank=10, frac=0.05, seed=2, nonneg=False,
               name="rpca 100kx512 FP64 rank10+5%sparse (BASELINE configs[1])"),
    "c3": dict(kind="ga", M=2_000_000, N=256, rank=10, seed=3,
               name="rpca_ga(X,10) 2Mx256 FP64 10% gross outliers (BASELINE configs[2])"),
    "c5": dict(kind="lrf", M=50_000_000, N=256, seed=5,
               name="lowrankfilter(y,256) 50M-sample sinusoid sum, 10% missing (BASELINE configs[4]; implicit Hankel "
                    "49999745x256)"),
}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0}, "fallback"


DUMP_LIMIT_BYTES = 64_000_000
DUMP_SEED = 20240


def dump_outputs(path, rows, small):
    """Write the outputs of one solve to `path`/<name>.npy as float64 so that two builds can be compared output for
    output.  `rows`: arrays that share their first (row) dimension (torch tensors or NumPy arrays); when they do not
    fit in DUMP_LIMIT_BYTES a fixed, seeded sample of rows is written, and `row_index.npy` names the rows.  `small`:
    arrays written whole."""
    import numpy as np
    os.makedirs(path, exist_ok=True)

    def host(v):
        return np.asarray(v.cpu().numpy() if hasattr(v, "cpu") else v, dtype=np.float64)
    out = {k: host(v) for k, v in small.items()}
    m = next(iter(rows.values())).shape[0]
    per_row = 8 * (1 + sum(math.prod(v.shape[1:]) for v in rows.values()))           # + 8 bytes of row_index
    room = DUMP_LIMIT_BYTES - sum(a.nbytes for a in out.values()) - 128 * (len(out) + len(rows) + 1)   # npy headers
    k = min(m, room // per_row)
    idx = np.arange(m) if k == m else np.sort(np.random.default_rng(DUMP_SEED).choice(m, size=k, replace=False))
    for name, v in rows.items():
        if hasattr(v, "index_select"):                                 # torch: gather the sample on the device
            import torch
            v = v.index_select(0, torch.from_numpy(idx).to(v.device))
        else:
            v = v[idx]
        out[name] = host(v)
    out["row_index"] = idx.astype(np.float64)
    for name, a in out.items():
        np.save(os.path.join(path, f"{name}.npy"), a)


# ----------------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi in the background during the timed region)
# ----------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc = index, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        for line in out.splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port on a bounded row sample
# ----------------------------------------------------------------------------------------------------------
def pin_cpu_threads():
    """torchrun exports OMP_NUM_THREADS=1; the CPU arm must use every host core like the Julia reference would
    (OpenBLAS threads inside dgesdd/dgemm).  Called before NumPy/SciPy are imported, and enforced again at run time."""
    n = str(os.cpu_count() or 1)
    for k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[k] = n


class _AllThreads:
    def __enter__(self):
        try:
            from threadpoolctl import threadpool_limits
            self.ctx = threadpool_limits(limits=os.cpu_count() or 1)
            self.ctx.__enter__()
        except Exception:
            self.ctx = None
        return self

    def __exit__(self, *a):
        if self.ctx is not None:
            self.ctx.__exit__(*a)


def cpu_rpca_sample(w, sample_rows: int, iters: int):
    """iterations/s of the oracle on the first `sample_rows` rows, EXTRAPOLATED to the full row count (cost is linear in
    the number of rows: dgesdd on M x n, n fixed, and the element-wise sweeps)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import warnings

    import numpy as np
    import tls_oracle as O
    import tlsq_b200 as T
    D = T.synth.lowrank_sparse_np(sample_rows, w["N"], w["rank"], w["frac"], w["seed"], w["nonneg"])
    with warnings.catch_warnings(), _AllThreads():
        warnings.simplefilter("ignore")
        t0 = time.perf_counter()
        res = O.rpca(D, iters=iters, tol=0.0, nonnegA=w["nonneg"], lam=1.0 / math.sqrt(w["M"]))
        dt = time.perf_counter() - t0
    its_per_s_sample = res.iters / dt
    return its_per_s_sample * sample_rows / w["M"], dt, res.iters


def cpu_ga_sample(w, sample_rows: int, r: int):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import tls_oracle as O
    import tlsq_b200 as T
    X, q0 = T.synth.ga_data_np(sample_rows, w["N"], w["rank"], w["seed"])
    with _AllThreads():
        t0 = time.perf_counter()
        _, its = O.rpca_ga(X, r, q0=q0[:, :r], exact_order=False, return_iters=True)
        dt = time.perf_counter() - t0
    return sum(its) / dt * sample_rows / w["M"], dt, sum(its)


def cpu_lrf_sample(w, sample_ns: int, iters: int):
    """ALM iterations/s of the oracle's lowrankfilter core (rpca on the MATERIALISED Hankel embedding, which is what the
    reference does, src/robustPCA.jl:120-122) on `sample_ns` samples, extrapolated linearly in the number of Hankel rows."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import warnings

    import tls_oracle as O
    import tlsq_b200 as T
    _, yn = T.synth.sinusoid_np(sample_ns, seed=w["seed"])
    H = O.hankel(yn, w["N"])
    with warnings.catch_warnings(), _AllThreads():
        warnings.simplefilter("ignore")
        t0 = time.perf_counter()
        res = O.rpca(H, iters=iters, tol=0.0)
        dt = time.perf_counter() - t0
    K_full = w["M"] - w["N"] + 1
    return res.iters / dt * H.shape[0] / K_full, dt, res.iters


def cpu_cores():
    try:
        from threadpoolctl import threadpool_info
        n = [p.get("num_threads") for p in threadpool_info() if p.get("user_api") == "blas"]
        if n:
            return int(max(n))
    except Exception:
        pass
    return os.cpu_count() or 1


def cpu_leg(w):
    """one bounded CPU sample of the workload -> (value, seconds, description, unit)"""
    if w["kind"] == "rpca":
        sample_rows, its = (50_000 if w["N"] <= 256 else 20_000), 3
        v, dt, its = cpu_rpca_sample(w, sample_rows, its)
        return v, dt, (f"{its} ALM iterations of the oracle port (LAPACK dgesdd/dgemm via SciPy OpenBLAS) on the first "
                       f"{sample_rows} rows ({dt:.1f} s), EXTRAPOLATED x{sample_rows}/{w['M']} (cost linear in rows)"), \
            "ALM iterations/s"
    if w["kind"] == "ga":
        v, dt, its = cpu_ga_sample(w, 100_000, 2)
        return v, dt, (f"rpca_ga(X,2) of the oracle port on the first 100000 rows ({dt:.1f} s), EXTRAPOLATED "
                       f"x100000/{w['M']}"), "GA iterations/s"
    v, dt, its = cpu_lrf_sample(w, 100_000, 2)
    return v, dt, (f"{its} ALM iterations of the oracle port on the materialised Hankel embedding of the first 100000 "
                   f"samples ({dt:.1f} s), EXTRAPOLATED linearly in the Hankel rows (the reference cannot hold the "
                   f"full 102 GB x 5 buffers)"), "ALM iterations/s"


def run_reference(args, w, rank):
    if rank != 0:
        return
    import numpy  # noqa: F401  (loads OpenBLAS so that cpu_cores() sees it)
    import scipy.linalg  # noqa: F401
    vals, dts = [], []
    sample, unit = "", ""
    for i in range(args.warmup + args.steps):
        v, dt, sample, unit = cpu_leg(w)
        if i >= args.warmup:
            vals.append(v); dts.append(dt)
    value = sum(vals) / len(vals)
    line = {"metric": metric_name(w), "value": value, "unit": unit, "impl": "reference", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sum(dts) / len(dts),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": w["name"], "cpu_sample": "bounded row sample, extrapolated linearly to the full size"},
            "cpu_baseline": {"value": value, "unit": unit, "cores": cpu_cores(), "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    EMIT(json.dumps(line))


def metric_name(w):
    return {"rpca": "rpca_alm_iterations_per_s", "ga": "rpca_ga_iterations_per_s",
            "lrf": "lowrankfilter_alm_iterations_per_s"}[w["kind"]]


# ----------------------------------------------------------------------------------------------------------
# B200 arm
# ----------------------------------------------------------------------------------------------------------
def c5_signal(Ns, dev, seed):
    """C5 signal on the device (every rank builds the same full signal: same Philox stream on every GPU)."""
    import torch
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    t = torch.arange(1, Ns + 1, device=dev, dtype=torch.float64)
    y = torch.sin(0.1 * t) + 0.5 * torch.sin(0.37 * t + 1.0) + 0.25 * torch.sin(0.013 * t + 2.0)
    del t
    mask = torch.rand(Ns, device=dev, generator=g) < 0.1
    yn = y + 1e2 * mask.double()
    return y, yn


def run_b200(args, w, rank, world, local_rank):
    import numpy as np
    import torch
    import torch.distributed as dist

    import tlsq_b200 as T

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        T.init_distributed(local_rank)
    M, N = w["M"], w["N"]
    r0, r1 = T.synth.shard_rows(M, world, rank, align=T.synth.CHUNK_ROWS)
    m = r1 - r0
    lam = 1.0 / math.sqrt(max(M, N))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allsum(x):
        t = torch.tensor([float(x)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t)
        return float(t.item())

    parity = {}
    last = {}                                                     # outputs of the last timed step (--dump-outputs)
    if w["kind"] == "rpca":
        D = T.synth.lowrank_sparse_cuda(r0, r1, N, dev, w["rank"], w["frac"], w["seed"], w["nonneg"])
        kw = dict(nonnegA=w["nonneg"], lam=lam)

        def step(keep=False):
            A, E, s, sv, info = T.rpca(D, return_info=True, **kw)
            if keep:
                last["rows"] = {"A": A, "E": E, "U": s.U}
                last["small"] = {"S": s.S, "Vt": s.Vt, "sv": sv, "iters": info["iters"]}
            return info["iters"]

        def parity_solve():
            A, E, s, sv, info = T.rpca(D, return_info=True, **kw)
            return {"iters": info["iters"], "sv": int(sv), "A_fro": math.sqrt(allsum((A * A).sum().item())),
                    "E_fro": math.sqrt(allsum((E * E).sum().item())), "E_nnz": int(allsum((E != 0).sum().item())),
                    "S_head": [float(v) for v in s.S[:3].cpu()], "S_tail": float(s.S[-1].item()),
                    "note": "same global matrix at every N (chunk-seeded generator): compare across the N lines"}
    elif w["kind"] == "ga":
        X, q0 = T.synth.ga_data_cuda(r0, r1, N, dev, w["rank"], w["seed"])

        def step(keep=False):
            Q, info = T.rpca_ga(X, w["rank"], q0=q0, return_info=True)
            if keep:
                last["rows"], last["small"] = {"Q": Q}, {"iters": info["iters"]}
            return sum(info["iters"])

        def parity_solve():
            Q, info = T.rpca_ga(X, w["rank"], q0=q0, return_info=True)
            cs = Q.sum(dim=0)
            if world > 1:
                dist.all_reduce(cs)
            return {"iters": [int(v) for v in info["iters"]], "abs_colsum_Q": [abs(float(v)) for v in cs.cpu()]}
    else:
        y_clean, yn = c5_signal(M, dev, w["seed"])
        m = M                                                     # every rank holds the (small) signal
        lrf_last = {}

        def step(keep=False):
            yf, info = T.lowrankfilter(yn, N, return_info=True)
            lrf_last["yf"], lrf_last["info"] = yf, info
            if keep:
                last["rows"], last["small"] = {"yf": yf}, {"iters": info["iters"], "sv": info["sv"]}
            return info["iters"]

        def parity_solve():
            it = step()
            yf = lrf_last["yf"]
            return {"iters": it, "sv": int(lrf_last["info"].get("sv", 0)),
                    "normalised_mse_out": (torch.mean((y_clean - yf) ** 2) / torch.mean(y_clean ** 2)).item(),
                    "normalised_mse_in": (torch.mean((y_clean - yn) ** 2) / torch.mean(y_clean ** 2)).item(),
                    "yf_norm": float(torch.linalg.norm(yf).item())}

    # ---- device-resident timing ---------------------------------------------------------------------------
    for _ in range(args.warmup):
        step()
    sampler = ClockSampler(local_rank)
    barrier()
    if rank == 0:
        sampler.start()
    l0 = T.launch_count(local_rank)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    iters_total = 0
    for i in range(args.steps):
        iters_total += step(keep=args.dump_outputs is not None and i == args.steps - 1)
    e1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    launches = T.launch_count(local_rank) - l0
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    value = iters_total / (ms * 1e-3)
    if args.dump_outputs is not None:
        dump_outputs(args.dump_outputs, last.pop("rows"), last.pop("small"))

    # ---- one profiled solve: per-phase device times for the roofline; one more for the cross-N parity digest ---
    T.set_profiling(True, local_rank)
    it_prof = step()
    prof = T.get_profile(local_rank)
    T.set_profiling(False, local_rank)
    parity = parity_solve()

    # ---- end-to-end through the host-buffer API (pinned host memory) ----------------------------------------
    def time_host(fn, nst):
        fn()
        barrier()
        t0 = time.perf_counter()
        it_e = 0
        for _ in range(nst):
            it_e += fn()
        barrier()
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        return it_e / float(dt.item()), 1e3 * float(dt.item()) / nst

    def pinned_cm(rows, cols):
        return torch.empty((cols, rows), dtype=torch.float64, pin_memory=True).numpy().T

    e2e = None
    extra = {}
    if w["kind"] == "rpca":
        Dh = torch.empty((N, m), dtype=torch.float64, pin_memory=True)
        Dh.copy_(D.t())
        Dn = Dh.numpy().T                                          # column-major (m, N) view of pinned memory
        Ah, Eh = pinned_cm(m, N), pinned_cm(m, N)
        del D
        torch.cuda.empty_cache()
        nst = args.steps

        dd = min(M, N)
        Uh, Vth = pinned_cm(m, dd), pinned_cm(dd, N)
        Sh = torch.empty((dd,), dtype=torch.float64, pin_memory=True).numpy()

        def step_e2e_svd():                                        # what rpca returns: (A, E, s, sv)
            _, _, s, _, info = T.rpca(Dn, return_info=True, want_svd=True, out=(Ah, Eh, Uh, Sh, Vth), **kw)
            return info["iters"]

        def step_e2e():
            _, _, _, _, info = T.rpca(Dn, return_info=True, want_svd=False, out=(Ah, Eh), **kw)
            return info["iters"]
        v1, ms1 = time_host(step_e2e_svd, nst)
        v2, ms2 = time_host(step_e2e, nst)
        d = min(M, N)
        e2e = {"value": v1, "unit": "ALM iterations/s", "h2d_bytes_per_step": int(m * N * 8),
               "d2h_bytes_per_step": int(2 * m * N * 8 + m * d * 8 + d * 8 + d * N * 8), "ms_per_step": ms1, "steps": nst,
               "api": "tlsq_b200.rpca(numpy pinned D) -> tlsq_rpca_f64: A, E AND the SVD s = (U, S, Vt) returned to the "
                      "host, like the reference's (A, E, s, sv)"}
        extra["e2e_no_svd"] = {"value": v2, "unit": "ALM iterations/s", "h2d_bytes_per_step": int(m * N * 8),
                               "d2h_bytes_per_step": int(2 * m * N * 8), "ms_per_step": ms2, "steps": nst,
                               "api": "same call with want_svd=False (A and E only)"}
    elif w["kind"] == "ga":
        Xh = torch.empty((N, m), dtype=torch.float64, pin_memory=True)
        Xh.copy_(X.t())
        Xn, q0n = Xh.numpy().T, np.asfortranarray(q0.cpu().numpy())

        def step_e2e():
            _, info = T.rpca_ga(Xn, w["rank"], q0=q0n, return_info=True)
            return sum(info["iters"])
        v1, ms1 = time_host(step_e2e, max(1, min(args.steps, 3)))
        e2e = {"value": v1, "unit": "GA iterations/s", "h2d_bytes_per_step": int(m * N * 8 + m * w["rank"] * 8),
               "d2h_bytes_per_step": int(m * w["rank"] * 8), "ms_per_step": ms1}
    else:
        yh = torch.empty((M,), dtype=torch.float64, pin_memory=True)
        yh.copy_(yn)
        ynp = yh.numpy()

        def step_e2e():
            _, info = T.lowrankfilter(ynp, N, return_info=True)
            return info["iters"]
        v1, ms1 = time_host(step_e2e, max(1, min(args.steps, 2)))
        e2e = {"value": v1, "unit": "ALM iterations/s", "h2d_bytes_per_step": int(M * 8), "d2h_bytes_per_step": int(M * 8),
               "ms_per_step": ms1, "api": "tlsq_b200.lowrankfilter(numpy pinned y) -> tlsq_lowrankfilter_f64"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks, peak_src = measured_peaks()
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    unit = "GA iterations/s" if w["kind"] == "ga" else "ALM iterations/s"
    rows_local = m if w["kind"] != "lrf" else (M - N + 1 + world - 1) // world
    line = {"metric": metric_name(w), "value": value, "unit": unit, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": w["name"], "rows_per_gpu": rows_local, "cols": N,
                       "l2": "inputs (>=0.4 GB per pass) larger than the 126 MB L2"},
            "iters_per_step": iters_total / args.steps, "time_to_converge_s": ms * 1e-3 / args.steps,
            "gpu_launches": int(launches), "clocks": clocks, "e2e": e2e, "parity": parity}
    line.update(extra)
    m = rows_local
    if w["kind"] in ("rpca", "lrf"):
        g_ms, g_n = prof["gram"]
        e_ms, e_n = prof["epilogue"]
        j_ms, j_n = prof["eig"]
        f_ms, f_n = prof.get("fused", (0.0, 0))
        x_ms, x_n = prof.get("exact_cost", (0.0, 0))
        svp = w.get("rank", 6)
        S = m * N * 8
        gram_flops = m * N * (N + 1)                               # SYRK count per launch (SURVEY.md 8d)
        epi_flops = 4 * m * N * svp + 12 * m * N                   # low-rank reconstruction + element-wise (8d)
        peak_src64 = ("measured FP64 DMMA peak, profiles/r01_microbench_fp64_hbm.log "
                      "(MEASURED_PEAKS.json has no FP64 figure)")
        if f_n > 0:
            # one-pass pipeline: the dominant kernel is alm_fused_kernel (epilogue of iteration k + Gram of iteration
            # k+1).  Both halves run on the FP64 pipe (DMMA and DFMA share it), so the bound is FP64 arithmetic.
            t_f = f_ms / f_n * 1e-3
            ach = (gram_flops + epi_flops) / t_f * 1e-12
            line["roofline"] = {"kernel": "alm_fused_kernel (epilogue of iteration k + DMMA Gram of iteration k+1, "
                                          "one HBM pass)", "bound": "tensor", "achieved": ach,
                                "peak": FP64_TENSOR_PEAK_TFLOPS, "unit": "TFLOP/s", "frac": ach / FP64_TENSOR_PEAK_TFLOPS,
                                "peak_source": peak_src64, "algorithmic_flops": "M*N*(N+1) + 4*M*N*svp + 12*M*N "
                                "(SURVEY.md 8d: F_gram + F_epi)", "traffic": measured_traffic("alm_fused_kernel", m, N),
                                "traffic_unit": "GB per launch (dram read+write, ncu --set full, profiles/traffic.json)",
                                "avg_launch_ms": t_f * 1e3, "launches_profiled": f_n,
                                "hbm_view": {"algorithmic_GBps": 9 * S / t_f * 1e-9, "moved_GBps": 3 * S / t_f * 1e-9,
                                             "peak": hbm, "note": "9S = SURVEY 8d two-pass count; the kernel moves 3S "
                                                                   "(reads D, Y; writes Y)"}}
        else:
            t_gram = g_ms / max(g_n, 1) * 1e-3
            ach = gram_flops / t_gram * 1e-12 if t_gram > 0 else 0.0
            line["roofline"] = {"kernel": "syrk_tma_kernel (DMMA SYRK of the SVT input)", "bound": "tensor",
                                "achieved": ach, "peak": FP64_TENSOR_PEAK_TFLOPS, "unit": "TFLOP/s",
                                "frac": ach / FP64_TENSOR_PEAK_TFLOPS, "peak_source": peak_src64,
                                "algorithmic_flops": "M*N*(N+1) (SYRK count, SURVEY.md 8d)",
                                "traffic": measured_traffic("syrk_tma_kernel", m, N),
                                "traffic_unit": "GB per launch (dram read+write, ncu --set full, profiles/traffic.json)",
                                "avg_launch_ms": t_gram * 1e3}
            t_epi = e_ms / max(e_n, 1) * 1e-3
            moved = measured_traffic("epilogue_tma", m, N)
            line["roofline_epilogue"] = {"kernel": "tproj_tma_kernel + alm_ew_tma_kernel (T projection, element-wise pass; "
                                                   "TMA-staged)",
                                         "bound": "hbm", "traffic": moved,
                                         "achieved": 6 * S / t_epi * 1e-9 if t_epi > 0 else 0.0, "peak": hbm,
                                         "unit": "GB/s", "frac": (6 * S / t_epi * 1e-9) / hbm if t_epi > 0 else 0.0,
                                         "frac_of_moved_bytes": (moved / t_epi / hbm) if (moved and t_epi > 0) else None,
                                         "peak_source": f"MEASURED_PEAKS.json hbm_gbs ({peak_src})",
                                         "algorithmic_bytes": "6*S (reads D,A,Y; writes A,E,Y; SURVEY.md 8d); "
                                                              "frac_of_moved_bytes uses the ncu-measured DRAM bytes",
                                         "avg_launch_ms": t_epi * 1e3}
        # per-iteration roofline (SURVEY.md 8d):  max(F_gram/P64, 3S/BW) + max(F_epi/P64, 6S/BW)
        # (C5: implicit D, factored A, no E -> the byte counts are 1S + 2S, SURVEY.md 8d)
        b_gram, b_epi = (3 * S, 6 * S) if w["kind"] == "rpca" else (1 * S, 2 * S)
        t_roof = max(gram_flops / (FP64_TENSOR_PEAK_TFLOPS * 1e12), b_gram / (hbm * 1e9)) + \
            max(epi_flops / (FP64_TENSOR_PEAK_TFLOPS * 1e12), b_epi / (hbm * 1e9))
        t_iter = ms * 1e-3 / max(iters_total, 1)
        line["iteration_roofline"] = {"roofline_ms": t_roof * 1e3, "measured_ms": t_iter * 1e3,
                                      "frac": t_roof / t_iter if t_iter > 0 else 0.0,
                                      "phase_ms_per_iter": {k: v[0] / max(it_prof, 1) for k, v in prof.items()},
                                      "eig_avg_ms": j_ms / max(j_n, 1)}
    else:
        s_ms, s_n = prof["ga_sweep"]
        t_sw = s_ms / max(s_n, 1) * 1e-3
        bytes_ = m * N * 8
        line["roofline"] = {"kernel": "ga_sweep_tma_kernel<GA_PASS>", "bound": "hbm",
                            "achieved": bytes_ / t_sw * 1e-9 if t_sw > 0 else 0.0, "peak": hbm, "unit": "GB/s",
                            "frac": (bytes_ / t_sw * 1e-9) / hbm if t_sw > 0 else 0.0,
                            "peak_source": f"MEASURED_PEAKS.json hbm_gbs ({peak_src}); a read-only stream can exceed "
                                           "the copy figure (7.2 TB/s read-only, profiles/r01_microbench_fp64_hbm.log)",
                            "traffic": measured_traffic("ga_sweep_tma_kernel", m, N),
                            "traffic_unit": "GB per launch (dram read+write, ncu --set full, profiles/traffic.json)",
                            "avg_launch_ms": t_sw * 1e3}
    # CPU baseline beside it (rank 0, N == 1 only), bounded sample
    if world == 1 and not args.no_cpu:
        v, dt, sample, cunit = cpu_leg(w)
        line["cpu_baseline"] = {"value": v, "unit": cunit, "cores": cpu_cores(), "kind": "port", "sample": sample}
    EMIT(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def _quiet_stdout():
    """Route fd 1 to stderr while the benchmark runs (NCCL prints its version banner on stdout when NCCL_DEBUG is set)
    and hand back a writer for the one JSON line."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)

    def emit(text: str):
        sys.stdout.flush()
        os.write(real, (text + "\n").encode())
    return emit


EMIT = None


def main():
    global EMIT
    EMIT = _quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c4", choices=sorted(WORKLOADS))
    ap.add_argument("--rows", type=int, default=0, help="override the row count (debugging)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned to DIR/<name>.npy "
                    "(float64, at most 64 MB: a fixed, seeded row sample of the large outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and (args.impl != "b200" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs needs --impl b200 in a single process")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = max(args.warmup, 1)
    w = dict(WORKLOADS[args.workload])
    if args.rows:
        w["M"] = args.rows
        w["name"] += f" [rows overridden to {args.rows}]"
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        pin_cpu_threads()            # before NumPy / SciPy load OpenBLAS (torchrun exports OMP_NUM_THREADS=1)
        run_reference(args, w, rank)
        return
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    run_b200(args, w, rank, world, local_rank)


if __name__ == "__main__":
    main()
