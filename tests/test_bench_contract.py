"""bench.py contract checks.  Without a GPU: --dump-outputs keeps its size cap and row sample, the reference arm
(`--impl reference`) times the CPU oracle port on a bounded sample and prints ONE JSON line with the keys the driver
reads; the product arm refuses to run without a GPU (no CPU fallback).  On the GPU: --dump-outputs holds what the
last timed solve returned."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, timeout=300):
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], cwd=ROOT, env=env, timeout=timeout,
                          capture_output=True, text=True)


def test_reference_arm_prints_the_contract_line():
    r = _run("--impl", "reference", "--steps", "1", "--warmup", "0")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "rpca_alm_iterations_per_s"
    assert d["unit"] == "ALM iterations/s" and d["higher_is_better"] is True and d["dtype"] == "f64"
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 0 and d["vs_baseline"] is None
    assert d["value"] > 0 and d["ms_per_step"] > 0
    assert "workload" in d["config"] and "1Mx256" in d["config"]["workload"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "EXTRAPOLATED" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_dump_outputs_stays_under_64_mb_with_a_fixed_row_sample(tmp_path):
    import numpy as np
    import torch

    import bench
    rng = np.random.default_rng(0)
    rows = {"A": torch.from_numpy(rng.standard_normal((40_000, 256))), "y": rng.standard_normal(40_000)}
    small = {"S": rng.standard_normal(256), "sv": 7, "iters": [3, 4]}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), rows, small)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["A.npy", "S.npy", "iters.npy", "row_index.npy", "sv.npy", "y.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64_000_000
    out = {f[:-4]: np.load(tmp_path / "a" / f) for f in files}
    assert all(a.dtype == np.float64 for a in out.values())
    idx = out["row_index"].astype(np.int64)
    assert 10_000 < len(idx) < 40_000 and np.all(np.diff(idx) > 0)
    assert np.array_equal(out["A"], rows["A"].numpy()[idx]) and np.array_equal(out["y"], rows["y"][idx])
    assert np.array_equal(out["S"], small["S"]) and out["sv"] == 7 and list(out["iters"]) == [3, 4]
    for f in files:                                           # same arguments, same sample
        assert np.array_equal(np.load(tmp_path / "b" / f), out[f[:-4]])


def test_steps_must_be_positive():
    r = _run("--impl", "reference", "--steps", "0", "--warmup", "0")
    assert r.returncode != 0 and "--steps" in r.stderr


@pytest.mark.gpu
def test_dump_outputs_holds_what_the_timed_solve_returned(tmp_path):
    import math

    import numpy as np
    import torch

    import tlsq_b200 as T
    M, N = 31_250, 256
    r = _run("--rows", str(M), "--steps", "2", "--warmup", "1", "--no-cpu", "--dump-outputs", str(tmp_path), timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][0])
    assert d["steps"] == 2
    out = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert sum(a.nbytes for a in out.values()) <= 64_000_000
    D = T.synth.lowrank_sparse_cuda(0, M, N, torch.device("cuda", 0), 10, 0.05, seed=4, nonneg=True)
    A, E, s, sv, info = T.rpca(D, nonnegA=True, lam=1.0 / math.sqrt(M), return_info=True)
    idx = torch.from_numpy(out["row_index"].astype(np.int64)).cuda()
    assert 0 < len(idx) < M and int(out["sv"]) == sv and int(out["iters"]) == info["iters"]
    for name, ref in (("A", A), ("E", E)):
        ref = ref.index_select(0, idx).cpu().numpy()
        assert np.linalg.norm(out[name] - ref) <= 1e-9 * np.linalg.norm(ref), name
    assert np.allclose(out["S"], s.S.cpu().numpy(), rtol=0, atol=1e-12 * float(s.S[0]))


def test_product_arm_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        return                                   # on the GPU box the bench itself is the check
    r = _run("--steps", "1", "--warmup", "0", timeout=120)
    assert r.returncode != 0
    assert not any(ln.startswith("{") for ln in r.stdout.splitlines())
