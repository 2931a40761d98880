"""lowrankfilter at n = 256 with rank estimates between 16 and 32 on the one-pass kernel (fused.cu, rank pads 24 and 32
of the implicit Hankel form), against the live CPU oracle.

The signals are sums of k sinusoids (synth.sinusoids_np): a rank estimate of about 2k.  An odd Hankel row count, Y
updated in place, or a sharded solve whose last shard has an odd row count keep the solve on the one-pass kernel, which
used to stop at rank 16."""
import os
import subprocess
import sys
import warnings

import numpy as np
import pytest

import tls_oracle as O
import tlsq_b200 as T

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
TOL = 1e-9
N_EMB = 256

_refs = {}


def relF(a, b):
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


def oracle(Ns, k, **kw):
    key = (Ns, k, tuple(sorted(kw.items())))
    if key not in _refs:
        _, y = T.synth.sinusoids_np(Ns, k, seed=5)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            _refs[key] = (y, O.rpca(O.hankel(y, N_EMB), **kw))
    return _refs[key]


def solve(y, env, monkeypatch, **kw):
    """lowrankfilter under `env`; also returns the per-phase spans (profiling on for the call)."""
    for k_, v_ in env.items():
        monkeypatch.setenv(k_, v_)
    try:
        T.set_profiling(True)
        yf, info = T.lowrankfilter(y, N_EMB, return_info=True, **kw)
        prof = T.get_profile()
        T.set_profiling(False)
    finally:
        for k_ in env:
            monkeypatch.delenv(k_)
    return yf, info, prof


def check(yf, info, ref):
    assert info["iters"] == ref.iters, (info["iters"], ref.iters)
    assert np.array_equal(info["hist"][:, 1], ref.hist[:, 1]), (info["hist"][:, 1], ref.hist[:, 1])
    assert info["sv"] == ref.sv
    err = relF(yf, O.unhankel_fast(ref.A))
    assert err < TOL, err


@pytest.mark.parametrize("k", [10, 13, 15])
def test_odd_row_count_runs_above_rank_16_on_the_one_pass_kernel(k, monkeypatch):
    """Ns = 20 256: K = 20 001 Hankel rows, odd, so the two-kernel pipeline is not available and the streaming pipeline
    cannot take over.  No environment switch: this is the default route."""
    y, ref = oracle(20_256, k, tol=1e-3)
    assert 16 < ref.hist[:, 1].max() <= 32
    yf, info, prof = solve(y, {}, monkeypatch)
    check(yf, info, ref)
    assert prof["fused"][1] > 0 and prof["epilogue"][1] == 0      # one-pass kernel throughout, no handover


def test_even_row_count_pipelines_agree(monkeypatch):
    """Ns = 20 255 (K = 20 000, rank up to 26): the two-kernel pipeline, the one-pass kernel, and the one-pass kernel
    with Y updated in place."""
    y, ref = oracle(20_255, 13, tol=1e-3)
    assert 16 < ref.hist[:, 1].max() <= 32
    out = []
    for env in ({"TLSQ_FUSED": "0"}, {"TLSQ_FUSED": "1"}, {"TLSQ_FUSED": "1", "TLSQ_INPLACE_Y": "1"}):
        yf, info, prof = solve(y, env, monkeypatch)
        check(yf, info, ref)
        if env["TLSQ_FUSED"] == "1":
            assert prof["fused"][1] > 0 and prof["epilogue"][1] == 0
        out.append(yf)
    assert relF(out[1], out[0]) < 1e-12 and relF(out[2], out[0]) < 1e-12 and relF(out[2], out[1]) < 1e-12


def test_inplace_dual_without_prediction_repeats_the_solve_above_rank_16(monkeypatch):
    """Y in place with the Z prediction off: an undecided Frobenius bracket is met without Z'Z at hand, and the solve is
    repeated with the two-phase iteration forced from there.  It stops at the reference's iteration."""
    y, ref = oracle(20_255, 13, tol=1e-3)
    yf0, info0, _ = solve(y, {"TLSQ_FUSED": "1", "TLSQ_INPLACE_Y": "1"}, monkeypatch)
    n0 = T.launch_count()
    yf1, info1, _ = solve(y, {"TLSQ_FUSED": "1", "TLSQ_INPLACE_Y": "1"}, monkeypatch)
    n1 = T.launch_count()
    yf2, info2, _ = solve(y, {"TLSQ_FUSED": "1", "TLSQ_INPLACE_Y": "1", "TLSQ_NO_PREDICT_Z": "1"}, monkeypatch)
    n2 = T.launch_count()
    check(yf2, info2, ref)
    assert info0["iters"] == info1["iters"] == ref.iters
    assert relF(yf1, yf2) < 1e-12
    assert n2 - n1 > 1.3 * (n1 - n0)                                   # it really ran (most of) the solve twice


def test_repeated_solves_at_rank_pad_32_are_bit_identical(monkeypatch):
    """Fixed-order reductions of the Gram partials, the T row sums and ||Z||^2: same input, same rank history, same
    ||Z||_F of every iteration the Frobenius bracket decides, same filtered signal.  The cost of the stopping iteration
    comes from the exact stop test (lambda_max of Z'Z by repeated squaring or Jacobi), outside this kernel, and is not
    compared bit for bit."""
    _, y = T.synth.sinusoids_np(20_256, 15, seed=5)                    # rank estimate up to 30: rank pad 32
    runs = [solve(y, {}, monkeypatch)[:2] for _ in range(4)]
    h0 = runs[0][1]["hist"]
    assert h0[:, 1].max() > 28
    for yf, info in runs[1:]:
        h = info["hist"]
        assert h.shape == h0.shape and np.array_equal(h[:, :2], h0[:, :2])
        assert np.array_equal(h[:-1, 2], h0[:-1, 2])
        assert np.array_equal(yf, runs[0][0])


def test_multi_gpu_sharded_odd_last_shard_above_rank_16():
    """2-rank sharded lowrankfilter whose last shard has an odd row count (tools/mgpu_fused_rank_check.py under
    torch.distributed.run).  Skipped with fewer than two GPUs."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29573",
                          os.path.join(ROOT, "tools", "mgpu_fused_rank_check.py")], capture_output=True, text=True,
                         env=env, timeout=1500)
    sys.stdout.write(out.stdout[-4000:])
    assert out.returncode == 0, out.stderr[-2000:]
    assert "MGPU_FUSED_RANK PASS" in out.stdout
