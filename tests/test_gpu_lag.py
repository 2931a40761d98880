"""lowrankfilter with lag > 1 on the factored route: the implicit Hankel matrix H[k, l] = y[k lag + l] on the one-pass
kernel (fused.cu, every Hankel rank pad) or the two-kernel pipeline, and the factored unhankel for that lag
(elementwise.cu), against the live CPU oracle (src/robustPCA.jl:53-68, 76-92, 119-128).

The signals are sums of k sinusoids (synth.sinusoids_np): a rank estimate of about 2k whatever the lag.  An odd Hankel
row count keeps the solve on the one-pass kernel; an even one takes the two-kernel pipeline unless TLSQ_FUSED=1."""
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


def unhankel_lag(A, lag, Ns):
    """The reference's unhankel (:53-68) for one channel, vectorised over the rows: terms in increasing l, then
    y ./= max.(counts, 1)."""
    K, L = A.shape
    s = np.zeros(Ns)
    cnt = np.zeros(Ns)
    for l in range(L):
        s[l:l + (K - 1) * lag + 1:lag] += A[:, l]
        cnt[l:l + (K - 1) * lag + 1:lag] += 1
    return s / np.maximum(cnt, 1)


def signal_len(K, lag, n=N_EMB, tail=0):
    """Ns with (Ns - n) // lag + 1 == K Hankel rows and `tail` (< lag) samples after the last window."""
    return (K - 1) * lag + n + tail


def oracle(Ns, k, lag, n=N_EMB, **kw):
    key = (Ns, k, lag, n, tuple(sorted(kw.items())))
    if key not in _refs:
        _, y = T.synth.sinusoids_np(Ns, k, seed=5)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            ref = O.rpca(O.hankel(y, n, lag), **kw)
        _refs[key] = (y, ref, unhankel_lag(ref.A, lag, Ns))
    return _refs[key]


def solve(y, lag, env, monkeypatch, n=N_EMB, **kw):
    """lowrankfilter under `env`; also returns the per-phase spans (profiling on for the call)."""
    for k_, v_ in env.items():
        monkeypatch.setenv(k_, v_)
    try:
        T.set_profiling(True)
        yf, info = T.lowrankfilter(y, n, lag=lag, return_info=True, **kw)
        prof = T.get_profile()
        T.set_profiling(False)
    finally:
        for k_ in env:
            monkeypatch.delenv(k_)
    return yf, info, prof


def check(yf, info, ref, yo):
    assert info["iters"] == ref.iters, (info["iters"], ref.iters)
    assert np.array_equal(info["hist"][:, 1], ref.hist[:, 1]), (info["hist"][:, 1], ref.hist[:, 1])
    assert info["sv"] == ref.sv
    err = relF(yf, yo)
    assert err < TOL, err


def one_pass_only(prof):
    return prof["fused"][1] > 0 and prof["epilogue"][1] == 0


@pytest.mark.parametrize("lag", [2, 3, 7])
def test_default_route(lag, monkeypatch):
    """K = 20 000 Hankel rows (even): the two-kernel pipeline with the factored unhankel of that lag."""
    Ns = signal_len(20_000, lag)
    y, ref, yo = oracle(Ns, 5, lag, tol=1e-3)
    yf, info, _ = solve(y, lag, {}, monkeypatch)
    check(yf, info, ref, yo)


def test_even_row_count_pipelines_agree(monkeypatch):
    """lag 2, K = 20 000: the two-kernel pipeline, the one-pass kernel, and the one-pass kernel with Y in place."""
    lag = 2
    y, ref, yo = oracle(signal_len(20_000, lag), 6, lag, tol=1e-3)
    out = []
    for env in ({"TLSQ_FUSED": "0"}, {"TLSQ_FUSED": "1"}, {"TLSQ_FUSED": "1", "TLSQ_INPLACE_Y": "1"}):
        yf, info, prof = solve(y, lag, env, monkeypatch)
        check(yf, info, ref, yo)
        if env["TLSQ_FUSED"] == "1":
            assert one_pass_only(prof), prof
        out.append(yf)
    assert relF(out[1], out[0]) < 1e-12 and relF(out[2], out[0]) < 1e-12 and relF(out[2], out[1]) < 1e-12


def test_odd_row_count_takes_the_one_pass_kernel(monkeypatch):
    """lag 2, K = 20 001 (odd): no TMA SYRK on the padded iterate, so the default route is the one-pass kernel."""
    lag = 2
    y, ref, yo = oracle(signal_len(20_001, lag), 6, lag, tol=1e-3)
    yf, info, prof = solve(y, lag, {}, monkeypatch)
    check(yf, info, ref, yo)
    assert one_pass_only(prof), prof


@pytest.mark.parametrize("k,lag", [(13, 2), (15, 2), (13, 3)])
def test_rank_above_16_with_a_lag(k, lag, monkeypatch):
    """Rank estimates 17-32 (rank pads 24 and 32, Hankel form only) with a lag, odd row count: one-pass kernel."""
    y, ref, yo = oracle(signal_len(20_001, lag), k, lag, tol=1e-3)
    assert 16 < ref.hist[:, 1].max() <= 32
    yf, info, prof = solve(y, lag, {}, monkeypatch)
    check(yf, info, ref, yo)
    assert one_pass_only(prof), prof


def test_inplace_dual_without_prediction_repeats_the_solve(monkeypatch):
    """Y in place with the Z prediction off (the repeated-solve path), lag 2: same stopping iteration as the oracle."""
    lag = 2
    y, ref, yo = oracle(signal_len(20_000, lag), 6, lag, tol=1e-3)
    yf1, info1, _ = solve(y, lag, {"TLSQ_FUSED": "1", "TLSQ_INPLACE_Y": "1"}, monkeypatch)
    yf2, info2, prof2 = solve(y, lag, {"TLSQ_FUSED": "1", "TLSQ_INPLACE_Y": "1", "TLSQ_NO_PREDICT_Z": "1"}, monkeypatch)
    check(yf1, info1, ref, yo)
    check(yf2, info2, ref, yo)
    assert relF(yf1, yf2) < 1e-12
    assert prof2["fused"][1] > 0


@pytest.mark.parametrize("lag,tail", [(3, 2), (7, 5)])
def test_uncovered_tail_is_zero(lag, tail, monkeypatch):
    """(Ns - n) % lag != 0: the last `tail` samples lie in no window and come back as exactly 0 (y ./= max.(counts, 1))."""
    Ns = signal_len(20_001, lag, tail=tail)
    assert (Ns - N_EMB) % lag == tail
    y, ref, yo = oracle(Ns, 6, lag, tol=1e-3)
    yf, info, _ = solve(y, lag, {}, monkeypatch)
    check(yf, info, ref, yo)
    assert np.all(yf[Ns - tail:] == 0.0) and np.all(yf[Ns - tail - 1] != 0.0)


@pytest.mark.parametrize("K", [8191, 8192])
def test_lag_equal_to_the_window(K, monkeypatch):
    """lag = n: non-overlapping windows, every sample in exactly one row.  The rank estimate of the stopping iteration
    climbs past 32 here.  With an odd row count the solve starts on the one-pass kernel, which then has no pipeline to
    hand over to, and it is repeated on the materialising route with its dense iterate.  Even K: the two-kernel
    pipeline."""
    lag = N_EMB
    y, ref, yo = oracle(signal_len(K, lag), 5, lag, tol=1e-3)
    yf, info, prof = solve(y, lag, {}, monkeypatch)
    check(yf, info, ref, yo)
    if K % 2:
        assert prof["fused"][1] > 0, prof
        if ref.hist[:, 1].max() > 32:
            assert prof["epilogue"][1] > 0, prof


def test_large_embedding_with_a_lag(monkeypatch):
    """n = 600, lag 3, K = 6000 (even): the large-n two-kernel pipeline and the factored unhankel of that lag."""
    n, lag = 600, 3
    y, ref, yo = oracle(signal_len(6000, lag, n=n), 6, lag, n=n, tol=1e-3)
    yf, info, prof = solve(y, lag, {}, monkeypatch, n=n)
    check(yf, info, ref, yo)
    assert prof["fused"][1] == 0 and prof["epilogue"][1] > 0


def test_large_embedding_rank_above_32_continues_on_the_dense_path(monkeypatch):
    """n = 600, lag 2, K = 6000 (even) on twenty sinusoids: the rank estimate outgrows the 32-column factors at n > 512,
    and the solve continues on the dense device path (materialised embedding) as it did before the factored route
    took lag > 1."""
    n, lag = 600, 2
    y, ref, yo = oracle(signal_len(6000, lag, n=n), 20, lag, n=n, tol=1e-3)
    assert ref.hist[:, 1].max() > 32
    yf, info, _ = solve(y, lag, {}, monkeypatch, n=n)
    check(yf, info, ref, yo)


def test_repeated_solves_on_the_one_pass_kernel_are_bit_identical(monkeypatch):
    """Four lag-2 solves (odd K: one-pass kernel, rank pad 24 or 32): the same filtered signal and rank history, bit for
    bit."""
    lag = 2
    _, y = T.synth.sinusoids_np(signal_len(20_001, lag), 13, seed=5)
    runs = [solve(y, lag, {}, monkeypatch) for _ in range(4)]
    yf0, info0, prof0 = runs[0]
    assert one_pass_only(prof0) and info0["hist"][:, 1].max() > 16
    for yf, info, _ in runs[1:]:
        assert np.array_equal(info["hist"][:, :2], info0["hist"][:, :2])
        assert np.array_equal(yf, yf0)


def test_multi_gpu_sharded_with_a_lag():
    """2-rank sharded lowrankfilter with lag 2 and 3, one shard with an odd row count (tools/mgpu_lag_check.py under
    torch.distributed.run).  Skipped with fewer than two GPUs."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29577",
                          os.path.join(ROOT, "tools", "mgpu_lag_check.py")], capture_output=True, text=True,
                         env=env, timeout=1500)
    sys.stdout.write(out.stdout[-4000:])
    assert out.returncode == 0, out.stderr[-2000:]
    assert "MGPU_LAG PASS" in out.stdout
