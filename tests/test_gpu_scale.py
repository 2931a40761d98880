"""GPU parity at BASELINE scale and for the host-side overlap logic (run with -m gpu on the B200 box).

* tests/golden/oracle_scale.npz (made by tests/golden/make_golden_scale.py): the CPU oracle run on problems shaped like
  BASELINE.json's configurations -- C4 at 100 000 x 256 to convergence, C2 at its full 100 000 x 512 for 6 iterations,
  C3 at 200 000 x 256, lowrankfilter n = 256 on 40 000 samples.  The inputs are regenerated from the seeded generators;
  the fixture holds every 1497-th row of A-hat / E-hat plus column sums, Frobenius norms and nnz of the full matrices.
* the speculative rank guess / run-ahead of solver.cu against the synchronous schedule (bit-identical results);
* the in-place dual variable with the Z prediction switched off (the solve is repeated, same stopping iteration);
* multi-GPU parity (tools/mgpu_check.py under torchrun) when the box has at least two GPUs.
"""
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


def relF(a, b):
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


@pytest.fixture(scope="module")
def scale():
    return np.load(os.path.join(HERE, "golden", "oracle_scale.npz"))


def check_rpca_case(g, name, A, E, s, sv, info, fixed):
    st = int(g["stride"])
    assert relF(A[::st], g[f"{name}_A_rows"]) < TOL, relF(A[::st], g[f"{name}_A_rows"])
    assert relF(E[::st], g[f"{name}_E_rows"]) < TOL
    # support of the stored rows: identical outside a 1e-12 band around the threshold
    Er, Eo = E[::st], g[f"{name}_E_rows"]
    diff = (Er != 0) != (Eo != 0)
    near = np.minimum(np.abs(Er), np.abs(Eo)) <= 1e-12 * float(g[f"{name}_Dmax"])
    assert int(np.sum(diff & ~near)) == 0
    # whole-matrix digests: the rows that are not stored are pinned by column sums and norms
    assert relF(A.sum(axis=0), g[f"{name}_A_colsum"]) < TOL
    assert relF(E.sum(axis=0), g[f"{name}_E_colsum"]) < TOL
    assert abs(np.linalg.norm(A) / float(g[f"{name}_A_fro"]) - 1.0) < TOL
    assert abs(np.linalg.norm(E) / float(g[f"{name}_E_fro"]) - 1.0) < TOL
    assert abs(int(np.count_nonzero(E)) - int(g[f"{name}_E_nnz"])) <= 2          # entries exactly at the threshold
    assert np.array_equal(info["hist"][:, 1], g[f"{name}_hist"][:, 1])           # identical rank history
    assert sv == int(g[f"{name}_sv"])
    if not fixed:
        assert info["converged"] and info["iters"] == int(g[f"{name}_iters"])    # same stopping iteration (:225-231)
    S = g[f"{name}_S"]
    assert np.allclose(s.S, S, rtol=0, atol=1e-12 * S[0]), np.abs(s.S - S).max() / S[0]


def test_c4_shaped_100k_x_256_to_convergence(scale, monkeypatch):
    D = T.synth.lowrank_sparse_np(100_000, 256, 10, 0.05, seed=4, nonneg=True)
    for env in ({"TLSQ_FUSED": "0"}, {"TLSQ_FUSED": "1"}):
        for k_, v_ in env.items():
            monkeypatch.setenv(k_, v_)
        A, E, s, sv, info = T.rpca(D, nonnegA=True, return_info=True)
        for k_ in env:
            monkeypatch.delenv(k_)
        check_rpca_case(scale, "c4s", A, E, s, sv, info, fixed=False)
        assert (A >= 0).all()


def test_c2_full_size_100k_x_512_six_iterations(scale):
    D = T.synth.lowrank_sparse_np(100_000, 512, 10, 0.05, seed=2)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        A, E, s, sv, info = T.rpca(D, iters=6, tol=0.0, return_info=True)
    check_rpca_case(scale, "c2s", A, E, s, sv, info, fixed=True)


def test_c3_shaped_rpca_ga_200k_x_256(scale):
    X, q0 = T.synth.ga_data_np(200_000, 256, 10, seed=3)
    Q, info = T.rpca_ga(X, 3, q0=q0[:, :3], return_info=True)
    st = int(scale["stride"])
    Qo = scale["c3s_Q_rows"]
    sgn = np.sign(np.sum(Q[::st] * Qo, axis=0))
    assert np.abs(Q[::st] * sgn - Qo).max() < TOL
    assert np.allclose(np.abs(Q.sum(axis=0)), scale["c3s_Q_colsum_abs"], rtol=0, atol=1e-7)
    assert info["iters"] == [int(v) for v in scale["c3s_iters"]]


def test_lowrankfilter_n256_40k_samples(scale, monkeypatch):
    y, yn = T.synth.sinusoid_np(40_000, seed=5)
    yo = scale["lrfs_yf"]
    for env in ({"TLSQ_FUSED": "0"}, {"TLSQ_FUSED": "1"}, {"TLSQ_FUSED": "1", "TLSQ_INPLACE_Y": "1"}):
        for k_, v_ in env.items():
            monkeypatch.setenv(k_, v_)
        yf = T.lowrankfilter(yn, 256)
        for k_ in env:
            monkeypatch.delenv(k_)
        assert relF(yf, yo) < TOL, (env, relF(yf, yo))


def test_inplace_dual_without_prediction_repeats_the_solve(monkeypatch):
    """solver.cu rpca_core: with Y updated in place an undecided Frobenius bracket that was not predicted cannot be
    resolved after the fact; the solve is repeated with the two-phase iteration forced -- same stopping iteration."""
    y, yn = T.synth.sinusoid_np(12255, seed=2)                             # noise-free: the rank stays at 6
    kw = dict(tol=1e-6)                                                    # the residual crosses the 16x-wide bracket slowly
    monkeypatch.setenv("TLSQ_FUSED", "1")
    yf, info = T.lowrankfilter(yn, 256, return_info=True, **kw)
    n0 = T.launch_count()
    monkeypatch.setenv("TLSQ_INPLACE_Y", "1")
    yf1, info1 = T.lowrankfilter(yn, 256, return_info=True, **kw)          # predicted two-phase iterations
    n1 = T.launch_count()
    monkeypatch.setenv("TLSQ_NO_PREDICT_Z", "1")
    yf2, info2 = T.lowrankfilter(yn, 256, return_info=True, **kw)          # prediction off: the solve is repeated
    n2 = T.launch_count()
    for k_ in ("TLSQ_INPLACE_Y", "TLSQ_NO_PREDICT_Z", "TLSQ_FUSED"):
        monkeypatch.delenv(k_)
    H = O.hankel(yn, 256)
    ref = O.rpca(H, tol=1e-6)
    assert info["iters"] == ref.iters and info1["iters"] == ref.iters and info2["iters"] == ref.iters
    assert relF(yf2, O.unhankel_fast(ref.A)) < TOL and relF(yf, yf2) < 1e-12 and relF(yf1, yf2) < 1e-12
    assert n2 - n1 > 1.3 * (n1 - n0)                                        # it really ran (most of) the solve twice


def test_runahead_schedule_is_bit_identical_to_the_synchronous_one(monkeypatch):
    """Two-kernel pipeline: speculative rank guess + run-ahead Gram/eigen step (solver.cu) change the host schedule only."""
    for (M, N, r, kw) in [(20000, 256, 10, {"nonnegA": True}), (12000, 128, 20, {}), (30000, 192, 4, {})]:
        D = T.synth.lowrank_sparse_np(M, N, r, 0.05, seed=4, nonneg=bool(kw.get("nonnegA")))
        monkeypatch.setenv("TLSQ_FUSED", "0")
        A1, E1, s1, sv1, i1 = T.rpca(D, return_info=True, **kw)
        monkeypatch.setenv("TLSQ_NO_RUNAHEAD", "1")
        A2, E2, s2, sv2, i2 = T.rpca(D, return_info=True, **kw)
        monkeypatch.delenv("TLSQ_NO_RUNAHEAD")
        monkeypatch.delenv("TLSQ_FUSED")
        assert i1["iters"] == i2["iters"] and sv1 == sv2 and np.array_equal(i1["hist"][:, 1], i2["hist"][:, 1])
        assert relF(A1, A2) < 1e-13 and relF(E1, E2) < 1e-13 and np.array_equal(E1 != 0, E2 != 0)
        assert np.allclose(s1.S, s2.S, rtol=0, atol=1e-13 * s2.S[0])


def test_factored_unhankel_with_large_rank_and_n_above_256():
    """ADVICE r1: n in (256, 512] with a final rank estimate of 23..32 used to fail at finalisation (shared memory of
    the factored unhankel)."""
    rng = np.random.default_rng(8)
    Ns, n = 9000, 384
    t = np.arange(Ns)
    y = sum(rng.standard_normal() * np.sin((0.01 + 0.05 * k) * t + rng.uniform(0, 6)) for k in range(14))   # rank 28
    yn = y + 1e2 * (rng.random(Ns) < 0.02)
    yf, info = T.lowrankfilter(yn, n, return_info=True)
    assert 23 <= info["sv"] <= 32, info["sv"]
    assert relF(yf, O.lowrankfilter(yn, n)) < TOL


def test_multi_gpu_parity_two_ranks():
    """Row-sharded solves on 2 GPUs against the oracle (tools/mgpu_check.py: both n = 256 pipelines, rpca_ga,
    lowrankfilter incl. the sharded implicit Hankel matrix).  Skipped on single-GPU boxes."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29571",
                          os.path.join(ROOT, "tools", "mgpu_check.py")], capture_output=True, text=True, env=env,
                         timeout=1500)
    sys.stdout.write(out.stdout[-4000:])
    assert out.returncode == 0, out.stderr[-2000:]
    assert "MGPU_CHECK PASS" in out.stdout


def test_rtls_parity_5000_x_8():
    """rtls = rpca([A y]; nukeA=false) then tls! on the TRAILING column of the returned s.V
    (src/TotalLeastSquares.jl:65-69, 152-156): needs the tail of the SVD to LAPACK accuracy."""
    rng = np.random.default_rng(12)
    x = rng.standard_normal(7)
    A = rng.standard_normal((5000, 7))
    y = A @ x
    An = A + 0.01 * rng.standard_normal(A.shape)
    yn = y + 0.01 * rng.standard_normal(5000)
    An[rng.random(A.shape) < 0.02] += 10.0
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        xr = T.rtls(An, yn).ravel()
        ref = O.rpca(np.hstack([An, yn.reshape(-1, 1)]), nukeA=False)
    V = ref.s.Vt.T
    xo = (-np.linalg.solve(V[7:, 7:].T, V[:7, 7:].T).T).ravel()
    assert np.allclose(xr, xo, rtol=1e-8, atol=1e-10), np.abs(xr - xo).max()


# ---- large embeddings: min(M, N) > 512 (src/robustPCA.jl:119: lowrankfilter's default n = min(N / 20, 2000)) ------------
@pytest.fixture(scope="module")
def largen():
    return np.load(os.path.join(HERE, "golden", "oracle_largen.npz"))


def test_lowrankfilter_default_embedding_50k_samples(largen):
    """lowrankfilter(y) with the reference's default n = 2000 on 50 000 samples (Hankel 48 001 x 2000, odd row count):
    large-n subspace iteration + certificate, GEMM projection, column-chunked element-wise pass."""
    y, yn = T.synth.sinusoid_np(50_000, seed=6)
    yf, info = T.lowrankfilter(yn, return_info=True)
    assert info["iters"] == int(largen["lrf50k_iters"]) and info["sv"] == int(largen["lrf50k_sv"])
    assert np.array_equal(info["hist"][:, 1], largen["lrf50k_hist"][:, 1])
    assert relF(yf, largen["lrf50k_yf"]) < TOL, relF(yf, largen["lrf50k_yf"])
    assert np.mean((y - yf) ** 2) / np.mean(y ** 2) < 1e-3


def test_rpca_3000_x_1000_with_returned_svd(largen):
    """min(M,N) = 1000: generic Gram (too few rows for the TMA SYRK), full Jacobi out of L2 for the returned spectrum."""
    D = T.synth.lowrank_sparse_np(3000, 1000, 8, 0.05, seed=21)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        A, E, s, sv, info = T.rpca(D, iters=4, tol=0.0, return_info=True)
    st = int(largen["r1000_stride"])
    assert relF(A[::st], largen["r1000_A_rows"]) < TOL and relF(E[::st], largen["r1000_E_rows"]) < TOL
    assert relF(A.sum(axis=0), largen["r1000_A_colsum"]) < TOL and relF(E.sum(axis=0), largen["r1000_E_colsum"]) < TOL
    assert abs(np.linalg.norm(A) / float(largen["r1000_A_fro"]) - 1) < TOL
    assert abs(np.linalg.norm(E) / float(largen["r1000_E_fro"]) - 1) < TOL
    assert np.array_equal(info["hist"][:, 1], largen["r1000_hist"][:, 1])
    S = largen["r1000_S"]
    assert np.allclose(s.S, S, rtol=0, atol=1e-12 * S[0]), np.abs(s.S - S).max() / S[0]
    assert np.abs(s.Vt @ s.Vt.T - np.eye(1000)).max() < 1e-11


def test_rank_above_32_with_n_above_512_takes_the_dense_device_path():
    """512 < min(M,N) with a rank estimate of 40: outside the 32-column factored kernels.  tlsq_rpca_f64 repeats the solve
    on the dense device path (full Jacobi SVT, exact stop test) instead of failing."""
    import torch
    D = T.synth.lowrank_sparse_np(3000, 600, 40, 0.05, seed=7)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        A, E, s, sv, info = T.rpca(D, iters=5, tol=0.0, return_info=True)
        ref = O.rpca(D, iters=5, tol=0.0)
    assert np.array_equal(info["hist"][:, 1], ref.hist[:, 1]) and ref.hist[-1, 1] == 40
    assert relF(A, ref.A) < TOL and relF(E, ref.E) < TOL
    assert np.allclose(info["hist"][:, 2], ref.hist[:, 2], rtol=1e-8)
    assert np.allclose(s.S, ref.s.S, rtol=0, atol=1e-12 * ref.s.S[0])
    with warnings.catch_warnings():                                        # device pointers take the same route
        warnings.simplefilter("ignore")
        Ad, Ed, sd, _ = T.rpca(torch.from_numpy(D).cuda(), iters=5, tol=0.0)
    assert np.array_equal(Ad.cpu().numpy(), A) and np.array_equal(Ed.cpu().numpy(), E)
    assert np.array_equal(sd.S.cpu().numpy(), s.S)


def test_hankel_true_with_n_above_512_takes_the_dense_device_path():
    """hankel=true (soft_hankel! every iteration, src/robustPCA.jl:214-216, 234-236) on a 1801 x 600 Hankel matrix: the
    accelerated hankel=true kernels stop at min(M,N) = 512; host-buffer solves continue on the dense device path."""
    rng = np.random.default_rng(11)
    t = np.arange(2400)
    y = np.sin(0.01 * t) + 0.5 * np.sin(0.037 * t) + 0.05 * rng.standard_normal(2400)
    y[rng.random(2400) < 0.02] += 3.0
    H = O.hankel(y, 600)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        A, E, s, sv, info = T.rpca(H, hankel=True, iters=4, tol=0.0, return_info=True)
        ref = O.rpca(H, hankel=True, iters=4, tol=0.0)
    assert np.array_equal(info["hist"][:, 1], ref.hist[:, 1])
    assert relF(A, ref.A) < TOL and relF(E, ref.E) < TOL


def test_lowrankfilter_default_embedding_with_rank_above_32():
    """lowrankfilter(y) with the default n = 600 on twenty sinusoids + outliers: the rank estimate runs 32, 36, ... 82, past
    the 32-column factors of the implicit-Hankel kernels; the solve continues on the dense device path (materialised
    embedding) and still matches the reference's iteration count, rank history and filtered signal."""
    rng = np.random.default_rng(5)
    Ns = 12000
    t = np.arange(Ns)
    freqs = 0.02 + 0.9 * rng.random(20)
    y0 = sum(np.sin(f * t + rng.random() * 6.28) * (0.5 + rng.random()) for f in freqs)
    y = y0 + 0.05 * rng.standard_normal(Ns)
    y[rng.random(Ns) < 0.01] += 5.0
    yf, info = T.lowrankfilter(y, return_info=True)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ref = O.rpca(O.hankel(y, 600), tol=1e-3)
    assert ref.hist[:, 1].max() > 32
    assert info["iters"] == ref.iters and info["sv"] == ref.sv
    assert np.array_equal(info["hist"][:, 1], ref.hist[:, 1])
    assert relF(yf, O.unhankel_fast(ref.A)) < TOL
    assert np.mean((yf - y0) ** 2) / np.mean(y0 ** 2) < 1e-3


def test_lowrankfilter_default_embedding_16k_samples_live_oracle():
    """n = 800 (default for 16 000 samples), even row count -> TMA SYRK at N = 800; oracle run on the host cores."""
    y, yn = T.synth.sinusoid_np(16_001, seed=9, noise=0.02)
    yf, info = T.lowrankfilter(yn, return_info=True)
    H = O.hankel(yn, 800)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ref = O.rpca(H, tol=1e-3)
    assert info["iters"] == ref.iters and info["sv"] == ref.sv
    assert relF(yf, O.unhankel_fast(ref.A)) < TOL


def test_repeated_solves_are_deterministic():
    """The TMA-staged streaming kernels refill a ring stage behind a CTA barrier; an early refill raced with in-flight
    shared-memory loads and produced sporadically different cost histories.  Same input, same build -> same history."""
    import torch
    D = T.synth.lowrank_sparse_cuda(0, 300_000, 256, torch.device("cuda", 0), 10, 0.05, seed=4, nonneg=True)
    hists = []
    for _ in range(6):
        A, E, s, sv, info = T.rpca(D, nonnegA=True, return_info=True, want_svd=False, exact_cost=True)
        hists.append(info["hist"][:, 2].copy())
    assert len({len(h) for h in hists}) == 1
    H = np.stack(hists)
    assert np.abs(H / np.median(H, axis=0) - 1.0).max() < 1e-9
