"""GPU parity tests (run with -m gpu on the B200 box): the CUDA path, called through the C ABI (host-buffer entry
points via the Python mirror), against the CPU oracle on the same seeded inputs, against the committed golden
vectors, and -- at larger sizes -- through size-independent properties.

Tolerances (BASELINE.json north_star): A-hat, E-hat relative Frobenius error <= 1e-9 at a fixed iteration count;
supp(E-hat) identical outside a 1e-12 band around the threshold; rpca_ga components <= 1e-9 up to sign.
"""
import json
import os
import warnings

import numpy as np
import pytest

import tls_oracle as O
import tlsq_b200 as T

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
TOL = 1e-9
SQRT_EPS = np.sqrt(np.finfo(float).eps)


def relF(a, b):
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


def support_mismatch(E, Eo, ref_scale, band=1e-12):
    """entries whose zero/non-zero status differs, ignoring those within `band` (relative) of the threshold"""
    diff = (E != 0) != (Eo != 0)
    near = np.minimum(np.abs(E), np.abs(Eo)) <= band * ref_scale
    return int(np.sum(diff & ~near))


def fixed_iters(D, iters, **kw):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        A, E, s, sv, info = T.rpca(D, iters=iters, tol=0.0, return_info=True, **kw)
        ref = O.rpca(D, iters=iters, tol=0.0, **kw)
    return A, E, s, sv, info, ref


def test_library_runs_on_gpu():
    assert T.load().tlsq_device_count() >= 1
    n0 = T.launch_count()
    T.rpca(np.random.default_rng(0).random((64, 8)), iters=2, tol=0.0, want_svd=False)
    assert T.launch_count() > n0          # our kernels ran (no fallback exists)


def test_known_answer_5x5():
    """reference test/runtests.jl:143-169"""
    g = json.load(open(os.path.join(HERE, "golden", "rpca_5x5.json")))
    D = np.array(g["D"])
    A, E, s, sv = T.rpca(D, nonnegE=True, nonnegA=True)
    assert np.abs(A - np.array(g["A"])).max() < g["atol"]
    assert np.abs(E - np.array(g["E"])).max() < g["atol"]
    assert np.linalg.norm(D - (A + E)) / np.linalg.norm(D) < SQRT_EPS
    A, E, _, _ = T.rpca(D)
    assert np.linalg.norm(D - (A + E)) / np.linalg.norm(D) < SQRT_EPS


def test_golden_vectors():
    g = np.load(os.path.join(HERE, "golden", "oracle_vectors.npz"))
    warnings.simplefilter("ignore")
    D = g["rpca_D"]
    for name, kw, Dk in [("plain", {}, D), ("nonneg", {"nonnegA": True, "nonnegE": True}, np.abs(D)),
                         ("nonuke", {"nukeA": False}, D)]:
        A, E, s, sv, info = T.rpca(Dk, iters=10, tol=0.0, return_info=True, **kw)
        assert relF(A, g[f"rpca_{name}_A"]) < TOL and relF(E, g[f"rpca_{name}_E"]) < TOL
        assert np.array_equal(info["hist"][:, 1], g[f"rpca_{name}_hist"][:, 1])
        assert np.allclose(s.S, g[f"rpca_{name}_S"], rtol=0, atol=1e-12 * g[f"rpca_{name}_S"][0])
    A, E, _, _ = T.rpca(g["rpca_wide_D"], iters=8, tol=0.0)
    assert relF(A, g["rpca_wide_A"]) < TOL and relF(E, g["rpca_wide_E"]) < TOL
    A, E, s, sv, info = T.rpca(D, return_info=True)
    assert info["iters"] == int(g["rpca_conv_iters"]) and sv == int(g["rpca_conv_sv"])
    assert relF(A, g["rpca_conv_A"]) < TOL and relF(E, g["rpca_conv_E"]) < TOL
    Q = T.rpca_ga(g["ga_X"], 3, q0=g["ga_q0"])
    sgn = np.sign(np.sum(Q * g["ga_Q"], axis=0))
    assert np.abs(Q * sgn - g["ga_Q"]).max() < TOL
    assert relF(T.lowrankfilter(g["lrf_y"], 10), g["lrf_yf"]) < TOL
    assert relF(T.lowrankfilter(g["lrf_y"], 10, lag=2), g["lrf_yf_lag2"]) < TOL


@pytest.mark.parametrize("M,N,r,kw,its", [
    (2000, 64, 5, {}, 12),                                   # generic kernels (n <= 64)
    (3000, 40, 3, {"nonnegA": True}, 12),
    (496, 5, 2, {}, 20),                                     # README shape (C1)
    (5001, 200, 5, {"nukeA": False}, 9),                     # odd leading dimension: no TMA, generic Gram
    (8192, 256, 10, {}, 14),                                 # n = 256: fused one-pass kernel + fast eigen path
    (20002, 256, 10, {"nonnegA": True, "nonnegE": True}, 12),  # fused, row count not a multiple of the 32-row tile
    (6000, 256, 3, {"nukeA": False}, 8),                     # fused, nukeA = false
    (8000, 256, 20, {}, 12),                                 # fused until svp > 16, then the streaming pipeline
    (8192, 192, 10, {}, 14),                                 # TMA SYRK + fast eigen path + streaming epilogue
    (10000, 128, 6, {"nonnegA": True, "nonnegE": True}, 14),
    (3000, 96, 40, {}, 10),                                  # svp > 32: fused tile epilogue, full Jacobi
    (6000, 512, 8, {}, 5),                                   # n = 512: cooperative-grid Jacobi
    (9000, 512, 28, {}, 7),                                  # n = 512, rank 25..32: column-chunked streaming epilogue
    (300, 500, 4, {}, 8),                                    # wide: solved on the transpose
    (33, 7, 2, {}, 6), (1, 5, 1, {}, 3), (7, 1, 1, {}, 3),   # ragged / degenerate
])
def test_rpca_parity_fixed_iterations(M, N, r, kw, its, monkeypatch):
    D = T.synth.lowrank_sparse_np(M, N, r, 0.05, seed=M + N, nonneg=bool(kw.get("nonnegA")))
    # n = 256: two-kernel pipeline and the one-pass kernel
    pipelines = [{}]
    if N == 256 and M >= 4096:
        pipelines = [{"TLSQ_FUSED": "0"}, {"TLSQ_FUSED": "1"}]
    ref = None
    for env in pipelines:
        for k_, v_ in env.items():
            monkeypatch.setenv(k_, v_)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            A, E, s, sv, info = T.rpca(D, iters=its, tol=0.0, return_info=True, **kw)
            if ref is None:
                ref = O.rpca(D, iters=its, tol=0.0, **kw)
        for k_ in env:
            monkeypatch.delenv(k_)
        assert relF(A, ref.A) < TOL, (env, relF(A, ref.A))
        assert relF(E, ref.E) < TOL or np.linalg.norm(ref.E) == 0
        assert support_mismatch(E, ref.E, np.abs(D).max()) == 0
        assert np.array_equal(info["hist"][:, 1], ref.hist[:, 1])      # identical rank history (full-SVD semantics)
        assert sv == ref.sv
        d = min(M, N)
        assert s.U.shape == (M, d) and s.S.shape == (d,) and s.Vt.shape == (d, N)
        # singular values of the last SVT input to LAPACK accuracy (the Gram route alone gives eps*S[0]^2/S[i]; the
        # CholeskyQR2-style refinement in solver.cu restores eps*S[0])
        assert np.allclose(s.S, ref.s.S, rtol=0, atol=1e-12 * ref.s.S[0]), np.abs(s.S - ref.s.S).max() / ref.s.S[0]
        # ... and the factors are orthonormal
        assert np.abs(s.Vt @ s.Vt.T - np.eye(d)).max() < 1e-12
        if M >= N and ref.s.S[-1] > 1e-6 * ref.s.S[0]:
            assert np.abs(s.U.T @ s.U - np.eye(d)).max() < 1e-8
        # the returned SVD reproduces the last SVT input like the reference's does
        Wg, Wo = (s.U * s.S) @ s.Vt, (ref.s.U * ref.s.S) @ ref.s.Vt
        assert relF(Wg, Wo) < 1e-7


@pytest.mark.parametrize("M,N,r,kw", [(2000, 64, 5, {}), (20000, 256, 10, {"nonnegA": True}), (12000, 128, 20, {})])
def test_rpca_converges_like_the_reference(M, N, r, kw, monkeypatch):
    D = T.synth.lowrank_sparse_np(M, N, r, 0.05, seed=4, nonneg=bool(kw.get("nonnegA")))
    ref = O.rpca(D, **kw)
    for fused in (("0", "1") if N == 256 else ("0",)):
        monkeypatch.setenv("TLSQ_FUSED", fused)
        A, E, s, sv, info = T.rpca(D, return_info=True, **kw)
        assert info["converged"] and info["iters"] == ref.iters
        assert relF(A, ref.A) < TOL and relF(E, ref.E) < TOL
        assert np.linalg.norm(D - A - E) / np.linalg.norm(D) < SQRT_EPS
        # exact cost evaluation (verbose path) reproduces the reference's cost sequence
        _, _, _, _, info2 = T.rpca(D, return_info=True, exact_cost=True, want_svd=False, **kw)
        assert info2["iters"] == ref.iters
        assert np.allclose(info2["hist"][:, 2], ref.hist[:, 2], rtol=1e-6)
    monkeypatch.delenv("TLSQ_FUSED")


@pytest.mark.parametrize("Ns,L,kw", [(1000, 50, {"nukeA": False}), (600, 24, {}), (4500, 200, {"nukeA": False})])
def test_rpca_hankel_true_matches_the_oracle(Ns, L, kw):
    """hankel=true: soft_hankel! of the iterate every iteration and of E at the end (src/robustPCA.jl:9-21, 214-216,
    234-236; reference tests test/runtests.jl:309-348)."""
    rng = np.random.default_rng(Ns + L)
    H = O.hankel(rng.standard_normal(Ns), L)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        A, E, s, sv, info = T.rpca(H, hankel=True, iters=15, tol=0.0, return_info=True, **kw)
        ref = O.rpca(H, hankel=True, iters=15, tol=0.0, **kw)
    assert relF(A, ref.A) < TOL and relF(E, ref.E) < TOL
    assert np.array_equal(info["hist"][:, 1], ref.hist[:, 1])
    A2, E2, _, _, info2 = T.rpca(H, hankel=True, return_info=True, **kw)
    ref2 = O.rpca(H, hankel=True, **kw)
    assert info2["iters"] == ref2.iters and relF(A2, ref2.A) < TOL
    if kw.get("nukeA") is False:                                             # test/runtests.jl:331-332 (nukeA=false)
        assert O.ishankel(A2) and O.ishankel(E2)


def test_rtls_beats_tls_on_outliers():
    """test/runtests.jl:203-235 (statistical, reduced): rtls = rpca([A y]; nukeA=false) + tls! on the returned SVD."""
    rng = np.random.default_rng(3)
    wins = 0
    for _ in range(20):
        x = rng.standard_normal(3)
        A = rng.standard_normal((50, 3))
        y = A @ x
        An = A + 0.01 * rng.standard_normal(A.shape)
        yn = y + 0.01 * rng.standard_normal(50)
        An[rng.random(A.shape) < 0.05] += 10.0 * rng.standard_normal()
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            xr = T.rtls(An, yn).ravel()
            xo = O_rtls(An, yn).ravel()
        assert np.allclose(xr, xo, rtol=1e-6, atol=1e-8)
        xt = T.tls(An, yn).ravel()
        wins += np.linalg.norm(xr - x) < np.linalg.norm(xt - x)
    assert wins >= 14


def O_rtls(A, y):
    ref = O.rpca(np.hstack([A, y.reshape(-1, 1)]), nukeA=False)
    V = ref.s.Vt.T
    n = A.shape[1]
    return -np.linalg.solve(V[n:, n:].T, V[:n, n:].T).T


def test_max_iterations_warning_and_outputs():
    D = T.synth.lowrank_sparse_np(500, 20, 3, 0.05, seed=1)
    with pytest.warns(UserWarning, match="Maximum number of iterations"):
        A, E, s, sv = T.rpca(D, iters=3)
    assert A.shape == D.shape and A.flags.f_contiguous


def test_torch_device_path_matches_host_path():
    import torch
    D = T.synth.lowrank_sparse_np(9000, 256, 8, 0.05, seed=5)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        A, E, s, sv = T.rpca(D, iters=8, tol=0.0)
        Dd = torch.from_numpy(np.ascontiguousarray(D.T)).cuda().t()
        Ad, Ed, sd, svd_ = T.rpca(Dd, iters=8, tol=0.0)
    assert Ad.is_cuda and svd_ == sv
    assert np.array_equal(Ad.cpu().numpy(), A) and np.array_equal(Ed.cpu().numpy(), E)    # same kernels, same bits
    # a row-major tensor is accepted too (one transposing copy)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        Ar, _, _, _ = T.rpca(torch.from_numpy(D).cuda(), iters=8, tol=0.0, want_svd=False)
    assert np.array_equal(Ar.cpu().numpy(), A)


def test_hankel_unhankel_exact():
    """reference test/runtests.jl:293-294, 356-371"""
    x = np.arange(1.0, 21.0)
    assert np.array_equal(T.hankel(x, 2), O.hankel(x, 2))
    assert np.array_equal(T.hankel(x, 3, 2), O.hankel(x, 3, 2))
    Tn = 1000
    y = np.sin(0.1 * np.arange(1, Tn + 1))
    assert np.array_equal(T.unhankel(T.hankel(y, 2)), y)
    assert np.array_equal(T.unhankel(T.hankel(y, 2, 2), 2, Tn), y)
    assert np.allclose(T.unhankel(T.hankel(y, 5, 2), 2, Tn)[:-1], y[:-1])
    A = np.random.default_rng(0).standard_normal((37, 6))
    assert np.allclose(T.unhankel(A), O.unhankel(A), rtol=0, atol=1e-14)


def test_lowrankfilter_parity_and_statistics():
    """README.md:85-92 / test/runtests.jl:172-185, 378-380"""
    rng = np.random.default_rng(4)
    res = []
    for i in range(20):
        N = 500
        y = np.sin(0.1 * np.arange(1, N + 1)) + 0.1 * rng.standard_normal(N)
        yn = y + (rng.random(N) < 0.1) * 1e2
        yf, info = T.lowrankfilter(yn, 40, return_info=True)
        if i < 3:
            assert relF(yf, O.lowrankfilter(yn, 40)) < TOL
        res.append(np.mean((y - yf) ** 2) / np.mean(y ** 2))
    assert np.mean(res) < 0.025
    Tn = 1000
    qn = lambda x: x / np.quantile(np.abs(x), 0.9)
    y = qn(np.sin(0.1 * np.arange(1, Tn + 1)))
    n = 20 * rng.standard_normal(Tn) * (rng.random(Tn) < 0.01) + 0.1 * rng.standard_normal(Tn)
    yf = qn(T.lowrankfilter(y + n))
    assert np.mean((y - yf) ** 2) / np.mean(n ** 2) < 0.001
    # implicit Hankel == rpca on the materialised embedding
    y, yn = T.synth.sinusoid_np(3000, seed=2, noise=0.05)
    yf = T.lowrankfilter(yn, 100)
    H = O.hankel(yn, 100)
    A, _, _, _ = T.rpca(H, tol=1e-3, want_svd=False)
    assert relF(yf, O.unhankel_fast(A)) < TOL
    # lag > 1
    assert relF(T.lowrankfilter(yn[:600], 30, lag=3), O.lowrankfilter(yn[:600], 30, lag=3)) < TOL


def test_fused_pipeline_equals_two_kernel_pipeline(monkeypatch):
    """n = 256: the one-pass cluster kernel (fused.cu) against the streaming epilogue + SYRK pipeline it replaces, and
    the implicit-Hankel / in-place-Y / factored-unhankel variants of lowrankfilter against the oracle."""
    D = T.synth.lowrank_sparse_np(16384, 256, 7, 0.05, seed=9)
    monkeypatch.setenv("TLSQ_FUSED", "1")
    A1, E1, s1, sv1, i1 = T.rpca(D, return_info=True)
    monkeypatch.setenv("TLSQ_FUSED", "0")
    A2, E2, s2, sv2, i2 = T.rpca(D, return_info=True)
    monkeypatch.setenv("TLSQ_FUSED", "1")
    assert i1["iters"] == i2["iters"] and sv1 == sv2
    assert relF(A1, A2) < 1e-12 and relF(E1, E2) < 1e-12 and np.array_equal(E1 != 0, E2 != 0)
    assert np.allclose(s1.S, s2.S, rtol=0, atol=1e-12 * s2.S[0])
    y, yn = T.synth.sinusoid_np(12255, seed=2, noise=0.05)                # K = 12000 Hankel rows x 256
    yo = O.lowrankfilter(yn, 256)
    yf, info = T.lowrankfilter(yn, 256, return_info=True)
    assert relF(yf, yo) < TOL
    monkeypatch.setenv("TLSQ_INPLACE_Y", "1")                             # dual variable updated in place
    yf2, info2 = T.lowrankfilter(yn, 256, return_info=True)
    monkeypatch.delenv("TLSQ_INPLACE_Y")
    assert relF(yf2, yo) < TOL and info2["iters"] == info["iters"]
    monkeypatch.delenv("TLSQ_FUSED")
    yf3 = T.lowrankfilter(yn[:-1], 256)                                   # odd row count: two-kernel pipeline
    assert relF(yf3, O.lowrankfilter(yn[:-1], 256)) < TOL


def test_multichannel_and_ssa_forms():
    """test/runtests.jl:361-376 (exact round trips incl. lag 2 and two channels), :401-405 (sv=2 plain SSA) and
    :408-439 (multi-channel lowrankfilter) against the oracle and the reference's statistical bounds."""
    rng = np.random.default_rng(11)
    Tn = 1000
    t = np.arange(1, Tn + 1)
    qn = lambda x: x / np.quantile(np.abs(x), 0.9)
    y = qn(np.sin(0.1 * t))
    assert np.array_equal(T.unhankel(T.hankel(y, 2)), y)
    assert np.array_equal(T.unhankel(T.hankel(y, 2, 2), 2, Tn), y)
    yh = T.unhankel(T.hankel(y, 5, 2), 2, Tn)
    assert np.allclose(yh[:-1], y[:-1])
    Y2 = np.column_stack([y, rng.standard_normal(Tn)])
    H = T.hankel(Y2, 5, 2)
    assert np.array_equal(H, O.hankel(Y2, 5, 2))
    yh = T.unhankel(H, 2, Tn, 2)
    assert np.allclose(yh[:-1], Y2[:-1]) and np.allclose(yh, O.unhankel(H, 2, Tn, 2), rtol=0, atol=1e-14)
    # plain SSA branch
    noise = rng.standard_normal(Tn)
    yf = T.lowrankfilter(y + noise, sv=2)
    assert relF(yf, O.lowrankfilter(y + noise, sv=2)) < TOL
    assert np.mean((y - qn(yf)) ** 2) / np.mean(noise ** 2) < 0.05
    yf_w = T.lowrankfilter((y + noise)[:90], 40, sv=3)                      # K = 51 < n = 40?  no: wide when K < n D
    assert relF(yf_w, O.lowrankfilter((y + noise)[:90], 40, sv=3)) < TOL
    # multi-channel lowrankfilter
    y1, y2 = np.sin(0.1 * t), np.sin(0.3 * t)
    Y = np.column_stack([y1, y2 + 0.5 * y1])
    Yn = Y + 0.1 * rng.standard_normal(Y.shape) + (rng.random(Y.shape) < 0.01) * 5 * rng.standard_normal(Y.shape)
    Yf = T.lowrankfilter(Yn, 20)
    assert Yf.shape == Y.shape and relF(Yf, O.lowrankfilter(Yn, 20)) < TOL
    assert np.mean((Y - Yf) ** 2) / np.mean((Y - Yn) ** 2) < 0.05
    yf1 = T.lowrankfilter(Yn[:, 0].copy(), 20)
    assert np.mean((y1 - yf1) ** 2) / np.mean((y1 - Yf[:, 0]) ** 2) > 1.02   # joint filtering helps (:420-422)
    assert relF(T.lowrankfilter(Yn, 12, lag=2, sv=4), O.lowrankfilter(Yn, 12, lag=2, sv=4)) < TOL


@pytest.mark.parametrize("d,N,r", [(10, 40, 3), (40, 10, 5), (1000, 256, 4), (5000, 300, 3), (777, 1000, 2)])
def test_rpca_ga_parity(d, N, r):
    X, q0 = T.synth.ga_data_np(d, N, min(d, N, 10), seed=d + N)
    Q, info = T.rpca_ga(X, r, q0=q0[:, :r], return_info=True)
    Qo, its = O.rpca_ga(X, r, q0=q0[:, :r], exact_order=False, return_iters=True)
    sgn = np.sign(np.sum(Q * Qo, axis=0))
    assert np.abs(Q * sgn - Qo).max() < TOL
    assert info["iters"] == its
    assert np.linalg.norm(Q.T @ Q - np.eye(r)) < SQRT_EPS                 # test/runtests.jl:453


@pytest.mark.parametrize("d,N,r", [(10, 1000, 3), (3000, 256, 3), (517, 100, 2), (40, 3000, 2)])
def test_rpca_ga_robust_averages(d, N, r):
    """rpca_ga(...; μ = entrywise_trimmed_mean / entrywise_median) (src/robustPCA.jl:323-357, test/runtests.jl:491-523):
    per-row sorts on the GPU against the oracle restatement, same start vectors."""
    rng = np.random.default_rng(d + N)
    U0, S0, Vt0 = np.linalg.svd(rng.standard_normal((d, N)), full_matrices=False)
    A = (U0[:, :r] * S0[:r]) @ Vt0[:r] + 1e-3 * rng.standard_normal((d, N))
    A += 1000.0 * rng.standard_normal((d, N)) * (rng.random((d, N)) < 0.01)
    A = np.asfortranarray(A)
    q0 = np.asfortranarray(rng.standard_normal((d, r)))
    for tag, omu in ((T.entrywise_trimmed_mean, O.entrywise_trimmed_mean), (T.entrywise_median, O.entrywise_median)):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            Q, info = T.rpca_ga(A, r, mu=tag, q0=q0, iters=30, return_info=True)
            Qo, its = O.rpca_ga(A, r, q0=q0, mu=omu, exact_order=False, iters=30, return_iters=True)
        sgn = np.sign(np.sum(Q * Qo, axis=0))
        assert info["iters"] == its
        assert np.abs(Q * sgn - Qo).max() < 1e-8, (tag.__name__, np.abs(Q * sgn - Qo).max())


def test_rpca_ga_orthonormal_reference_cases():
    """test/runtests.jl:447-464 (subset), start vectors drawn by the host mirror like the reference's randn(d)"""
    rng = np.random.default_rng(1)
    np.random.seed(1)
    for shape in [(10, 40), (40, 10)]:
        for r in (1, 4, 10):
            for eps in (1e-8, 1e-3, 1.0):
                U, S, Vt = np.linalg.svd(rng.standard_normal(shape), full_matrices=False)
                A = (U[:, :r] * (10.0 * np.arange(1, r + 1))) @ Vt[:r] + eps * rng.standard_normal(shape)
                Q = T.rpca_ga(A, r)
                assert np.linalg.norm(Q.T @ Q - np.eye(r)) < SQRT_EPS


def test_large_problem_properties():
    """BASELINE-sized columns (n = 256), 200k rows: size-independent properties instead of an oracle run."""
    import torch
    D = T.synth.lowrank_sparse_cuda(0, 200_000, 256, torch.device("cuda", 0), 10, 0.05, seed=4, nonneg=True)
    A, E, s, sv, info = T.rpca(D, nonnegA=True, return_info=True)
    assert info["converged"] and sv == 10
    # the stop test bounds the SPECTRAL norm ratio by sqrt(eps) (src/robustPCA.jl:225); the Frobenius ratio of a
    # 200000 x 256 residual is within sqrt(256) of it
    res = (torch.linalg.norm(D - A - E) / torch.linalg.norm(D)).item()
    assert res < 16 * SQRT_EPS
    assert (A >= 0).all().item()
    assert abs((E != 0).double().mean().item() - 0.05) < 0.01            # the 5 % outliers are what E picks up
    UtU = s.U[:, :10].t() @ s.U[:, :10]
    assert (UtU - torch.eye(10, device=D.device, dtype=torch.float64)).abs().max().item() < 1e-8
    # idempotence: the recovered low-rank part is a fixed point (no sparse part left)
    A2, E2, _, sv2 = T.rpca(A, nonnegA=True, want_svd=False)
    assert sv2 == 10 and (torch.linalg.norm(E2) / torch.linalg.norm(A)).item() < 1e-6


def test_golden_vectors_extended():
    """tests/golden/oracle_vectors_ext.npz: hankel=true, channels, plain SSA (continuous maps -> 1e-9 against the
    committed oracle outputs; the discontinuous robust averages are compared with a live oracle run elsewhere)."""
    g = np.load(os.path.join(HERE, "golden", "oracle_vectors_ext.npz"))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        A, E, s, sv, info = T.rpca(g["hk_H"], hankel=True, nukeA=False, iters=12, tol=0.0, return_info=True)
    assert relF(A, g["hk_A"]) < TOL and relF(E, g["hk_E"]) < TOL
    assert np.array_equal(info["hist"][:, 1], g["hk_hist"][:, 1])
    assert np.array_equal(T.hankel(g["mc_Yn"], 5, 2), g["mc_H"])
    assert np.allclose(T.unhankel(g["mc_H"], 2, 300, 2), g["mc_unh"], rtol=0, atol=1e-13)
    assert relF(T.lowrankfilter(g["mc_Yn"], 12), g["mc_yf"]) < TOL
    assert relF(T.lowrankfilter(g["mc_Yn"], 12, lag=2, sv=4), g["mc_yf_ssa"]) < TOL
    assert relF(T.lowrankfilter(g["ssa_y"], 20, sv=2), g["ssa_yf"]) < TOL
