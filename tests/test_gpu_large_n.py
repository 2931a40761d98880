"""GPU parity for 2048 < min(M, N) <= 4096 against the live CPU oracle (run with -m gpu on the B200 box).

TMA SYRK with 18 and 32 blocks per edge, the generic 64-block Gram (M < 4096), the large-n subspace iteration, the full
Jacobi and the Cholesky of the returned SVD above 48 KB of shared memory, lowrankfilter's implicit, SSA and
multi-channel forms, the dense continuation for rank estimates above 32, and the 4096-column limit itself.
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
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL = 1e-9


def relF(a, b):
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


def solve_both(D, **kw):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        out = T.rpca(D, return_info=True, **kw)
        ref = O.rpca(D, **kw)
    return out, ref


def check_parity(out, ref, converged=False):
    A, E, s, sv, info = out
    assert relF(A, ref.A) < TOL, relF(A, ref.A)
    assert relF(E, ref.E) < TOL, relF(E, ref.E)
    assert np.array_equal(info["hist"][:, 1], ref.hist[:, 1])
    assert sv == ref.sv
    if converged:
        assert info["converged"] and info["iters"] == ref.iters
    S = ref.s.S
    assert np.abs(s.S - S).max() <= 1e-12 * S[0], np.abs(s.S - S).max() / S[0]
    d = s.Vt.shape[0]
    assert np.abs(s.Vt @ s.Vt.T - np.eye(d)).max() < 1e-11


@pytest.mark.parametrize("wide", [False, True])
def test_rpca_4400_x_2200_tma_syrk_18_blocks_per_edge(wide):
    """18 x 18 blocks of 128 columns, the last one partial; the wide form is solved on the transpose."""
    D = T.synth.lowrank_sparse_np(4400, 2200, 10, 0.05, seed=31)
    if wide:
        D = np.asfortranarray(D.T)
    check_parity(*solve_both(D, iters=5, tol=0.0))


def test_rpca_4200_x_2100_nonnegA_to_convergence():
    D = T.synth.lowrank_sparse_np(4200, 2100, 8, 0.05, seed=32, nonneg=True)
    check_parity(*solve_both(D, nonnegA=True), converged=True)


def test_rpca_3000_x_2500_generic_gram():
    """M < 4096: the Gram runs on the generic 64-block kernel (40 x 40 blocks)."""
    D = T.synth.lowrank_sparse_np(3000, 2500, 10, 0.05, seed=33)
    check_parity(*solve_both(D, iters=4, tol=0.0))


def test_rpca_8192_x_4096_at_the_limit():
    D = T.synth.lowrank_sparse_np(8192, 4096, 10, 0.05, seed=34)
    check_parity(*solve_both(D, iters=3, tol=0.0))


def test_more_than_4096_is_unsupported():
    import torch
    with pytest.raises(T.TlsqError) as ei:
        T.rpca(np.zeros((4097, 4097), order="F"), iters=1)
    assert ei.value.code == T._cabi.TLSQ_ERR_UNSUPPORTED and "4096" in str(ei.value)
    with pytest.raises(T.TlsqError) as ei:
        T.rpca(torch.zeros((4097, 5000), dtype=torch.float64, device="cuda").t(), iters=1)
    assert ei.value.code == T._cabi.TLSQ_ERR_UNSUPPORTED
    with pytest.raises(T.TlsqError) as ei:
        T.lowrankfilter(np.sin(0.01 * np.arange(9000.0)), 4097)
    assert ei.value.code == T._cabi.TLSQ_ERR_UNSUPPORTED and "4096" in str(ei.value)
    with pytest.raises(T.TlsqError) as ei:
        T.eigh(torch.eye(4097, dtype=torch.float64, device="cuda"))
    assert ei.value.code == T._cabi.TLSQ_ERR_UNSUPPORTED and "4096" in str(ei.value)


def test_lowrankfilter_n2304_implicit_ssa_and_two_channels():
    y, yn = T.synth.sinusoid_np(12_000, seed=35, noise=0.05)
    yf, info = T.lowrankfilter(yn, 2304, return_info=True)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ref = O.rpca(O.hankel(yn, 2304), tol=1e-3)
    assert info["iters"] == ref.iters and info["sv"] == ref.sv
    assert np.array_equal(info["hist"][:, 1], ref.hist[:, 1])
    assert relF(yf, O.unhankel_fast(ref.A)) < TOL
    # plain SSA branch (sv > 0): Gram + full Jacobi at n = 2304
    assert relF(T.lowrankfilter(yn, 2304, sv=4), O.lowrankfilter(yn, 2304, sv=4)) < TOL
    # two channels, n D = 2200 columns of the materialised trajectory matrix
    rng = np.random.default_rng(36)
    t = np.arange(5000)
    Y = np.column_stack([np.sin(0.01 * t), np.sin(0.03 * t) + 0.5 * np.sin(0.01 * t)])
    Yn = Y + 0.05 * rng.standard_normal(Y.shape) + (rng.random(Y.shape) < 0.01) * 3.0
    Yf = T.lowrankfilter(Yn, 1100)
    assert Yf.shape == Y.shape and relF(Yf, O.lowrankfilter(Yn, 1100)) < TOL


def test_rank_40_at_3000_x_2200_takes_the_dense_device_path():
    D = T.synth.lowrank_sparse_np(3000, 2200, 40, 0.05, seed=37)
    out, ref = solve_both(D, iters=3, tol=0.0)
    assert ref.hist[-1, 1] > 32
    check_parity(out, ref)
    # with tol = 0 the accelerated loop records the negative Frobenius bound as the cost; only the dense path evaluates
    # the exact opnorm(Z) every iteration, so exact positive costs show that the solve continued there
    assert np.all(out[4]["hist"][:, 2] > 0)
    assert np.allclose(out[4]["hist"][:, 2], ref.hist[:, 2], rtol=1e-8)


def test_eigh_3000_psd():
    import torch
    rng = np.random.default_rng(38)
    X = rng.standard_normal((3500, 3000)) * np.logspace(0, -3, 3000)
    G = X.T @ X
    lam, V = T.eigh(torch.from_numpy(G).cuda())
    lam, V = lam.cpu().numpy(), V.cpu().numpy()
    ref = np.linalg.eigvalsh(G)[::-1]
    assert np.abs(lam - ref).max() <= 1e-12 * ref[0], np.abs(lam - ref).max() / ref[0]
    assert np.abs(G @ V - V * lam).max() < 1e-11 * ref[0]
    assert np.abs(V.T @ V - np.eye(3000)).max() < 1e-11


def test_repeated_solves_at_8192_x_4096_are_deterministic():
    import torch
    D = T.synth.lowrank_sparse_cuda(0, 8192, 4096, torch.device("cuda", 0), 10, 0.05, seed=39, nonneg=True)
    hists = []
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for _ in range(2):
            A, E, s, sv, info = T.rpca(D, nonnegA=True, iters=3, tol=0.0, return_info=True, want_svd=False,
                                       exact_cost=True)
            hists.append(info["hist"].copy())
    assert np.array_equal(hists[0], hists[1])


def test_multi_gpu_parity_large_n_two_ranks():
    """Row-sharded solves at n = 2304 and n = 4096 on 2 GPUs (tools/mgpu_large_n_check.py).  Skipped below 2 GPUs."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29573",
                          os.path.join(ROOT, "tools", "mgpu_large_n_check.py")], capture_output=True, text=True, env=env,
                         timeout=3000)
    sys.stdout.write(out.stdout[-4000:])
    assert out.returncode == 0, out.stderr[-2000:]
    assert "MGPU_LARGE_N_CHECK PASS" in out.stdout
