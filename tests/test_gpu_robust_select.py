"""Robust Grassmann averages for any number of observations: the per-row radix selection kernels (ga_select.cu).

* the building block tlsq_robust_average_f64_dev (always the selection kernels) against the oracle's
  entrywise_trimmed_mean / entrywise_median (src/robustPCA.jl:323-333, :349-357) on continuous, heavily tied
  (small integers, exact +-0.0) and mixed-sign data, from 1 to 1 000 003 observations;
* rpca_ga(X, r, mu=...) above 16 384 observations (where the per-row sort stops) against the oracle, from NumPy and
  from CUDA tensors; repeat determinism; the robust averages' point on a large contaminated problem;
* a 2-rank row-sharded solve against the 1-GPU one (tools/mgpu_robust_check.py under torchrun, 2 GPUs only).
"""
import ctypes
import os
import subprocess
import sys
import warnings

import numpy as np
import pytest

import tls_oracle as O
import tlsq_b200 as T

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
PS = (0.0, 0.1, 0.25, 0.49)


def _data(kind, d, N, seed):
    rng = np.random.default_rng(seed)
    if kind == "tied":
        U = rng.integers(-3, 4, size=(d, N)).astype(np.float64)
        U[(U == 0) & (rng.random((d, N)) < 0.5)] = -0.0                     # exact +-0.0 must compare equal
        w = rng.choice(np.array([-2.0, -1.0, -0.5, 0.5, 1.0, 2.0]), size=N)
    else:
        U = rng.standard_normal((d, N))
        w = np.abs(rng.standard_normal(N)) + 0.1
        if kind == "mixed":
            w *= np.where(rng.random(N) < 0.5, -1.0, 1.0)
    return np.asfortranarray(U), w


def _cuda(a):
    import torch
    a = np.asarray(a)
    if a.ndim == 2:
        return torch.from_numpy(np.ascontiguousarray(a.T)).cuda().t()
    return torch.from_numpy(a).cuda()


def _trim_scale(U, w, P):
    """(sum |w u| + |s| sum |w|) / |sum w| over each row's kept set: what a reordered sum may move s by, in units of
    the rounding unit.  The rows' kept sets come from the same stable argsort as the oracle's."""
    N = U.shape[1]
    lo, hi = int(np.floor(P * N)), int(np.floor((1 - P) * N))
    out = np.zeros(U.shape[0])
    for j in range(U.shape[0]):
        I = np.argsort(U[j], kind="stable")[lo:hi]
        den = abs(np.sum(w[I]))
        s = abs(np.sum(w[I] * U[j, I]) / den) if den else 0.0
        out[j] = (np.abs(w[I]) @ np.abs(U[j, I]) + s * np.abs(w[I]).sum()) / den if den else 0.0
    return out


CASES = [(N, d, kind) for N in (1, 2, 3, 17, 1000, 16_385, 100_000) for d in (1, 7, 64)
         for kind in ("cont", "tied", "mixed")]
CASES += [(1_000_003, d, kind) for d in (1, 7) for kind in ("cont", "tied", "mixed")]
BIG = [(1_000_003, 64, "tied"), (1_000_003, 64, "mixed")]               # one P per case: the oracle sorts 64 rows


def _check(U, w, Ps):
    import torch
    Ut, wt = _cuda(U), _cuda(w)
    with warnings.catch_warnings(), np.errstate(invalid="ignore", divide="ignore"):
        warnings.simplefilter("ignore")
        med = T.robust_average(Ut, wt, T.entrywise_median).cpu().numpy()
        medo = O.entrywise_median(np.zeros(U.shape[0]), w, U)
        assert np.array_equal(med.view(np.int64), medo.view(np.int64)), np.nonzero(med != medo)
        for P in Ps:
            tm = T.robust_average(Ut, wt, T.entrywise_trimmed_mean, P).cpu().numpy()
            tmo = O.entrywise_trimmed_mean(np.zeros(U.shape[0]), w, U, P).copy()
            assert np.array_equal(np.isnan(tm), np.isnan(tmo)), P
            ok = ~np.isnan(tmo)
            tol = 1e-12 * np.maximum(_trim_scale(U, w, P), np.abs(tmo))[ok]
            same = tm[ok] == tmo[ok]                         # incl. +-inf: tied weights that sum to exactly 0
            err = np.where(same, 0.0, np.abs(tm[ok] - tmo[ok]))
            assert np.all(err <= tol), (P, float(np.max(err / np.maximum(tol, 1e-300))))
    torch.cuda.synchronize()


@pytest.mark.gpu
@pytest.mark.parametrize("N,d,kind", CASES)
def test_building_block_matches_the_oracle(N, d, kind):
    """median bit-equal; trimmed mean within 1e-12 of the sum's scale (only the summation order differs)"""
    U, w = _data(kind, d, N, seed=N + 31 * d + len(kind))
    _check(U, w, PS)


@pytest.mark.gpu
@pytest.mark.parametrize("N,d,kind", BIG)
def test_building_block_matches_the_oracle_wide(N, d, kind):
    U, w = _data(kind, d, N, seed=N + d)
    _check(U, w, (0.1,))


@pytest.mark.gpu
def test_building_block_nan_keys_do_not_hang():
    """a zero column gives NaN keys in rpca_ga (0 / ||x_n||); here NaN entries of U: they sort last, the call returns"""
    U, w = _data("cont", 5, 40_000, seed=3)
    U[:, 123] = np.nan
    U[2, 7] = np.nan
    Ut, wt = _cuda(U), _cuda(w)
    med = T.robust_average(Ut, wt, T.entrywise_median).cpu().numpy()
    tm = T.robust_average(Ut, wt, T.entrywise_trimmed_mean, 0.1).cpu().numpy()
    assert np.all(np.isfinite(med)) and np.all(np.isfinite(tm))    # the NaNs are among the dropped top 10 %


def _ga_problem(d, N, r, seed, scale=1.0, with_basis=False):
    """rank r (planted basis U0[:, :r], entries of size ~scale) + 1e-3 noise + gross outliers of size 1000 on 1 % of
    the entries; start vectors q0"""
    rng = np.random.default_rng(seed)
    U0, S0, Vt0 = np.linalg.svd(rng.standard_normal((d, N)), full_matrices=False)
    A = scale * (U0[:, :r] * S0[:r]) @ Vt0[:r] + 1e-3 * rng.standard_normal((d, N))
    A += 1000.0 * rng.standard_normal((d, N)) * (rng.random((d, N)) < 0.01)
    out = (np.asfortranarray(A), np.asfortranarray(rng.standard_normal((d, r))))
    return out + (U0[:, :r],) if with_basis else out


@pytest.mark.gpu
@pytest.mark.parametrize("d,N,r", [(16, 40_000, 2), (32, 100_000, 2)])
def test_rpca_ga_robust_averages_above_the_sort_limit(d, N, r):
    """rpca_ga(...; μ = entrywise_trimmed_mean / entrywise_median) beyond 16 384 observations, host and device entry,
    against the oracle with the same start vectors (data as test_gpu_parity.py::test_rpca_ga_robust_averages)."""
    A, q0 = _ga_problem(d, N, r, seed=d + N)
    for tag, omu in ((T.entrywise_trimmed_mean, O.entrywise_trimmed_mean), (T.entrywise_median, O.entrywise_median)):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            Qo, its = O.rpca_ga(A, r, q0=q0, mu=omu, exact_order=False, iters=30, return_iters=True)
            Qh, infh = T.rpca_ga(A, r, mu=tag, q0=q0, iters=30, return_info=True)
            Qd, infd = T.rpca_ga(_cuda(A), r, mu=tag, q0=_cuda(q0), iters=30, return_info=True)
        for Q, info in ((Qh, infh), (Qd.cpu().numpy(), infd)):
            sgn = np.sign(np.sum(Q * Qo, axis=0))
            assert info["iters"] == its, (tag.__name__, info["iters"], its)
            assert np.abs(Q * sgn - Qo).max() < 1e-8, (tag.__name__, np.abs(Q * sgn - Qo).max())


@pytest.mark.gpu
def test_rpca_ga_robust_averages_are_deterministic():
    A, q0 = _ga_problem(24, 60_000, 2, seed=5)
    Ad, qd = _cuda(A), _cuda(q0)
    for tag in (T.entrywise_trimmed_mean, T.entrywise_median):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            Q1, i1 = T.rpca_ga(Ad, 2, mu=tag, q0=qd, iters=30, return_info=True)
            Q2, i2 = T.rpca_ga(Ad, 2, mu=tag, q0=qd, iters=30, return_info=True)
        assert i1 == i2
        assert np.array_equal(Q1.cpu().numpy().view(np.int64), Q2.cpu().numpy().view(np.int64)), tag.__name__


@pytest.mark.gpu
def test_robust_averages_resist_outliers_at_50k_observations():
    """test/runtests.jl:491-523 at N = 50 000: gross outliers (size 1000) on 1 % of the entries of a rank-2 signal of
    size ~10 drag the plain Grassmann average away from the planted subspace; both robust averages stay clearly closer.

    The advantage is the reference's, not a property of the kernels, and it depends on the regime.  The averages weight
    every observation by its norm, and 1 % outlier entries corrupt ~10 % of the columns.  With a much weaker signal
    those columns dominate every row's weight sum and the trimmed mean does no better than mu!; with a much stronger
    one mu! is barely moved.  So the errors are also checked against the oracle's: with this seed the oracle gives
    1.22 (mu!), 0.60 (trimmed mean) and 0.37 (median)."""
    d, N, r = 10, 50_000, 2
    X, q0, B = _ga_problem(d, N, r, seed=5, scale=10.0, with_basis=True)
    err, erro = {}, {}
    for tag, omu in ((T.mu_mean, None), (T.entrywise_trimmed_mean, O.entrywise_trimmed_mean),
                     (T.entrywise_median, O.entrywise_median)):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            Q = T.rpca_ga(X, r, mu=tag, q0=q0, iters=100)
            Qo = O.rpca_ga(X, r, q0=q0, mu=omu, exact_order=False, iters=100)
        err[tag.__name__] = float(np.linalg.norm(B - Q @ (Q.T @ B)))
        erro[tag.__name__] = float(np.linalg.norm(B - Qo @ (Qo.T @ B)))
    for k in err:
        assert abs(err[k] - erro[k]) < 1e-6, (k, err, erro)
    assert err["entrywise_trimmed_mean"] < 0.75 * err["mu_mean"], err
    assert err["entrywise_median"] < 0.75 * err["mu_mean"], err


@pytest.mark.gpu
def test_sharded_robust_averages_match_one_gpu(tmp_path):
    """2 ranks, rows of X sharded: the selection is per row, so the shards need no extra collective; Q and the
    iteration counts equal the 1-GPU solve's."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    A, q0 = _ga_problem(32, 40_000, 2, seed=11)
    ref = {}
    for name, tag in (("trimmed", T.entrywise_trimmed_mean), ("median", T.entrywise_median)):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            Q, info = T.rpca_ga(_cuda(A), 2, mu=tag, q0=_cuda(q0), iters=30, return_info=True)
        ref[f"Q_{name}"], ref[f"its_{name}"] = Q.cpu().numpy(), np.array(info["iters"])
    path = str(tmp_path / "robust_ref.npz")
    np.savez(path, A=A, q0=q0, **ref)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29573",
                          os.path.join(ROOT, "tools", "mgpu_robust_check.py"), path], capture_output=True, text=True,
                         env=env, timeout=900)
    sys.stdout.write(out.stdout[-4000:])
    assert out.returncode == 0, out.stderr[-2000:]
    assert "MGPU_ROBUST PASS" in out.stdout


def test_building_block_is_exported_and_needs_a_gpu():
    lib = ctypes.CDLL(T._cabi.LIB_PATH)
    assert hasattr(lib, "tlsq_robust_average_f64_dev")
    if T.load().tlsq_device_count() != 0:
        return
    U = np.zeros((3, 4))
    w = np.ones(4)
    s = np.zeros(3)
    dp = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    for kind in (1, 2):
        rc = T.load().tlsq_robust_average_f64_dev(None, dp(U), 3, 4, dp(w), kind, 0.1, dp(s))
        assert rc == T._cabi.TLSQ_ERR_NO_DEVICE
