"""Every kernel path of rpca_ga against the oracle (oracle/tls_oracle.py, exact_order=False, same start vectors).

* The robust averages (src/robustPCA.jl:323-333 entrywise_trimmed_mean, :349-357 entrywise_median) on both sides of
  each regime boundary of launch_ga_robust: the tiled per-row sort with 32 rows per tile (N <= 512) and with 8 rows
  per tile (N <= 1024), one row per CTA (N <= 16 384), and the radix selection of ga_select.cu above that (16 385).
  Also the shapes where a CTA loops over several row tiles.  The data are continuous, tied (integer columns that are
  power-of-two multiples of signed permutations of one vector, so the keys tie exactly), tied with -0.0 entries, and
  either of these with all-zero columns.  A zero column has the key 0 / 0 = NaN, which both orders put after +inf.
* Single-average probes (one iteration, r = 1) pin one robust average; full r = 2 solves pin the whole iteration,
  including the fused TMA deflation feeding the sort (d = 8 194).
* mu! on the TMA sweep's edges: partial column boxes (N < 256), a partial last row tile (d mod 32 != 0), and the
  shapes just outside it (odd d, N = 7, N = 257).
* One process on two GPUs: kernels whose dynamic shared memory attribute must be set on each device.
"""
import warnings

import numpy as np
import pytest

import tls_oracle as O
import tlsq_b200 as T


def _trim_scale(U, w, P):
    """(sum |w u| + |s| sum |w|) / |sum w| over each row's kept set: what a reordered sum may move s by, in units of
    the rounding unit.  The rows' kept sets come from the same stable argsort as the oracle's (NaN keys last)."""
    N = U.shape[1]
    lo, hi = int(np.floor(P * N)), int(np.floor((1 - P) * N))
    out = np.zeros(U.shape[0])
    for j in range(U.shape[0]):
        I = np.argsort(U[j], kind="stable")[lo:hi]
        den = abs(np.sum(w[I]))
        s = abs(np.sum(w[I] * U[j, I]) / den) if den else 0.0
        out[j] = (np.abs(w[I]) @ np.abs(U[j, I]) + s * np.abs(w[I]).sum()) / den if den else 0.0
    return out


def _start(d, seed):
    """a start vector with positive entries: with the tied data's mostly positive entries, the rows' keys are not
    symmetric about 0, so the median of a row is rarely an exact 0 (all-zero medians would leave q = 0 / 0)"""
    return np.abs(np.random.default_rng(seed).standard_normal(d)) + 0.5


def _data(kind, d, N, q0, seed):
    """d x N observations for the start vector q0.

    cont:  standard normal.
    tied:  column n is 2^e_n (0 <= e_n <= 10) times a signed permutation of one integer vector v (0 < v_i < 2^12
           but one v_i = 0; 70 % of the signs +).  Scaling by a power of two is exact, so every key of row j is
           exactly one of +-v_i / ||v||: the keys tie across all columns while the weights +-2^e_n ||v|| differ (equal
           weights of both signs can cancel a weight sum exactly).  Sums of squares are exact in any order and the
           division is correctly rounded, so GPU and oracle keys are bit-equal.  Zero entries are +0.0.
    tied0: tied, with the zero entries' signs kept (-0.0 and +0.0 mixed).
    *_z:   k = floor(N / 10) columns set to zero at scattered positions (k <= floor(P N) for P >= 0.1: their NaN keys
           fall in the trimmed mean's dropped range).
    Every tenth column is flipped to x_n'q0 < 0 and the others to x_n'q0 > 0: at most ~10 % negative weights, so the
    trimmed mean's weight sum over any kept half of a row stays well away from 0 (it can cancel exactly otherwise).
    """
    rng = np.random.default_rng(seed)
    base = kind.split("_")[0]
    if base == "cont":
        X = rng.standard_normal((d, N))
    else:
        v = rng.integers(1, 1 << 12, size=d).astype(np.float64)
        if d > 1:
            v[0] = 0.0
        X = np.empty((d, N))
        for n in range(N):
            X[:, n] = v[rng.permutation(d)] * np.where(rng.random(d) < 0.7, 1.0, -1.0)
        X *= 2.0 ** rng.integers(0, 11, size=N)
        if base == "tied":
            X += 0.0                                                          # -0.0 -> +0.0
    want = np.where(np.arange(N) % 10 == 9, -1.0, 1.0)
    X *= np.where(np.sign(q0 @ X) == want, 1.0, -1.0)
    if kind.endswith("_z"):
        X[:, rng.choice(N, size=N // 10, replace=False)] = 0.0
    return np.asfortranarray(X)


def _signs_well_defined(X, q0):
    """precondition of the one-iteration probe: every sign(x_n'q) is far from a rounding decision"""
    nx = np.linalg.norm(X, axis=0)
    dots = np.abs((q0 / np.linalg.norm(q0)) @ X)
    nz = nx > 0
    assert np.all(dots[nz] > 1e-9 * nx[nz]), "start vector nearly orthogonal to an observation: pick another seed"


def _oracle_weights(X, q0):
    """U and w of the oracle's first iteration (src/robustPCA.jl:265-266, :291-293)"""
    with np.errstate(invalid="ignore", divide="ignore"):
        nx = np.sqrt(np.sum(X * X, axis=0))
        U = X / nx
        w = np.sign(U.T @ (q0 / np.linalg.norm(q0))) * nx
    return U, w


def _probe(X, q0, tag, P=None):
    """rpca_ga(X, 1; mu, q0, iters=1): one robust average with the signs from q0, normalised"""
    mu = tag if P is None else (tag, P)
    q = T.rpca_ga(X, 1, mu=mu, q0=q0[:, None], iters=1)[:, 0]
    return q


KINDS = ("cont", "tied", "tied0", "cont_z", "tied0_z")
PROBES = [(d, N, kind) for N in (2, 3, 31, 512, 513, 1024, 1025, 16_384, 16_385) for d in (1, 7, 33)
          for kind in KINDS if not (kind.endswith("_z") and N < 10)]
PROBES += [(d, N, kind) for d, N in ((12_000, 300), (2_500, 700), (400, 2_000)) for kind in KINDS]


@pytest.mark.gpu
@pytest.mark.parametrize("d,N,kind", PROBES)
def test_one_robust_average_matches_the_oracle(d, N, kind):
    """median within 1e-13 per entry (only the normalisation differs; a wrong selection moves an entry by a gap between
    order statistics); trimmed mean within 1e-12 of each row's summation scale over ||s||"""
    seed = 7919 * d + N + len(kind)
    q0 = _start(d, seed)
    X = _data(kind, d, N, q0, seed)
    _signs_well_defined(X, q0)
    U, w = _oracle_weights(X, q0)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        q = _probe(X, q0, T.entrywise_median)
        qo = O.rpca_ga(X, 1, q0=q0[:, None], mu=O.entrywise_median, exact_order=False, iters=1)[:, 0]
    assert np.all(np.isfinite(qo))
    err = np.abs(q - qo)
    assert np.all(err <= 1e-13), ("median", int(np.argmax(err)), float(np.nanmax(err)))
    for P in (0.1, 0.25):
        omu = lambda s_, w_, U_: O.entrywise_trimmed_mean(s_, w_, U_, P)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            q = _probe(X, q0, T.entrywise_trimmed_mean, P)
            qo = O.rpca_ga(X, 1, q0=q0[:, None], mu=omu, exact_order=False, iters=1)[:, 0]
            s = O.entrywise_trimmed_mean(np.zeros(d), w, U, P)
        assert np.all(np.isfinite(qo)) and np.linalg.norm(s) > 0
        tol = 1e-12 * np.maximum(_trim_scale(U, w, P), np.abs(s)) / np.linalg.norm(s)
        err = np.where(q == qo, 0.0, np.abs(q - qo))
        assert np.all(err <= tol), ("trimmed", P, int(np.argmax(err / tol)), float(np.nanmax(err / tol)))


def _full_problem(kind, d, N, seed):
    """rank-2 signal + 1e-3 noise + gross outliers on 1 % of the entries (as test_gpu_parity.py), optionally with zero
    columns; or the tied integer data of _data (with -0.0 and zero columns)"""
    rng = np.random.default_rng(seed)
    q0 = np.asfortranarray(rng.standard_normal((d, 2)))
    if kind == "tied0_z":
        q0[:, 0] = _start(d, seed)
        return _data(kind, d, N, q0[:, 0], seed), q0
    U0, S0, Vt0 = np.linalg.svd(rng.standard_normal((d, N)), full_matrices=False)
    A = (U0[:, :2] * S0[:2]) @ Vt0[:2] + 1e-3 * rng.standard_normal((d, N))
    A += 1000.0 * rng.standard_normal((d, N)) * (rng.random((d, N)) < 0.01)
    if kind == "cont_z":
        A[:, rng.choice(N, size=N // 10, replace=False)] = 0.0
    return np.asfortranarray(A), q0


FULL = [(40, N, kind) for N in (400, 800, 3_000) for kind in ("cont_z", "tied0_z")]
FULL += [(8_194, 200, "cont_z")]


@pytest.mark.gpu
@pytest.mark.parametrize("d,N,kind", FULL)
def test_robust_solves_match_the_oracle(d, N, kind):
    """r = 2 to convergence: identical iteration counts, Q within 1e-8 up to sign.  At d = 8 194 the fused TMA
    deflation supplies the second component's norms and first dot products to the sort."""
    X, q0 = _full_problem(kind, d, N, seed=d + N + len(kind))
    for tag, omu in ((T.entrywise_trimmed_mean, O.entrywise_trimmed_mean), (T.entrywise_median, O.entrywise_median)):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            Q, info = T.rpca_ga(X, 2, mu=tag, q0=q0, iters=30, return_info=True)
            Qo, its = O.rpca_ga(X, 2, q0=q0, mu=omu, exact_order=False, iters=30, return_iters=True)
        assert np.all(np.isfinite(Qo))
        sgn = np.sign(np.sum(Q * Qo, axis=0))
        assert info["iters"] == its, (tag.__name__, info["iters"], its)
        assert np.abs(Q * sgn - Qo).max() < 1e-8, (tag.__name__, np.abs(Q * sgn - Qo).max())


def _mean_problem(d, N, seed):
    """rank 3 with well separated scales + 0.01 noise: three components that converge quickly"""
    rng = np.random.default_rng(seed)
    X = (rng.standard_normal((d, 3)) * np.array([8.0, 4.0, 2.0])) @ rng.standard_normal((3, N))
    X += 0.01 * rng.standard_normal((d, N))
    return np.asfortranarray(X), np.asfortranarray(rng.standard_normal((d, 3)))


TMA_EDGES = [(d, N) for d in (8_192, 8_194) for N in (8, 100, 255, 256)] + [(8_193, 100), (8_192, 7), (8_192, 257)]


@pytest.mark.gpu
@pytest.mark.parametrize("d,N", TMA_EDGES)
def test_mean_sweep_edges_match_the_oracle(d, N):
    """mu! with r = 3 (two fused deflations where the TMA sweep applies): identical iteration counts, Q within 1e-9 up
    to sign.  N < 256 leaves the column box partly out of bounds, d = 8 194 the last row tile; d = 8 193 (odd leading
    dimension), N = 7 and N = 257 take the register sweep and the separate deflation."""
    X, q0 = _mean_problem(d, N, seed=d + N)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        Q, info = T.rpca_ga(X, 3, q0=q0, iters=200, return_info=True)
        Qo, its = O.rpca_ga(X, 3, q0=q0, exact_order=False, iters=200, return_iters=True)
    sgn = np.sign(np.sum(Q * Qo, axis=0))
    assert info["iters"] == its, (info["iters"], its)
    assert np.abs(Q * sgn - Qo).max() < 1e-9, np.abs(Q * sgn - Qo).max()


@pytest.mark.gpu
def test_two_devices_in_one_process():
    """Kernels with more than 48 KB of dynamic shared memory need the attribute on every device they run on: rpca at
    8192 x 192 (SYRK TMA, the DMMA GEMM of the returned SVD), lowrankfilter with n = 256 on a rank-10 signal (factored
    unhankel) and rpca_ga with the trimmed mean at N = 600, first on cuda:0 and then on cuda:1."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    D = T.synth.lowrank_sparse_np(8192, 192, 6, 0.05, seed=3)
    t = np.arange(1, 6001, dtype=np.float64)
    y = sum(np.sin(f * t + p) for f, p in ((0.05, 0.0), (0.13, 1.0), (0.29, 2.0), (0.41, 0.5), (0.7, 1.5)))
    y += 50.0 * (np.random.default_rng(2).random(t.size) < 0.05)
    X, q0 = _full_problem("cont_z", 64, 600, seed=9)
    out = []
    for dev in (0, 1):
        with torch.cuda.device(dev):
            cu = lambda a: torch.from_numpy(np.ascontiguousarray(a.T)).to(f"cuda:{dev}").t() if a.ndim == 2 \
                else torch.from_numpy(a).to(f"cuda:{dev}")
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                A, E, s, sv = T.rpca(cu(D), iters=8, tol=0.0)
                yf = T.lowrankfilter(cu(y), 256)
                Q = T.rpca_ga(cu(X), 2, mu=T.entrywise_trimmed_mean, q0=cu(q0), iters=30)
            torch.cuda.synchronize()
            host = lambda a: a.cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
            out.append([host(a) for a in (A, E, s.U, s.S, s.Vt, yf, Q)])
    for name, a0, a1 in zip(("A", "E", "U", "S", "Vt"), out[0][:5], out[1][:5]):
        assert np.array_equal(a0.view(np.int64), a1.view(np.int64)), name          # rpca: bit-equal across devices
    for name, a0, a1 in zip(("yf", "Q"), out[0][5:], out[1][5:]):
        assert np.abs(a0 - a1).max() <= 1e-12 * max(1.0, np.abs(a0).max()), name
