"""Synthetic workloads of BASELINE.json / SURVEY.md 8(d) (C1..C5).  NumPy generators for parity-sized problems and
chunk-seeded torch generators for the full-size shapes, so that every rank of a row-sharded run can build exactly
its own rows of the same global matrix."""
from __future__ import annotations

import math

import numpy as np

SPARSE_MAG = 10.0 * math.sqrt(10.0)
CHUNK_ROWS = 15625          # 1_000_000 / 64: shard boundaries of 1/2/4/8 ranks fall on chunk boundaries


def shard_rows(M: int, nranks: int, rank: int, align: int = 1):
    """Contiguous row range [r0, r1) of rank `rank`; boundaries are multiples of `align` (except the last)."""
    units = (M + align - 1) // align
    base, rem = divmod(units, nranks)
    u0 = rank * base + min(rank, rem)
    u1 = u0 + base + (1 if rank < rem else 0)
    return min(u0 * align, M), min(u1 * align, M)


def lowrank_sparse_np(M: int, N: int, r: int = 10, frac: float = 0.05, seed: int = 0, nonneg: bool = False):
    """D = L + S, L = G1 G2 (|G1||G2| when nonneg), S_ij = 10 sqrt(10) U(-1,1) (U(0,1) when nonneg) w.p. frac."""
    rng = np.random.default_rng(seed)
    G1 = rng.standard_normal((M, r))
    G2 = rng.standard_normal((r, N))
    if nonneg:
        G1, G2 = np.abs(G1), np.abs(G2)
    mask = rng.random((M, N)) < frac
    u = rng.random((M, N)) if nonneg else rng.uniform(-1.0, 1.0, (M, N))
    return np.asfortranarray(G1 @ G2 + SPARSE_MAG * u * mask)


def ga_data_np(d: int, N: int, r: int = 10, seed: int = 3, out_frac: float = 0.1):
    """X = G1 diag(1..r) G2 + 0.01 noise; a fraction of the columns gets +100 N(0,1) in every entry (C3)."""
    rng = np.random.default_rng(seed)
    X = (rng.standard_normal((d, r)) * np.arange(1, r + 1)) @ rng.standard_normal((r, N))
    X += 0.01 * rng.standard_normal((d, N))
    out = rng.random(N) < out_frac
    X[:, out] += 100.0 * rng.standard_normal((d, int(out.sum())))
    q0 = rng.standard_normal((d, r))
    return np.asfortranarray(X), np.asfortranarray(q0)


def sinusoid_np(Ns: int, seed: int = 5, miss_frac: float = 0.1, noise: float = 0.0):
    """C5 / README signal: sum of three sinusoids, `miss_frac` of the samples replaced by +1e2 (README.md:83)."""
    rng = np.random.default_rng(seed)
    t = np.arange(1, Ns + 1, dtype=np.float64)
    y = np.sin(0.1 * t) + 0.5 * np.sin(0.37 * t + 1.0) + 0.25 * np.sin(0.013 * t + 2.0)
    yn = y + 1e2 * (rng.random(Ns) < miss_frac)
    if noise:
        yn = yn + noise * rng.standard_normal(Ns)
    return y, yn


def sinusoids_np(Ns: int, k: int, seed: int = 5, noise: float = 0.05, outlier_frac: float = 0.01):
    """Sum of k sinusoids (frequencies in [0.02, 0.92), random phases, amplitudes in [0.5, 1.5)), `noise` N(0,1) noise
    and `outlier_frac` of the samples shifted by +5.  The Hankel rank of the clean signal is 2k, so the rank estimate
    of lowrankfilter grows with k.  Returns (clean, noisy)."""
    rng = np.random.default_rng(seed)
    t = np.arange(Ns)
    freqs = 0.02 + 0.9 * rng.random(k)
    y0 = sum(np.sin(f * t + rng.random() * 6.28) * (0.5 + rng.random()) for f in freqs)
    y = y0 + noise * rng.standard_normal(Ns)
    y[rng.random(Ns) < outlier_frac] += 5.0
    return y0, y


def lowrank_sparse_cuda(r0: int, r1: int, N: int, device, r: int = 10, frac: float = 0.05, seed: int = 4,
                        nonneg: bool = True):
    """Rows [r0, r1) of the global low-rank + sparse matrix as a column-major CUDA tensor (shape (r1-r0, N)).
    Chunk-seeded: the global matrix does not depend on how many ranks build it."""
    import torch
    g = torch.Generator(device=device)
    g.manual_seed(seed * 1_000_003 + 17)
    G2 = torch.randn((r, N), dtype=torch.float64, device=device, generator=g)
    if nonneg:
        G2 = G2.abs()
    Dt = torch.empty((N, r1 - r0), dtype=torch.float64, device=device)       # row-major (N, m) == column-major (m, N)
    c = r0 // CHUNK_ROWS
    while c * CHUNK_ROWS < r1:
        a, b = max(c * CHUNK_ROWS, r0), min((c + 1) * CHUNK_ROWS, r1)
        g.manual_seed(seed * 1_000_003 + 1000 + c)
        rows = CHUNK_ROWS
        G1 = torch.randn((rows, r), dtype=torch.float64, device=device, generator=g)
        U = torch.rand((rows, N), dtype=torch.float64, device=device, generator=g)
        Mk = torch.rand((rows, N), dtype=torch.float64, device=device, generator=g) < frac
        if nonneg:
            G1 = G1.abs()
        else:
            U = 2.0 * U - 1.0
        blk = G1 @ G2 + SPARSE_MAG * U * Mk
        lo, hi = a - c * CHUNK_ROWS, b - c * CHUNK_ROWS
        Dt[:, a - r0:b - r0] = blk[lo:hi].t()
        c += 1
    return Dt.t()


def ga_data_cuda(r0: int, r1: int, N: int, device, r: int = 10, seed: int = 3, out_frac: float = 0.1):
    """Rows [r0, r1) of the C3 matrix X (d x N, columns are observations) and of q0 (d x r), column-major."""
    import torch
    g = torch.Generator(device=device)
    g.manual_seed(seed * 1_000_003 + 17)
    G2 = torch.randn((r, N), dtype=torch.float64, device=device, generator=g)
    out = (torch.rand((N,), dtype=torch.float64, device=device, generator=g) < out_frac).to(torch.float64)
    scale = torch.arange(1, r + 1, dtype=torch.float64, device=device)
    Xt = torch.empty((N, r1 - r0), dtype=torch.float64, device=device)
    q0t = torch.empty((r, r1 - r0), dtype=torch.float64, device=device)
    c = r0 // CHUNK_ROWS
    while c * CHUNK_ROWS < r1:
        a, b = max(c * CHUNK_ROWS, r0), min((c + 1) * CHUNK_ROWS, r1)
        g.manual_seed(seed * 1_000_003 + 1000 + c)
        rows = CHUNK_ROWS
        G1 = torch.randn((rows, r), dtype=torch.float64, device=device, generator=g)
        noise = torch.randn((rows, N), dtype=torch.float64, device=device, generator=g)
        gross = torch.randn((rows, N), dtype=torch.float64, device=device, generator=g)
        q = torch.randn((rows, r), dtype=torch.float64, device=device, generator=g)
        blk = (G1 * scale) @ G2 + 0.01 * noise + 100.0 * gross * out
        lo, hi = a - c * CHUNK_ROWS, b - c * CHUNK_ROWS
        Xt[:, a - r0:b - r0] = blk[lo:hi].t()
        q0t[:, a - r0:b - r0] = q[lo:hi].t()
        c += 1
    return Xt.t(), q0t.t()
