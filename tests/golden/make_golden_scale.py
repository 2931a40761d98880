"""BASELINE-scale oracle fixtures (tests/golden/oracle_scale.npz): the CPU oracle run to the reference's tolerance on
problems shaped like BASELINE.json's configurations, reduced to what fits in a small committed file.

    python tests/golden/make_golden_scale.py        (about 6 minutes on 8 cores)

The inputs are NOT stored: they are regenerated on the GPU box by the same seeded NumPy generators
(totalleastsquares.jl_b200/synth.py).  Stored per case: every `STRIDE`-th row of A-hat and E-hat, the column sums and
Frobenius norms of the full A-hat / E-hat (they pin the rows that are not stored), nnz(E-hat), the singular values of
the last SVT input, the (k, svp, cost) history and the iteration count.

  c4s   rpca(D; nonnegA=true) on 100 000 x 256, rank 10 + 5 % sparse, to convergence  (configs[3] at 1/10 of the rows)
  c2s   rpca(D) on 100 000 x 512, rank 10 + 5 % sparse, 6 iterations at tol = 0        (configs[1], full size)
  c3s   rpca_ga(X, 3) on 200 000 x 256 with 10 % gross outlier columns                 (configs[2] at 1/10 of the rows)
  lrfs  lowrankfilter(y, 256) on 40 000 samples                                        (configs[4] at 1/1250)
"""
import os
import sys
import time
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, ROOT)
import tls_oracle as O  # noqa: E402
import tlsq_b200 as T  # noqa: E402  (only the NumPy generators in synth.py are used)

STRIDE = 1497               # keeps the committed file under 1 MB; the digests pin the rows in between


def reduce_rpca(out, name, r, D):
    out[f"{name}_A_rows"] = np.ascontiguousarray(r.A[::STRIDE])
    out[f"{name}_E_rows"] = np.ascontiguousarray(r.E[::STRIDE])
    out[f"{name}_A_colsum"] = r.A.sum(axis=0)
    out[f"{name}_E_colsum"] = r.E.sum(axis=0)
    out[f"{name}_A_fro"] = np.linalg.norm(r.A)
    out[f"{name}_E_fro"] = np.linalg.norm(r.E)
    out[f"{name}_E_nnz"] = int(np.count_nonzero(r.E))
    out[f"{name}_S"] = r.s.S
    out[f"{name}_hist"] = r.hist
    out[f"{name}_iters"] = r.iters
    out[f"{name}_sv"] = r.sv
    out[f"{name}_Dmax"] = np.abs(D).max()


def main():
    warnings.simplefilter("ignore")
    out = {"stride": STRIDE}
    t0 = time.time()
    D = T.synth.lowrank_sparse_np(100_000, 256, 10, 0.05, seed=4, nonneg=True)
    r = O.rpca(D, nonnegA=True)
    reduce_rpca(out, "c4s", r, D)
    print(f"c4s: {r.iters} iterations, sv {r.sv}, {time.time() - t0:.0f} s", flush=True)
    t0 = time.time()
    D = T.synth.lowrank_sparse_np(100_000, 512, 10, 0.05, seed=2)
    r = O.rpca(D, iters=6, tol=0.0)
    reduce_rpca(out, "c2s", r, D)
    print(f"c2s: {r.iters} iterations, {time.time() - t0:.0f} s", flush=True)
    t0 = time.time()
    X, q0 = T.synth.ga_data_np(200_000, 256, 10, seed=3)
    Q, its = O.rpca_ga(X, 3, q0=q0[:, :3], exact_order=False, return_iters=True)
    out["c3s_Q_rows"] = np.ascontiguousarray(Q[::STRIDE])
    out["c3s_Q_colsum_abs"] = np.abs(Q.sum(axis=0))
    out["c3s_iters"] = np.array(its)
    print(f"c3s: iterations {its}, {time.time() - t0:.0f} s", flush=True)
    t0 = time.time()
    y, yn = T.synth.sinusoid_np(40_000, seed=5)
    out["lrfs_yf"] = O.lowrankfilter(yn, 256)
    print(f"lrfs: {time.time() - t0:.0f} s", flush=True)
    path = os.path.join(HERE, "oracle_scale.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
