"""Large-embedding fixture (tests/golden/oracle_largen.npz): the reference's DEFAULT lowrankfilter call
`lowrankfilter(y)` with n = min(N / 20, 2000) (src/robustPCA.jl:119) on N = 50 000 samples -> n = 2000, Hankel matrix
48 001 x 2000.  The CPU oracle needs a full dgesdd of that matrix twice per ALM iteration (tens of minutes in total), so
the result is committed instead of being recomputed in the test.  Also rpca on a 3000 x 1000 matrix (min(M,N) > 512)
for 4 iterations, with the returned singular values.

    python tests/golden/make_golden_largen.py
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
import tlsq_b200 as T  # noqa: E402

STRIDE = 74                 # stored rows of the 3000 x 1000 case; column sums and norms pin the rows in between

def main():
    warnings.simplefilter("ignore")
    out = {}
    t0 = time.time()
    D = T.synth.lowrank_sparse_np(3000, 1000, 8, 0.05, seed=21)
    r = O.rpca(D, iters=4, tol=0.0)
    out["r1000_stride"] = STRIDE
    out["r1000_A_rows"] = np.ascontiguousarray(r.A[::STRIDE])
    out["r1000_E_rows"] = np.ascontiguousarray(r.E[::STRIDE])
    out["r1000_A_colsum"], out["r1000_E_colsum"] = r.A.sum(axis=0), r.E.sum(axis=0)
    out["r1000_A_fro"], out["r1000_E_fro"] = np.linalg.norm(r.A), np.linalg.norm(r.E)
    out["r1000_S"], out["r1000_hist"] = r.s.S, r.hist
    print(f"rpca 3000x1000: {time.time() - t0:.0f} s", flush=True)
    t0 = time.time()
    y, yn = T.synth.sinusoid_np(50_000, seed=6)
    H = O.hankel(yn, 2000)
    res = O.rpca(H, tol=1e-3)
    out["lrf50k_yf"] = O.unhankel_fast(res.A)
    out["lrf50k_iters"], out["lrf50k_sv"], out["lrf50k_hist"] = res.iters, res.sv, res.hist
    print(f"lowrankfilter 50k (n=2000): {res.iters} iterations, sv {res.sv}, {time.time() - t0:.0f} s", flush=True)
    path = os.path.join(HERE, "oracle_largen.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
