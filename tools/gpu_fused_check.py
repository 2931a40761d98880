"""Debug driver for the fused one-pass ALM kernel (run on the GPU box): parity against the oracle + against the
two-kernel pipeline (TLSQ_FUSED=0), a few shapes, verbose numbers."""
import os, sys, time, warnings
sys.path.insert(0, '.'); sys.path.insert(0, 'oracle')
import numpy as np
import tls_oracle as O
import tlsq_b200 as T

warnings.simplefilter("ignore")
def relF(a, b): return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))

def case(M, N, r, its, **kw):
    D = T.synth.lowrank_sparse_np(M, N, r, 0.05, seed=M + N, nonneg=bool(kw.get("nonnegA")))
    A, E, s, sv, info = T.rpca(D, iters=its, tol=0.0, return_info=True, **kw)
    ref = O.rpca(D, iters=its, tol=0.0, **kw)
    Wg, Wo = (s.U * s.S) @ s.Vt, (ref.s.U * ref.s.S) @ ref.s.Vt
    print(f"fixed M={M} N={N} r={r} its={its} {kw}: relA={relF(A, ref.A):.2e} relE={relF(E, ref.E):.2e} "
          f"supp={int(np.sum((E != 0) != (ref.E != 0)))} hist_eq={np.array_equal(info['hist'][:,1], ref.hist[:,1])} "
          f"S={np.abs(s.S-ref.s.S).max()/ref.s.S[0]:.2e} W={relF(Wg, Wo):.2e}", flush=True)
    if not np.array_equal(info['hist'][:,1], ref.hist[:,1]):
        print("   svp gpu", info['hist'][:,1].tolist()); print("   svp ref", ref.hist[:,1].tolist())

def conv(M, N, r, **kw):
    D = T.synth.lowrank_sparse_np(M, N, r, 0.05, seed=4, nonneg=bool(kw.get("nonnegA")))
    A, E, s, sv, info = T.rpca(D, return_info=True, **kw)
    ref = O.rpca(D, **kw)
    print(f"conv  M={M} N={N} r={r} {kw}: iters {info['iters']} vs {ref.iters} conv={info['converged']} "
          f"relA={relF(A, ref.A):.2e} relE={relF(E, ref.E):.2e}", flush=True)
    _, _, _, _, info2 = T.rpca(D, return_info=True, exact_cost=True, want_svd=False, **kw)
    print(f"      exact-cost iters {info2['iters']} cost ok={np.allclose(info2['hist'][:,2], ref.hist[:info2['iters'],2], rtol=1e-6) if info2['iters']==ref.iters else None}", flush=True)

os.environ["TLSQ_FUSED"] = "1"
print("fused eligible path", flush=True)
case(8192, 256, 10, 14)
case(20002, 256, 10, 12, nonnegA=True, nonnegE=True)
case(6000, 256, 3, 8, nukeA=False)
case(8000, 256, 20, 12)          # svp > 16: leaves the fused path mid-run
conv(20000, 256, 10, nonnegA=True)
conv(12000, 256, 5)
# lowrankfilter through the fused implicit-Hankel path (n = 256)
y, yn = T.synth.sinusoid_np(12255, seed=2, noise=0.05)
t0 = time.time(); yf, info = T.lowrankfilter(yn, 256, return_info=True); t1 = time.time()
yo = O.lowrankfilter(yn, 256)
print(f"lowrankfilter n=256 Ns=12255: rel={relF(yf, yo):.2e} iters={info['iters']} ({t1-t0:.2f}s)", flush=True)
os.environ["TLSQ_INPLACE_Y"] = "1"
yf2, info2 = T.lowrankfilter(yn, 256, return_info=True)
print(f"  in-place Y: rel={relF(yf2, yo):.2e} iters={info2['iters']}", flush=True)
del os.environ["TLSQ_INPLACE_Y"]
os.environ["TLSQ_FUSED"] = "0"
yf3, info3 = T.lowrankfilter(yn, 256, return_info=True)
print(f"  two-kernel path: rel={relF(yf3, yo):.2e} iters={info3['iters']}", flush=True)
os.environ["TLSQ_FUSED"] = "1"
# odd number of Hankel rows on the one-pass path (padded leading dimension of Y / T)
y, yn = T.synth.sinusoid_np(12256, seed=3, noise=0.05)
yo = O.lowrankfilter(yn, 256)
yf, info = T.lowrankfilter(yn, 256, return_info=True)
print(f"lowrankfilter n=256 Ns=12256 (K odd): rel={relF(yf, yo):.2e} iters={info['iters']}", flush=True)
os.environ["TLSQ_INPLACE_Y"] = "1"
yf, info = T.lowrankfilter(yn, 256, return_info=True)
print(f"  in-place Y: rel={relF(yf, yo):.2e} iters={info['iters']}", flush=True)
del os.environ["TLSQ_INPLACE_Y"]
