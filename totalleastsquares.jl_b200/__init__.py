"""Python host mirror of the TotalLeastSquares.jl robust-PCA interface on top of the B200 C-ABI library.

The reference is a Julia package and Julia is not available in this image, so this module plays the role of the
Julia shim (``julia/TotalLeastSquaresB200.jl``) for tests and benchmarks: same function names, argument meaning,
defaults, return values and error behaviour as

    rpca(D; kwargs...)            -> (A, E, s::SVD, sv)     src/robustPCA.jl:156-239
    rpca_ga(X, r, U; kwargs...)   -> Q                      src/robustPCA.jl:255-306
    lowrankfilter(y, n; kwargs...)-> yf                     src/robustPCA.jl:119-128
    hankel(x, L, lag) / unhankel(A, lag, N, D)              src/robustPCA.jl:76-92 / :28-39, 53-68

All arithmetic happens in ``libtlsq_b200.so`` (hand-written sm_100a CUDA).  There is no CPU fallback: without the
library or without a B200 the calls raise ``TlsqError``.  Inputs may be NumPy arrays (host path: H2D/D2H inside the
C call) or CUDA ``torch`` tensors (device path, zero copies when the tensor is column-major).
"""
from __future__ import annotations

import ctypes as C
import math
import warnings
from typing import NamedTuple, Optional

import numpy as np

from . import _cabi, synth  # noqa: F401
from ._cabi import TlsqError, load  # noqa: F401

__all__ = ["rpca", "rpca_ga", "lowrankfilter", "hankel", "unhankel", "rtls", "tls", "entrywise_trimmed_mean",
           "entrywise_median", "mu_mean", "SVD", "TlsqError", "get_handle",
           "init_distributed", "launch_count", "gram", "eigh", "robust_average", "set_profiling", "get_profile", "PHASES"]


class SVD(NamedTuple):
    """Mirror of Julia's LinearAlgebra.SVD returned as ``s`` by rpca (src/robustPCA.jl:194,238)."""
    U: object
    S: object
    Vt: object

    @property
    def V(self):
        return self.Vt.T


# ------------------------------------------------------------------------------------------------------
# handles
# ------------------------------------------------------------------------------------------------------
_handles: dict = {}
_dist = {"nranks": 1, "rank": 0}


def get_handle(device: Optional[int] = None):
    lib = load()
    if device is None:
        device = _default_device()
    h = _handles.get(device)
    if h is None:
        hp = C.c_void_p()
        _cabi.check(lib.tlsq_create(int(device), C.byref(hp)))
        h = hp
        _handles[device] = h
    return h


def _default_device() -> int:
    try:
        import torch
        if torch.cuda.is_available():
            return torch.cuda.current_device()
    except Exception:
        pass
    return 0


def launch_count(device: Optional[int] = None) -> int:
    """Number of CUDA kernels this process launched through the handle (bench.py's gpu_launches)."""
    return int(load().tlsq_launch_count(get_handle(device)))


PHASES = ("gram", "eig", "epilogue", "exact_cost", "init", "finalize", "allreduce", "ga_sweep", "fused")


def set_profiling(on: bool, device: Optional[int] = None) -> None:
    """Switch the library's per-phase CUDA-event timing on/off (resets the accumulators)."""
    _cabi.check(load().tlsq_set_profiling(get_handle(device), 1 if on else 0))


def get_profile(device: Optional[int] = None) -> dict:
    """{phase: (milliseconds, spans)} accumulated since set_profiling(True)."""
    ms = (C.c_double * len(PHASES))()
    calls = (C.c_int64 * len(PHASES))()
    _cabi.check(load().tlsq_get_profile(get_handle(device), ms, calls))
    return {name: (float(ms[i]), int(calls[i])) for i, name in enumerate(PHASES)}


def init_distributed(device: Optional[int] = None) -> None:
    """Attach an NCCL communicator to this rank's handle.  torch.distributed must be initialised; it is used only to
    ship the 128-byte NCCL id from rank 0.  Afterwards rpca / rpca_ga treat their input as this rank's row shard."""
    import torch
    import torch.distributed as dist
    lib = load()
    h = get_handle(device)
    nranks, rank = dist.get_world_size(), dist.get_rank()
    ident = (C.c_ubyte * 128)()
    if rank == 0:
        _cabi.check(lib.tlsq_comm_unique_id(ident))
    dev = torch.device("cuda", _default_device() if device is None else device) \
        if dist.get_backend() == "nccl" else torch.device("cpu")
    t = torch.tensor(list(bytes(ident)), dtype=torch.uint8, device=dev)
    dist.broadcast(t, src=0)
    buf = (C.c_ubyte * 128)(*t.cpu().tolist())
    _cabi.check(lib.tlsq_comm_init(h, nranks, rank, buf))
    _dist["nranks"], _dist["rank"] = nranks, rank


def _global_rows(m_local: int) -> int:
    if _dist["nranks"] == 1:
        return m_local
    import torch
    import torch.distributed as dist
    dev = torch.device("cuda", _default_device()) if dist.get_backend() == "nccl" else torch.device("cpu")
    t = torch.tensor([m_local], dtype=torch.int64, device=dev)
    dist.all_reduce(t)
    return int(t.item())


# ------------------------------------------------------------------------------------------------------
# array plumbing (NumPy host arrays or torch CUDA tensors, always column-major like Julia)
# ------------------------------------------------------------------------------------------------------
def _is_torch(x) -> bool:
    return type(x).__module__.startswith("torch")


class _Arr:
    """Column-major view of a 1-D / 2-D float64 array: pointer + an owner object that keeps it alive."""

    def __init__(self, x, name: str):
        self.torch = _is_torch(x)
        if self.torch:
            import torch
            if x.dtype != torch.float64:
                raise TypeError(f"{name}: only Float64 is accelerated (got {x.dtype}); there is no CPU fallback")
            if not x.is_cuda:
                raise TypeError(f"{name}: torch tensors must live on the GPU (pass a NumPy array for host data)")
            if x.dim() == 2:
                xt = x.t()
                if not xt.is_contiguous():               # not column-major: one transposing copy
                    xt = xt.contiguous()
                x = xt.t()
            elif x.dim() == 1:
                x = x.contiguous()
            self.obj = x
            self.ptr = C.c_void_p(x.data_ptr())
            self.shape = tuple(x.shape)
            self.device = x.device.index if x.device.index is not None else 0
        else:
            a = np.asarray(x)
            if a.dtype != np.float64:
                if np.issubdtype(a.dtype, np.integer) or np.issubdtype(a.dtype, np.bool_):
                    a = a.astype(np.float64)
                else:
                    raise TypeError(f"{name}: only Float64 is accelerated (got {a.dtype}); there is no CPU fallback")
            a = np.asfortranarray(a)
            self.obj = a
            self.ptr = C.c_void_p(a.ctypes.data)
            self.shape = a.shape
            self.device = None


def _empty_like(ref: _Arr, shape):
    """Uninitialised column-major output of the same kind (NumPy / torch CUDA) as `ref`."""
    if ref.torch:
        import torch
        if len(shape) == 2:
            t = torch.empty((shape[1], shape[0]), dtype=torch.float64, device=ref.obj.device).t()
        else:
            t = torch.empty(shape, dtype=torch.float64, device=ref.obj.device)
        return t, C.c_void_p(t.data_ptr())
    a = np.empty(shape, dtype=np.float64, order="F")
    return a, C.c_void_p(a.ctypes.data)


def _handle_for(arr: _Arr):
    lib = load()
    if arr.torch:
        import torch
        h = get_handle(arr.device)
        _cabi.check(lib.tlsq_set_stream(h, C.c_void_p(torch.cuda.current_stream(arr.device).cuda_stream)))
        return h
    h = get_handle(None)
    _cabi.check(lib.tlsq_use_own_stream(h))
    return h


# ------------------------------------------------------------------------------------------------------
# rpca
# ------------------------------------------------------------------------------------------------------
def rpca(D, *, lam: Optional[float] = None, maxrank: Optional[int] = None, iters: int = 1000,
         tol: Optional[float] = None, rho: float = 1.5, verbose: bool = False, nonnegA: bool = False,
         nonnegE: bool = False, hankel: bool = False, nukeA: bool = True, svd=None, opnorm=None,
         return_info: bool = False, want_svd: bool = True, want_E: bool = True, exact_cost: bool = False,
         out=None, **kwargs):
    """``A, E, s, sv = rpca(D; lam, maxrank, iters, tol, rho, verbose, nonnegA, nonnegE, hankel, nukeA)``.

    Drop-in for src/robustPCA.jl:156-239 (``lam`` is the reference's ``λ``, ``rho`` its ``ρ``; the Greek names are
    accepted too).  Unknown keyword arguments are swallowed like the reference does (:170).  Non-default ``svd`` /
    ``opnorm`` callables cannot cross the C ABI and raise (no CPU fallback).  With an attached communicator
    (``init_distributed``) ``D`` is this rank's contiguous row shard.
    """
    lam = kwargs.pop("λ", lam)
    rho = kwargs.pop("ρ", rho)
    if svd is not None or opnorm is not None:
        # the reference's plugin hooks (:168-169): the callables run on the host, the rest of the iteration on the GPU
        return _rpca_callables(D, svd, opnorm, lam=lam, maxrank=maxrank, iters=iters, tol=tol, rho=rho, verbose=verbose,
                               nonnegA=nonnegA, nonnegE=nonnegE, hankel=hankel, nukeA=nukeA, return_info=return_info,
                               want_svd=want_svd)
    f32 = _as_float32_request(D)
    if f32 is not None:
        # Float32 inputs (reference: rpca(D::Matrix{Float32})): computed in Float64 on the GPU, returned as Float32
        res = rpca(f32, lam=lam, maxrank=maxrank, iters=iters, tol=tol if tol is not None else
                   math.sqrt(float(np.finfo(np.float32).eps)), rho=rho, verbose=verbose, nonnegA=nonnegA, nonnegE=nonnegE,
                   hankel=hankel, nukeA=nukeA, return_info=return_info, want_svd=want_svd, want_E=want_E,
                   exact_cost=exact_cost)
        return _cast_result_float32(res)
    lib = load()
    Da = _Arr(D, "D")
    if len(Da.shape) != 2:
        raise TypeError("rpca: D must be a matrix")
    M, N = Da.shape
    Mg = _global_rows(M)
    if lam is None:
        lam = 1.0 / math.sqrt(max(Mg, N))                                    # :157
    if tol is None:
        tol = math.sqrt(np.finfo(np.float64).eps)                            # :160
    d = min(Mg, N)
    flags = (_cabi.TLSQ_NONNEG_A if nonnegA else 0) | (_cabi.TLSQ_NONNEG_E if nonnegE else 0) | \
            (_cabi.TLSQ_HANKEL if hankel else 0) | (0 if nukeA else _cabi.TLSQ_NO_NUKE_A) | \
            (_cabi.TLSQ_EXACT_COST if (verbose or exact_cost) else 0)
    h = _handle_for(Da)
    if out is not None:                      # caller-provided (e.g. pinned) column-major outputs (A, E)
        Ao, Eo = _Arr(out[0], "out[0]"), (_Arr(out[1], "out[1]") if out[1] is not None else None)
        if Ao.obj is not out[0] or tuple(Ao.shape) != (M, N) or Ao.torch != Da.torch:
            raise ValueError("rpca: out[0] must be a column-major float64 M x N array of the same kind as D")
        A, pA = Ao.obj, Ao.ptr
        E, pE = (Eo.obj, Eo.ptr) if Eo is not None else (None, None)
        if Eo is not None and (Eo.obj is not out[1] or tuple(Eo.shape) != (M, N)):
            raise ValueError("rpca: out[1] must be a column-major float64 M x N array")
    else:
        A, pA = _empty_like(Da, (M, N))
        E, pE = _empty_like(Da, (M, N)) if want_E else (None, None)
    if want_svd and out is not None and len(out) == 5:
        # caller-provided (e.g. pinned) buffers for the SVD as well: out = (A, E, U, S, Vt)
        Uo, So, Vo = _Arr(out[2], "out[2]"), _Arr(out[3], "out[3]"), _Arr(out[4], "out[4]")
        if Uo.obj is not out[2] or tuple(Uo.shape) != (M, d) or So.obj is not out[3] or tuple(So.shape) != (d,) or \
                Vo.obj is not out[4] or tuple(Vo.shape) != (d, N):
            raise ValueError("rpca: out[2:5] must be column-major float64 arrays of shapes (M, d), (d,), (d, N)")
        (U, pU), (S, pS), (Vt, pVt) = (Uo.obj, Uo.ptr), (So.obj, So.ptr), (Vo.obj, Vo.ptr)
    elif want_svd:
        U, pU = _empty_like(Da, (M, d))
        S, pS = _empty_like(Da, (d,))
        Vt, pVt = _empty_like(Da, (d, N))
    else:
        U = S = Vt = None
        pU = pS = pVt = None
    sv = C.c_int64(0)
    its = C.c_int64(0)
    conv = C.c_int32(0)
    hist = np.zeros((max(int(iters), 1), 3), dtype=np.float64)
    fn = lib.tlsq_rpca_f64_dev if Da.torch else lib.tlsq_rpca_f64
    _cabi.check(fn(h, Da.ptr, M, N, float(lam), int(maxrank) if maxrank is not None else 0, int(iters), float(tol),
                   float(rho), flags, pA, pE, pU, pS, pVt, C.byref(sv), C.byref(its), C.byref(conv),
                   C.c_void_p(hist.ctypes.data)))
    k = int(its.value)
    hist = hist[:k]
    if verbose:                                                              # :226,229
        for row in hist:
            print(f"{int(row[0])} cost: {abs(row[2]):.4g}")
        if conv.value:
            print("converged")
    if not conv.value:                                                       # :232
        warnings.warn(f"Maximum number of iterations reached, cost: {abs(hist[-1, 2]) if k else float('nan')}, "
                      f"tol: {tol}")
    s = SVD(U, S, Vt) if want_svd else None
    if return_info:
        return A, E, s, int(sv.value), {"iters": k, "converged": bool(conv.value), "hist": hist}
    return A, E, s, int(sv.value)



# ------------------------------------------------------------------------------------------------------
# Float32 promotion and the plugin callables of rpca
# ------------------------------------------------------------------------------------------------------
def _as_float32_request(x):
    """Float64 copy of a Float32 NumPy array / CUDA tensor (None for anything else)."""
    if _is_torch(x):
        import torch
        return x.double() if x.dtype == torch.float32 else None
    a = np.asarray(x)
    return np.asfortranarray(a.astype(np.float64)) if a.dtype == np.float32 else None


def _cast_result_float32(res):
    def cast(v):
        if v is None or isinstance(v, (int, dict)):
            return v
        if isinstance(v, SVD):
            return SVD(cast(v.U), cast(v.S), cast(v.Vt))
        return v.float() if _is_torch(v) else np.asarray(v, dtype=np.float32, order="F")
    return tuple(cast(v) for v in res) if isinstance(res, tuple) else cast(res)


def _rpca_callables(D, svd, opnorm, *, lam, maxrank, iters, tol, rho, verbose, nonnegA, nonnegE, hankel, nukeA,
                    return_info, want_svd):
    """rpca(D; svd=f, opnorm=g): `f(Z, sv)` returns an object with fields U, S, Vt (or a (U, S, Vt) tuple) -- possibly
    truncated --, `g(Z)` a real number (src/robustPCA.jl:168-169, 177, 193-197, 225; test/runtests.jl:384-398)."""
    lib = load()
    Dn = np.asfortranarray(np.asarray(D.detach().cpu().numpy() if _is_torch(D) else D, dtype=np.float64))
    if Dn.ndim != 2:
        raise TypeError("rpca: D must be a matrix")
    M, N = Dn.shape
    d = min(M, N)
    if lam is None:
        lam = 1.0 / math.sqrt(max(M, N))
    if tol is None:
        tol = math.sqrt(np.finfo(np.float64).eps)
    errors = []

    def svd_tramp(_user, Zp, m, n, sv, Up, Sp, Vtp):
        try:
            Z = np.ctypeslib.as_array(Zp, shape=(n, m)).T                      # column-major M x N view
            res = svd(Z, int(sv))
            U, S, Vt = (res.U, res.S, res.Vt) if hasattr(res, "Vt") else res
            U, S, Vt = np.asarray(U, dtype=np.float64), np.asarray(S, dtype=np.float64), np.asarray(Vt, dtype=np.float64)
            r = int(min(S.shape[0], min(m, n)))
            np.ctypeslib.as_array(Up, shape=(r, m))[:] = U[:, :r].T             # M x r, column-major
            np.ctypeslib.as_array(Sp, shape=(r,))[:] = S[:r]
            np.ctypeslib.as_array(Vtp, shape=(n, r))[:] = Vt[:r, :].T           # r x N, leading dimension r
            return r
        except Exception as exc:                                                # noqa: BLE001 - re-raised after the C call
            errors.append(exc)
            return -1

    def opn_tramp(_user, Zp, m, n):
        try:
            return float(opnorm(np.ctypeslib.as_array(Zp, shape=(n, m)).T))
        except Exception as exc:                                                # noqa: BLE001
            errors.append(exc)
            return float("nan")

    svd_c = _cabi.SVD_FN(svd_tramp) if svd is not None else C.cast(None, _cabi.SVD_FN)
    opn_c = _cabi.OPNORM_FN(opn_tramp) if opnorm is not None else C.cast(None, _cabi.OPNORM_FN)
    flags = (_cabi.TLSQ_NONNEG_A if nonnegA else 0) | (_cabi.TLSQ_NONNEG_E if nonnegE else 0) | \
            (_cabi.TLSQ_HANKEL if hankel else 0) | (0 if nukeA else _cabi.TLSQ_NO_NUKE_A)
    A = np.empty((M, N), order="F"); E = np.empty((M, N), order="F")
    U = np.empty((M, d), order="F") if want_svd else None
    S = np.empty((d,)) if want_svd else None
    Vt = np.empty((d, N), order="F") if want_svd else None
    p = lambda a: C.c_void_p(a.ctypes.data) if a is not None else None          # noqa: E731
    sv, its, conv = C.c_int64(0), C.c_int64(0), C.c_int32(0)
    hist = np.zeros((max(int(iters), 1), 3))
    h = get_handle(None)
    _cabi.check(lib.tlsq_use_own_stream(h))
    code = lib.tlsq_rpca_cb_f64(h, p(Dn), M, N, float(lam), int(maxrank) if maxrank is not None else 0, int(iters),
                                float(tol), float(rho), flags, svd_c, opn_c, None, p(A), p(E), p(U), p(S), p(Vt),
                                C.byref(sv), C.byref(its), C.byref(conv), C.c_void_p(hist.ctypes.data))
    if errors:
        raise errors[0]
    _cabi.check(code)
    k = int(its.value)
    if verbose:
        for row in hist[:k]:
            print(f"{int(row[0])} cost: {abs(row[2]):.4g}")
        if conv.value:
            print("converged")
    if not conv.value:
        warnings.warn(f"Maximum number of iterations reached, cost: {abs(hist[k - 1, 2]) if k else float('nan')}, tol: {tol}")
    s = SVD(U, S, Vt) if want_svd else None
    if return_info:
        return A, E, s, int(sv.value), {"iters": k, "converged": bool(conv.value), "hist": hist[:k]}
    return A, E, s, int(sv.value)

# ------------------------------------------------------------------------------------------------------
# lowrankfilter / hankel / unhankel
# ------------------------------------------------------------------------------------------------------
def lowrankfilter(y, n: Optional[int] = None, *, sv: int = 0, lag: int = 1, tol: float = 1e-3, svd=None,
                  lam: Optional[float] = None, maxrank: Optional[int] = None, iters: int = 1000, rho: float = 1.5,
                  verbose: bool = False, nonnegA: bool = False, nonnegE: bool = False, hankel: bool = False,
                  nukeA: bool = True, opnorm=None, return_info: bool = False, **kwargs):
    """``yf = lowrankfilter(y, n=min(length(y) ÷ 20, 2000); lag=1, tol=1e-3, kwargs...)`` (src/robustPCA.jl:119-128).
    The Hankel embedding is indexed implicitly on the GPU and never materialised."""
    lam = kwargs.pop("λ", lam)
    rho = kwargs.pop("ρ", rho)
    if svd is not None or opnorm is not None:
        # plugin callables (test/runtests.jl:384-398): the reference's own composition (:120-127) with rpca on the
        # materialised trajectory matrix -- the callables need the whole matrix on the host anyway
        yn = np.asarray(y.detach().cpu().numpy() if _is_torch(y) else y, dtype=np.float64)
        Ns0 = yn.shape[0]
        Dch0 = 1 if yn.ndim == 1 else yn.shape[1]
        n0 = min(Ns0 // 20, 2000) if n is None else n
        A = rpca(globals()["hankel"](yn, n0, lag), lam=lam, maxrank=maxrank, iters=iters, tol=tol, rho=rho,
                 verbose=verbose, nonnegA=nonnegA, nonnegE=nonnegE, hankel=hankel, nukeA=nukeA, svd=svd, opnorm=opnorm,
                 want_svd=False)[0]
        return unhankel(A, lag, Ns0, Dch0)
    f32 = _as_float32_request(y)
    if f32 is not None:
        return _cast_result_float32(lowrankfilter(f32, n, sv=sv, lag=lag, tol=tol, lam=lam, maxrank=maxrank, iters=iters,
                                                  rho=rho, verbose=verbose, nonnegA=nonnegA, nonnegE=nonnegE,
                                                  hankel=hankel, nukeA=nukeA, return_info=return_info))
    ya = _Arr(y, "y")
    Dch = 1 if len(ya.shape) == 1 else int(ya.shape[1])
    Ns = ya.shape[0]
    if n is None:
        n = min(Ns // 20, 2000)                                              # :119
    if n > Ns / 2:
        raise AssertionError(f"L has to be less than N/2 = {Ns / 2}")        # :79
    if lag > n:
        raise AssertionError("lag must be <= L")                             # :80
    lib = load()
    h = _handle_for(ya)
    flags = (_cabi.TLSQ_NONNEG_A if nonnegA else 0) | (_cabi.TLSQ_NONNEG_E if nonnegE else 0) | \
            (_cabi.TLSQ_HANKEL if hankel else 0) | (0 if nukeA else _cabi.TLSQ_NO_NUKE_A) | \
            (_cabi.TLSQ_EXACT_COST if verbose else 0)
    yf, pyf = _empty_like(ya, (Ns,) if len(ya.shape) == 1 else (Ns, Dch))
    svo = C.c_int64(0)
    its = C.c_int64(0)
    conv = C.c_int32(0)
    hist = np.zeros((max(int(iters), 1), 3), dtype=np.float64)
    if Dch == 1 and sv <= 0:
        fn = lib.tlsq_lowrankfilter_f64_dev if ya.torch else lib.tlsq_lowrankfilter_f64
        _cabi.check(fn(h, ya.ptr, Ns, int(n), int(lag), float(lam) if lam is not None else 0.0,
                       int(maxrank) if maxrank is not None else 0, int(iters), float(tol), float(rho), flags, pyf,
                       C.byref(svo), C.byref(its), C.byref(conv), C.c_void_p(hist.ctypes.data)))
    else:
        # channels (:83-90, :53-68) and / or the sv > 0 plain-SSA branch (:123-125)
        fn = lib.tlsq_lowrankfilter_mc_f64_dev if ya.torch else lib.tlsq_lowrankfilter_mc_f64
        _cabi.check(fn(h, ya.ptr, Ns, Dch, int(n), int(lag), int(sv), float(lam) if lam is not None else 0.0,
                       int(maxrank) if maxrank is not None else 0, int(iters), float(tol), float(rho), flags, pyf,
                       C.byref(svo), C.byref(its), C.byref(conv), C.c_void_p(hist.ctypes.data)))
    k = int(its.value)
    if verbose:
        for row in hist[:k]:
            print(f"{int(row[0])} cost: {abs(row[2]):.4g}")
        if conv.value:
            print("converged")
    if not conv.value:
        warnings.warn(f"Maximum number of iterations reached, cost: {abs(hist[k - 1, 2]) if k else float('nan')}, "
                      f"tol: {tol}")
    if return_info:
        return yf, {"iters": k, "converged": bool(conv.value), "sv": int(svo.value), "hist": hist[:k]}
    return yf


def hankel(x, L: int, lag: int = 1):
    """``X = hankel(x, L, lag=1)``: K x (L D) trajectory matrix of an N (x D) signal, K = (N-L)÷lag+1
    (src/robustPCA.jl:76-92)."""
    xa = _Arr(np.asarray(x, dtype=np.float64) if not _is_torch(x) else x.detach().cpu().numpy(), "x")
    Ns = xa.shape[0]
    D = 1 if len(xa.shape) == 1 else int(xa.shape[1])
    if L > Ns / 2:
        raise AssertionError(f"L has to be less than N/2 = {Ns / 2}")
    if lag > L:
        raise AssertionError("lag must be <= L")
    K = (Ns - L) // lag + 1
    H = np.empty((K, L * D), dtype=np.float64, order="F")
    if D == 1:
        _cabi.check(load().tlsq_hankel_f64(get_handle(None), xa.ptr, Ns, int(L), int(lag), C.c_void_p(H.ctypes.data)))
    else:
        _cabi.check(load().tlsq_hankel_mc_f64(get_handle(None), xa.ptr, Ns, D, int(L), int(lag),
                                              C.c_void_p(H.ctypes.data)))
    return H


def unhankel(A, lag: int = 1, N: Optional[int] = None, D: int = 1):
    """``unhankel(A)`` / ``unhankel(A, lag, N, D=1)``: anti-diagonal averaging (src/robustPCA.jl:28-39, 53-68)."""
    Aa = _Arr(np.asarray(A, dtype=np.float64) if not _is_torch(A) else A.detach().cpu().numpy(), "A")
    K, LD = Aa.shape
    L = LD // int(D)
    if N is None:
        N = L + (K - 1) * lag
    if D == 1:
        y = np.empty(int(N), dtype=np.float64)
        _cabi.check(load().tlsq_unhankel_f64(get_handle(None), Aa.ptr, K, L, int(lag), int(N),
                                             C.c_void_p(y.ctypes.data)))
    else:
        y = np.empty((int(N), int(D)), dtype=np.float64, order="F")
        _cabi.check(load().tlsq_unhankel_mc_f64(get_handle(None), Aa.ptr, K, L, int(lag), int(N), int(D),
                                                C.c_void_p(y.ctypes.data)))
    return y


# ------------------------------------------------------------------------------------------------------
# rpca_ga
# ------------------------------------------------------------------------------------------------------
def mu_mean(*_a, **_k):
    """Tag for the default average ``μ!`` (src/robustPCA.jl:308-316) in ``rpca_ga(...; μ=...)``."""
    raise NotImplementedError("pass it as rpca_ga(X, r, mu=mu_mean); the average itself runs on the GPU")


def entrywise_trimmed_mean(*_a, **_k):
    """Tag for ``entrywise_trimmed_mean(s, w, U, P=0.1)`` (src/robustPCA.jl:323-333): ``rpca_ga(X, r, mu=entrywise_trimmed_mean)``
    or ``mu=(entrywise_trimmed_mean, P)``; the per-row sort runs on the GPU (ga.cu)."""
    raise NotImplementedError("pass it as rpca_ga(X, r, mu=entrywise_trimmed_mean); the average itself runs on the GPU")


def entrywise_median(*_a, **_k):
    """Tag for ``entrywise_median(s, w, U)`` (src/robustPCA.jl:349-357): ``rpca_ga(X, r, mu=entrywise_median)``."""
    raise NotImplementedError("pass it as rpca_ga(X, r, mu=entrywise_median); the average itself runs on the GPU")


def rpca_ga(X, r: Optional[int] = None, U=None, *, verbose: bool = False, tol: float = 1e-7, iters: int = 1000,
            mu=None, q0=None, return_info: bool = False, **kwargs):
    """``Q = rpca_ga(X, r=minimum(size(X)), U=similar(X); tol=1e-7, iters=1000)`` (src/robustPCA.jl:255-306).

    Columns of ``X`` are observations.  The start vector of every component is drawn here with ``randn(d)`` from the
    global NumPy RNG (the reference draws from Julia's global RNG, :286) unless ``q0`` (d x r) is given.  The optional
    buffer ``U`` is accepted for signature compatibility; the normalised copy is never formed on the GPU.
    """
    mu = kwargs.pop("μ", mu)
    mu_kind, mu_p = 0, 0.1
    if mu is not None and mu is not mu_mean:
        # the reference's pluggable averages (keyword μ, :255,294) map to device kernels; other callables cannot cross
        # the C ABI
        if mu is entrywise_trimmed_mean or mu == "entrywise_trimmed_mean":
            mu_kind = 1
        elif mu is entrywise_median or mu == "entrywise_median":
            mu_kind = 2
        elif isinstance(mu, tuple) and mu and mu[0] is entrywise_trimmed_mean:          # (entrywise_trimmed_mean, P)
            mu_kind, mu_p = 1, float(mu[1])
        else:
            raise NotImplementedError("rpca_ga: only mu!, entrywise_trimmed_mean and entrywise_median are accelerated; "
                                      "arbitrary callables cannot cross the C ABI (no CPU fallback)")
    f32 = _as_float32_request(X)
    if f32 is not None:
        q0d = None if q0 is None else (_as_float32_request(q0) if _as_float32_request(q0) is not None else q0)
        return _cast_result_float32(rpca_ga(f32, r, U, verbose=verbose, tol=tol, iters=iters, mu=mu, q0=q0d,
                                            return_info=return_info))
    Xa = _Arr(X, "X")
    if len(Xa.shape) != 2:
        raise TypeError("rpca_ga: X must be a matrix")
    d, N = Xa.shape
    dg = _global_rows(d)
    if r is None:
        r = min(dg, N)
    r = int(r)
    if q0 is None:
        if _dist["nranks"] > 1:
            raise ValueError("rpca_ga: sharded runs must pass this rank's rows of q0")
        q0 = np.asfortranarray(np.stack([np.random.randn(d) for _ in range(r)], axis=1))   # one randn(d) per component
        if Xa.torch:
            import torch
            q0 = torch.from_numpy(np.ascontiguousarray(q0.T)).to(Xa.obj.device).t()
    q0a = _Arr(q0, "q0")
    if tuple(q0a.shape) != (d, r):
        raise ValueError(f"rpca_ga: q0 must be {d} x {r}")
    if q0a.torch != Xa.torch:
        raise TypeError("rpca_ga: X and q0 must both be NumPy arrays or both CUDA tensors")
    lib = load()
    h = _handle_for(Xa)
    Q, pQ = _empty_like(Xa, (d, r))
    its = (C.c_int64 * r)()
    if mu_kind == 0:
        fn = lib.tlsq_rpca_ga_f64_dev if Xa.torch else lib.tlsq_rpca_ga_f64
        _cabi.check(fn(h, Xa.ptr, d, N, r, q0a.ptr, float(tol), int(iters), pQ, its))
    else:
        fn = lib.tlsq_rpca_ga_mu_f64_dev if Xa.torch else lib.tlsq_rpca_ga_mu_f64
        _cabi.check(fn(h, Xa.ptr, d, N, r, q0a.ptr, float(tol), int(iters), mu_kind, mu_p, pQ, its))
    its = [int(v) for v in its]
    if verbose:
        for i, v in enumerate(its):
            print(f"component {i + 1}: {v} iterations")
    if any(v >= iters for v in its):
        warnings.warn("Reached maximum number of iterations")                # :303
    if return_info:
        return Q, {"iters": its}
    return Q


# ------------------------------------------------------------------------------------------------------
# building blocks (tests / profiling)
# ------------------------------------------------------------------------------------------------------
# ----------------------------------------------------------------------------------------------------------
# rtls: the in-package caller of rpca that consumes the returned SVD (src/TotalLeastSquares.jl:48-69, 152-156)
# ----------------------------------------------------------------------------------------------------------
def _tls_from_v(V, n: int):
    """tls!(s::SVD, n): x = -V21 / V22 with V = s.V (src/TotalLeastSquares.jl:65-69).  Tiny host-side solve."""
    V = np.asarray(V.cpu().numpy() if _is_torch(V) else V)
    V21, V22 = V[:n, n:], V[n:, n:]
    return -np.linalg.solve(V22.T, V21.T).T                        # V21 / V22  (right division)


def tls(A, y):
    """``x = tls(A, y)``: total least squares by the SVD of [A y] (src/TotalLeastSquares.jl:48-55); host NumPy -- not
    part of the accelerated path, provided because rtls (below) is defined through it."""
    A = np.asarray(A, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64).reshape(A.shape[0], -1)
    _, _, Vt = np.linalg.svd(np.hstack([A, y]), full_matrices=False)
    return _tls_from_v(Vt.T, A.shape[1])


def rtls(A, y, **kwargs):
    """``x = rtls(A, y; kwargs...)``: robust TLS = rpca([A y]; nukeA=false, kwargs...) on the GPU followed by tls! on
    the returned SVD (src/TotalLeastSquares.jl:152-156)."""
    A = np.asarray(A, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64).reshape(A.shape[0], -1)
    kwargs.setdefault("nukeA", False)
    _, _, s, _ = rpca(np.asfortranarray(np.hstack([A, y])), **kwargs)
    return _tls_from_v(np.asarray(s.Vt).T, A.shape[1])


def gram(X):
    """G = X'X through the DMMA SYRK kernel (X: CUDA float64 tensor, column-major)."""
    import torch
    Xa = _Arr(X, "X")
    if not Xa.torch:
        raise TypeError("gram: pass a CUDA tensor")
    M, n = Xa.shape
    G = torch.empty((n, n), dtype=torch.float64, device=Xa.obj.device)
    _cabi.check(load().tlsq_gram_f64_dev(_handle_for(Xa), Xa.ptr, M, n, C.c_void_p(G.data_ptr())))
    return G


def eigh(G):
    """(lam, V) of a symmetric PSD CUDA tensor through the Jacobi kernels; lam descending, V columns."""
    import torch
    Ga = _Arr(G, "G")
    if not Ga.torch:
        raise TypeError("eigh: pass a CUDA tensor")
    n = Ga.shape[0]
    lam = torch.empty((n,), dtype=torch.float64, device=Ga.obj.device)
    Vc = torch.empty((n, n), dtype=torch.float64, device=Ga.obj.device)      # column-major n x n == V' row-major
    _cabi.check(load().tlsq_eigh_f64_dev(_handle_for(Ga), Ga.ptr, n, C.c_void_p(lam.data_ptr()),
                                         C.c_void_p(Vc.data_ptr())))
    return lam, Vc.t()


def robust_average(U, w, mu=entrywise_trimmed_mean, P: float = 0.1):
    """s = mu(s, w, U) for ``mu = entrywise_trimmed_mean`` (fraction ``P``, src/robustPCA.jl:323-333) or
    ``entrywise_median`` (:349-357) through the per-row selection kernels (U: d x N and w: N, CUDA float64 tensors)."""
    import torch
    Ua, wa = _Arr(U, "U"), _Arr(w, "w")
    if not (Ua.torch and wa.torch):
        raise TypeError("robust_average: pass CUDA tensors")
    if len(Ua.shape) != 2 or tuple(wa.shape) != (Ua.shape[1],):
        raise ValueError("robust_average: U must be d x N and w of length N")
    if mu is entrywise_trimmed_mean:
        kind = 1
    elif mu is entrywise_median:
        kind = 2
    else:
        raise NotImplementedError("robust_average: mu must be entrywise_trimmed_mean or entrywise_median")
    d, N = Ua.shape
    s = torch.empty((d,), dtype=torch.float64, device=Ua.obj.device)
    _cabi.check(load().tlsq_robust_average_f64_dev(_handle_for(Ua), Ua.ptr, d, N, wa.ptr, kind, float(P),
                                                   C.c_void_p(s.data_ptr())))
    return s
