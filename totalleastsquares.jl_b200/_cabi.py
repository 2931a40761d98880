"""ctypes binding of libtlsq_b200.so (include/tlsq_b200.h).  No compute happens in Python."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libtlsq_b200.so")

# status codes / flags (mirror of include/tlsq_b200.h)
TLSQ_OK, TLSQ_ERR_ARG, TLSQ_ERR_NO_DEVICE, TLSQ_ERR_CUDA, TLSQ_ERR_NCCL, TLSQ_ERR_UNSUPPORTED, TLSQ_ERR_NOMEM = range(7)
TLSQ_NONNEG_A, TLSQ_NONNEG_E, TLSQ_HANKEL, TLSQ_NO_NUKE_A, TLSQ_EXACT_COST = 1, 2, 4, 8, 16

c_dp = C.POINTER(C.c_double)
c_i64p = C.POINTER(C.c_int64)
c_i32p = C.POINTER(C.c_int32)
vp = C.c_void_p

_RPCA_ARGS = [vp, vp, C.c_int64, C.c_int64, C.c_double, C.c_int64, C.c_int64, C.c_double, C.c_double, C.c_uint32,
              vp, vp, vp, vp, vp, c_i64p, c_i64p, c_i32p, vp]
_LRF_ARGS = [vp, vp, C.c_int64, C.c_int64, C.c_int64, C.c_double, C.c_int64, C.c_int64, C.c_double, C.c_double,
             C.c_uint32, vp, c_i64p, c_i64p, c_i32p, vp]
_LRF_MC_ARGS = [vp, vp, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_double, C.c_int64, C.c_int64,
                C.c_double, C.c_double, C.c_uint32, vp, c_i64p, c_i64p, c_i32p, vp]
_GA_ARGS = [vp, vp, C.c_int64, C.c_int64, C.c_int64, vp, C.c_double, C.c_int64, vp, c_i64p]

# plugin callables (tlsq_svd_fn / tlsq_opnorm_fn of include/tlsq_b200.h)
SVD_FN = C.CFUNCTYPE(C.c_int64, vp, c_dp, C.c_int64, C.c_int64, C.c_int64, c_dp, c_dp, c_dp)
OPNORM_FN = C.CFUNCTYPE(C.c_double, vp, c_dp, C.c_int64, C.c_int64)
_RPCA_CB_ARGS = _RPCA_ARGS[:10] + [SVD_FN, OPNORM_FN, vp] + _RPCA_ARGS[10:]

SIGNATURES = {
    "tlsq_abi_version": (C.c_int, []),
    "tlsq_last_error": (C.c_char_p, []),
    "tlsq_device_count": (C.c_int, []),
    "tlsq_create": (C.c_int, [C.c_int, C.POINTER(vp)]),
    "tlsq_destroy": (C.c_int, [vp]),
    "tlsq_set_stream": (C.c_int, [vp, vp]),
    "tlsq_use_own_stream": (C.c_int, [vp]),
    "tlsq_launch_count": (C.c_int64, [vp]),
    "tlsq_set_profiling": (C.c_int, [vp, C.c_int]),
    "tlsq_get_profile": (C.c_int, [vp, c_dp, c_i64p]),
    "tlsq_comm_unique_id": (C.c_int, [vp]),
    "tlsq_comm_init": (C.c_int, [vp, C.c_int, C.c_int, vp]),
    "tlsq_rpca_f64": (C.c_int, _RPCA_ARGS),
    "tlsq_rpca_f64_dev": (C.c_int, _RPCA_ARGS),
    "tlsq_rpca_cb_f64": (C.c_int, _RPCA_CB_ARGS),
    "tlsq_lowrankfilter_f64": (C.c_int, _LRF_ARGS),
    "tlsq_lowrankfilter_f64_dev": (C.c_int, _LRF_ARGS),
    "tlsq_rpca_ga_f64": (C.c_int, _GA_ARGS),
    "tlsq_rpca_ga_f64_dev": (C.c_int, _GA_ARGS),
    "tlsq_rpca_ga_mu_f64": (C.c_int, [vp, vp, C.c_int64, C.c_int64, C.c_int64, vp, C.c_double, C.c_int64, C.c_int,
                                      C.c_double, vp, c_i64p]),
    "tlsq_rpca_ga_mu_f64_dev": (C.c_int, [vp, vp, C.c_int64, C.c_int64, C.c_int64, vp, C.c_double, C.c_int64, C.c_int,
                                          C.c_double, vp, c_i64p]),
    "tlsq_hankel_f64": (C.c_int, [vp, vp, C.c_int64, C.c_int64, C.c_int64, vp]),
    "tlsq_unhankel_f64": (C.c_int, [vp, vp, C.c_int64, C.c_int64, C.c_int64, C.c_int64, vp]),
    "tlsq_lowrankfilter_mc_f64": (C.c_int, _LRF_MC_ARGS),
    "tlsq_lowrankfilter_mc_f64_dev": (C.c_int, _LRF_MC_ARGS),
    "tlsq_hankel_mc_f64": (C.c_int, [vp, vp, C.c_int64, C.c_int64, C.c_int64, C.c_int64, vp]),
    "tlsq_unhankel_mc_f64": (C.c_int, [vp, vp, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int64, vp]),
    "tlsq_plan_pipeline": (C.c_int, [C.c_int, c_dp, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int),
                                     C.POINTER(C.c_int)]),
    "tlsq_plan_fused_strips": (C.c_int, [vp, vp]),
    "tlsq_plan_hankel_shard": (C.c_int, [C.c_int64, C.c_int, C.c_int, c_i64p, c_i64p]),
    "tlsq_plan_syrk": (C.c_int, [C.c_int64, C.c_int64, C.c_int, vp, vp, vp, vp, vp, c_i64p]),
    "tlsq_gram_f64_dev": (C.c_int, [vp, vp, C.c_int64, C.c_int64, vp]),
    "tlsq_eigh_f64_dev": (C.c_int, [vp, vp, C.c_int64, vp, vp]),
    "tlsq_robust_average_f64_dev": (C.c_int, [vp, vp, C.c_int64, C.c_int64, vp, C.c_int, C.c_double, vp]),
}


class TlsqError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"tlsq_b200 error {code}: {msg}")
        self.code = code


_lib = None


def _find_nccl() -> None:
    """Point the library's dlopen at the NCCL that ships with torch unless the user chose one."""
    if os.environ.get("TLSQ_NCCL_LIB"):
        return
    try:
        import importlib.util
        spec = importlib.util.find_spec("nvidia.nccl")
        if spec and spec.submodule_search_locations:
            cand = os.path.join(list(spec.submodule_search_locations)[0], "lib", "libnccl.so.2")
            if os.path.exists(cand):
                os.environ["TLSQ_NCCL_LIB"] = cand
    except Exception:
        pass


def load() -> C.CDLL:
    """Load the CUDA library.  There is NO fallback: a missing library is an error."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise TlsqError(-1, f"{LIB_PATH} is missing: build it with `python {os.path.join(HERE, 'build.py')}` "
                            "(nvcc, sm_100a).  There is no CPU fallback.")
    _find_nccl()
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(code: int) -> None:
    if code != TLSQ_OK:
        raise TlsqError(code, load().tlsq_last_error().decode("utf-8", "replace"))
