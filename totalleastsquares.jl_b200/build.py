"""Build recipe for libtlsq_b200.so (sm_100a only; nvcc cross-compiles without a GPU).

    python totalleastsquares.jl_b200/build.py [--force] [--verbose]

The shared library is built IN-TREE next to this file (git-ignored, but it travels to the GPU box with the
repository snapshot).  cudart is linked statically and NCCL is dlopen'ed at run time, so the library loads on
machines without a GPU driver (the CPU test-suite checks that it exports every symbol of include/tlsq_b200.h).
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libtlsq_b200.so")
SOURCES = ["gram.cu", "syrk_tma.cu", "eig.cu", "eig_fast.cu", "epilogue.cu", "stream.cu", "stream_tma.cu", "fused.cu", "gemm.cu", "elementwise.cu", "ga.cu", "ga_select.cu", "solver.cu"]
HEADERS = ["common.cuh", "kernels.h", os.path.join("..", "..", "include", "tlsq_b200.h")]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    objs = []
    flags = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "--cudart", "static"] + ARCH
    if verbose:
        flags += ["-Xptxas", "-v"]
    procs = []
    for s in SOURCES:
        obj = os.path.join(CSRC, s.replace(".cu", ".o"))
        objs.append(obj)
        procs.append((s, subprocess.Popen([_nvcc(), "-c", os.path.join(CSRC, s), "-o", obj] + flags,
                                          stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for s, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write(f"--- {s} ---\n{out}\n")
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    cmd = [_nvcc(), "-shared", "-o", LIB] + objs + ["--cudart", "static", "-ldl", "-lpthread", "-lrt"] + ARCH
    subprocess.run(cmd, check=True)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
