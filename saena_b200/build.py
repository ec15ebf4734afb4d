"""Builds saena_b200/libsaena_b200.so (CUDA kernels + the C ABI of include/saena_b200.h) in-tree
with nvcc for sm_100a.  nvcc cross-compiles without a GPU; the .so travels to the GPU box."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "libsaena_b200.so")
SOURCES = ["api.cu", "operator.cu", "vector_ops.cu", "solve.cu", "nccl_comm.cu", "p2p_halo.cu", "fused_halo.cu", "fused_restrict.cu", "lanczos.cu", "spgemm.cu", "refresh.cu", "spmv_block.cu", "spmv_f32.cu"]
HEADERS = ["common.h", "spmv_kernels.cuh", "halo_sync.cuh"]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]


def _nccl_include() -> list[str]:
    for d in ("/usr/include", os.path.join(sys.prefix, "lib", f"python{sys.version_info.major}.{sys.version_info.minor}",
                                           "site-packages", "nvidia", "nccl", "include")):
        if os.path.exists(os.path.join(d, "nccl.h")):
            return ["-I", d]
    raise RuntimeError("nccl.h not found")


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.join(ROOT, "include", "saena_b200.h"), __file__]
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return LIB
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: cannot build libsaena_b200.so")
    objdir = os.path.join(PKG, "build")
    os.makedirs(objdir, exist_ok=True)
    common = [nvcc, "-std=c++17", "-O3", "-lineinfo", *ARCH, "-Xcompiler", "-fPIC", "-I", os.path.join(ROOT, "include"),
              "-I", CSRC, *_nccl_include()]
    if verbose:
        common += ["-Xptxas", "-v"]
    procs = []
    objs = []
    for src in SOURCES:
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        objs.append(obj)
        procs.append((src, subprocess.Popen(common + ["-c", os.path.join(CSRC, src), "-o", obj],
                                            stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{out}")
        if verbose and out:
            print(out)
    subprocess.check_call([nvcc, "-shared", *ARCH, "-o", LIB, *objs, "-ldl"])
    return LIB


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
