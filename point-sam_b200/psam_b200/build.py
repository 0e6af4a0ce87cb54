"""Build libpsam_b200.so (CUDA kernels + C ABI) in-tree for sm_100a with nvcc."""
from __future__ import annotations

import os
import subprocess
from concurrent.futures import ThreadPoolExecutor

PKG = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(PKG, "csrc")
LIBDIR = os.path.join(PKG, "lib")
LIB = os.path.join(LIBDIR, "libpsam_b200.so")
SOURCES = ["fps.cu", "knn.cu", "gemm_tc.cu", "attention_tc.cu", "elementwise.cu", "masks.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "--use_fast_math=false"]


def _newer(target: str, deps) -> bool:
    if not os.path.exists(target):
        return False
    t = os.path.getmtime(target)
    return all(os.path.getmtime(d) <= t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(LIBDIR, exist_ok=True)
    headers = [os.path.join(CSRC, "psam_common.cuh"), os.path.join(os.path.dirname(PKG), "include", "psam_b200.h")]
    flags = [f for f in NVCC_FLAGS if not f.startswith("--use_fast_math")]

    def compile_one(src):
        obj = os.path.join(LIBDIR, src.replace(".cu", ".o"))
        path = os.path.join(CSRC, src)
        if force or not _newer(obj, [path] + headers):
            cmd = ["nvcc", *flags, "-c", path, "-o", obj]
            if verbose:
                print(" ".join(cmd))
            subprocess.check_call(cmd)
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    if force or not _newer(LIB, objs):
        subprocess.check_call(["nvcc", "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a"])
    return LIB


if __name__ == "__main__":
    print(build(verbose=True))
