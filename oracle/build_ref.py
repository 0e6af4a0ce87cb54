"""ORACLE tooling (NOT product code): compile the REFERENCE's own CUDA kernels for sm_100a, from the
reference source tree (nothing is copied), into oracle/_ref/ (git-ignored).  `python -m oracle.make_golden --ref-kernels`
runs them on a GPU and stores their outputs as tests/golden/ref_kernels.npz, against which the GPU tests pin FPS
bit-exactness (incl. the tie-break rule) and the nearest-neighbour distance.

Sources compiled: third_party/torkit3d/torkit3d/csrc/cuda/{sample_farthest_points,chamfer_distance}_kernel.cu
with a 10-line pybind shim (oracle/ref_binding.cpp) - the reference's setup.py is not run.
"""
from __future__ import annotations

import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
REF = "/root/reference/third_party/torkit3d/torkit3d/csrc"
OUT = os.path.join(HERE, "_ref")
NAME = "torkit3d_ref_ops"


def built_path():
    if not os.path.isdir(OUT):
        return None
    for f in os.listdir(OUT):
        if f.startswith(NAME) and f.endswith(".so"):
            return os.path.join(OUT, f)
    return None


def build(verbose=False):
    if built_path():
        return built_path()
    if not os.path.isdir(REF):
        return None
    os.makedirs(OUT, exist_ok=True)
    os.environ.setdefault("TORCH_CUDA_ARCH_LIST", "10.0")
    from torch.utils.cpp_extension import load

    load(name=NAME,
         sources=[os.path.join(HERE, "ref_binding.cpp"),
                  os.path.join(REF, "cuda", "sample_farthest_points_kernel.cu"),
                  os.path.join(REF, "cuda", "chamfer_distance_kernel.cu")],
         extra_include_paths=[os.path.join(REF, "include")],
         extra_cuda_cflags=["-gencode", "arch=compute_100a,code=sm_100a", "-O3"],
         build_directory=OUT, verbose=verbose, is_python_module=False)
    for f in os.listdir(OUT):  # keep only the shared object
        if not f.endswith(".so"):
            p = os.path.join(OUT, f)
            shutil.rmtree(p) if os.path.isdir(p) else os.remove(p)
    return built_path()


def load_ref():
    """Import the compiled reference ops (GPU box: uses the prebuilt .so that travelled with the repo)."""
    p = built_path()
    if p is None:
        return None
    import importlib.util

    import torch  # noqa: F401  (libtorch symbols must be loaded first)

    spec = importlib.util.spec_from_file_location(NAME, p)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


if __name__ == "__main__":
    print(build(verbose="-v" in sys.argv))
