"""Compile the reference's ONLY native source, demo/quantize_int4.cu, where it lies under
/root/reference, into oracle/_ref/ (git-ignored, travels to the GPU box).  TEST INFRASTRUCTURE ONLY:
the resulting module is the real reference implementation of INT4 quantise/dequantise (kernels K1/K2);
``tests/golden/make_golden.py int4-kernels`` runs it to write the fixture that pins both the NumPy oracle and the
product kernels.

The reference JIT-builds this file with ``torch.utils.cpp_extension.load(extra_cuda_cflags=
["--use_fast_math"])`` (demo/int4_kv.py:46-56); we do the same ahead of time for sm_100a.  No reference
source is copied into the repo — nvcc reads it in place."""
from __future__ import annotations

import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "_ref")
SRC = "/root/reference/demo/quantize_int4.cu"
NAME = "quantize_int4_ref"


def built_path():
    if not os.path.isdir(OUT):
        return None
    for f in os.listdir(OUT):
        if f.startswith(NAME) and f.endswith(".so"):
            return os.path.join(OUT, f)
    return None


def build(verbose=False):
    if not os.path.exists(SRC):
        return built_path()
    if built_path() and os.path.getmtime(built_path()) >= os.path.getmtime(SRC):
        return built_path()
    os.makedirs(OUT, exist_ok=True)
    os.environ.setdefault("TORCH_CUDA_ARCH_LIST", "10.0a")
    from torch.utils.cpp_extension import load

    load(
        name=NAME,
        sources=[SRC],
        extra_cuda_cflags=["--use_fast_math", "-gencode", "arch=compute_100a,code=sm_100a"],
        build_directory=OUT,
        verbose=verbose,
        is_python_module=False,
    )
    return built_path()


def load_module():
    """Import the prebuilt reference extension (GPU box: only the .so exists)."""
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
