"""oracle/build_ref.py -- TEST INFRASTRUCTURE.  Compiles the UNMODIFIED reference kernels
(/root/reference/raymarching/src/raymarching.cu + bindings.cpp) for sm_100a into oracle/_ref/ as the pybind module
`_raymarching_ref` (git-ignored; travels to the GPU box with gpurun).  Sources are compiled where they lie; nothing is
copied into the repo.  Differences from the reference's own recipe (raymarching/backend.py:6-12): -std=c++17 instead of
c++14 (torch >= 2.1 headers need it) and an explicit -gencode for sm_100a (the reference passes no arch at all).

Used by tests/golden/make_golden_ref_raymarching.py to record the real reference kernels' outputs, against which
tests/test_ref_parity_gpu.py and tests/test_backend_dropin_gpu.py pin the CPU oracle and the CUDA path.
"""
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = "/root/reference/raymarching/src"
OUT = os.path.join(HERE, "_ref")


def build(verbose=False):
    if not os.path.isdir(SRC):
        return None
    os.makedirs(OUT, exist_ok=True)
    so = os.path.join(OUT, "_raymarching_ref.so")
    if os.path.exists(so):
        return so
    from torch.utils.cpp_extension import load
    os.environ.setdefault("TORCH_CUDA_ARCH_LIST", "10.0a")
    load(name="_raymarching_ref",
         sources=[os.path.join(SRC, "raymarching.cu"), os.path.join(SRC, "bindings.cpp")],
         extra_cflags=["-O3", "-std=c++17"],
         extra_cuda_cflags=["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a",
                            "-U__CUDA_NO_HALF_OPERATORS__", "-U__CUDA_NO_HALF_CONVERSIONS__", "-U__CUDA_NO_HALF2_OPERATORS__"],
         build_directory=OUT, verbose=verbose, is_python_module=False)
    return so if os.path.exists(so) else None


def load_ref():
    """Import the compiled reference module (GPU box: only the prebuilt .so is used)."""
    so = os.path.join(OUT, "_raymarching_ref.so")
    if not os.path.exists(so):
        return None
    import importlib.util
    import torch  # noqa: F401  (the module links against libtorch)
    spec = importlib.util.spec_from_file_location("_raymarching_ref", so)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


if __name__ == "__main__":
    print(build(verbose="-v" in sys.argv))
