"""In-tree build of the two shared libraries (no JIT cache, nothing installed to site-packages).

  libddsp_b200.so        hand-written sm_100a CUDA kernels behind the C ABI (include/ddsp_b200.h);
                         nvcc only, no torch dependency -- this is what a non-Python host binds.
  libddsp_b200_torch.so  TORCH_LIBRARY shim (csrc/torch_ops.cpp) linked against the first.

    python -m ddsp_pytorch_b200.build [--force]

nvcc cross-compiles without a GPU, so this runs in the build container; the .so files travel to
the GPU box with the repo snapshot (they are git-ignored, not gpurun-ignored).
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
INCLUDE = os.path.join(ROOT, "include")
LIB_CORE = os.path.join(PKG, "libddsp_b200.so")
LIB_TORCH = os.path.join(PKG, "libddsp_b200_torch.so")

CU_SOURCES = ["controls.cu", "harmonic.cu", "noise.cu", "stft.cu", "mss_fused.cu", "fftconv.cu", "conv_stream.cu", "features.cu", "pitch.cu", "gru.cu", "gemm3x.cu", "layernorm.cu"]
CU_HEADERS = ["common.cuh", "fft.cuh", "regfft.cuh", "pfft.cuh"]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def _run(cmd):
    print("[ddsp_b200.build]", " ".join(cmd), flush=True)
    subprocess.run(cmd, check=True)


def build_core(force: bool = False) -> str:
    srcs = [os.path.join(CSRC, s) for s in CU_SOURCES]
    deps = srcs + [os.path.join(CSRC, h) for h in CU_HEADERS] + [os.path.join(INCLUDE, "ddsp_b200.h")]
    if force or _stale(LIB_CORE, deps):
        _run([_nvcc(), *ARCH, "-O3", "-lineinfo", "-std=c++17", "-shared", "-Xcompiler", "-fPIC",
              "-I", INCLUDE, "-I", CSRC, "-o", LIB_CORE, *srcs,
              "-cudart", "shared"])
    return LIB_CORE


def build_torch(force: bool = False) -> str:
    src = os.path.join(CSRC, "torch_ops.cpp")
    deps = [src, os.path.join(INCLUDE, "ddsp_b200.h"), LIB_CORE]
    if force or _stale(LIB_TORCH, deps):
        import torch
        from torch.utils import cpp_extension as ce
        try:
            paths = ce.include_paths("cuda")
        except TypeError:                      # older signature: include_paths(cuda=False)
            paths = ce.include_paths(cuda=True)
        inc = []
        for p in paths:
            inc += ["-isystem", p]
        tlib = os.path.join(os.path.dirname(torch.__file__), "lib")
        cuda_home = os.path.dirname(os.path.dirname(_nvcc()))
        abi = int(torch._C._GLIBCXX_USE_CXX11_ABI)
        _run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", f"-D_GLIBCXX_USE_CXX11_ABI={abi}",
              "-DTORCH_API_INCLUDE_EXTENSION_H", "-I", INCLUDE, *inc, "-isystem",
              os.path.join(cuda_home, "include"), src, "-o", LIB_TORCH,
              "-L", PKG, "-lddsp_b200", "-L", tlib, "-lc10", "-lc10_cuda", "-ltorch_cpu", "-ltorch_cuda",
              "-ltorch", "-L", os.path.join(cuda_home, "lib64"), "-lcudart",
              "-Wl,-rpath,$ORIGIN", f"-Wl,-rpath,{tlib}", "-Wl,--no-as-needed"])
    return LIB_TORCH


def build_all(force: bool = False):
    return build_core(force), build_torch(force)


if __name__ == "__main__":
    build_all("--force" in sys.argv)
