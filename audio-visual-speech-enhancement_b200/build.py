"""In-tree build of libavse_b200.so (hand-written CUDA for sm_100a + the C ABI of include/avse_b200.h).

nvcc cross-compiles without a GPU; the resulting .so is git-ignored but travels to the GPU box
with the repo snapshot.  No torch extension machinery is involved: the boundary is a plain C ABI.
"""
from __future__ import annotations

import os
import shutil
import subprocess

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG_DIR)
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.path.join(PKG_DIR, "libavse_b200.so")

SOURCES = ["avse_kernels.cu", "avse_inverse.cu", "avse_inverse_grad.cu", "avse_generic.cu", "avse_video.cu", "avse_tables.cpp", "avse_generic_tables.cpp"]
HEADERS = ["avse_common.h", "avse_dft.cuh", "avse_tables.h", "avse_ctx.h", "avse_fwd_stages.cuh", "avse_fwd4_stages.cuh", "avse_inv_stages.cuh", "avse_inv8_stages.cuh", "avse_inverse_grad_stages.cuh", "avse_generic.h",
           os.path.join(ROOT, "include", "avse_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared", "--expt-relaxed-constexpr",
]


def _nvcc():
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: libavse_b200.so cannot be built (there is no CPU fallback)")
    return nvcc


def _stale():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + [h if os.path.isabs(h) else os.path.join(CSRC, h) for h in HEADERS]
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in deps)


def build_library(force=False, verbose=False):
    """Compile the CUDA library if it is missing or older than its sources. Returns its path."""
    if not force and not _stale():
        return LIB_PATH
    cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB_PATH] + [os.path.join(CSRC, s) for s in SOURCES]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return LIB_PATH


def build_variant(out_path, defines, verbose=False):
    """Tuning helper: compile the same sources with extra -D macros into another .so (see AVSE_B200_LIB)."""
    cmd = [_nvcc()] + NVCC_FLAGS + ["-D%s" % d for d in defines] + (["-Xptxas", "-v"] if verbose else []) + \
        ["-o", out_path] + [os.path.join(CSRC, s) for s in SOURCES]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    return res.stderr


if __name__ == "__main__":
    import sys
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
