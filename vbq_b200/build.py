"""In-tree build of libvbq_b200.so (sm_100a only; nvcc cross-compiles without a GPU)."""
from __future__ import annotations

import os
import shutil
import subprocess

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
REPO_DIR = os.path.dirname(PKG_DIR)
SOURCES = [os.path.join(PKG_DIR, "csrc", f) for f in ("api.cu", "priors.cu", "quantize.cu", "quantize_strict.cu", "quantize_reference.cu", "quantize_fast.cu", "quantize_bisect.cu", "quantize_tma.cu", "quantize_tma_both.cu", "sweep_bisect.cu", "sweep_both.cu",
            "sweep.cu", "host_pipeline.cu", "operators.cu", "embeddings.cu", "serialize.cu", "rans.cu", "ranks.cu", "image_metrics.cu", "peer.cu")]
HEADERS = [os.path.join(REPO_DIR, "include", "vbq_b200.h"), os.path.join(PKG_DIR, "csrc", "common.h"),
           os.path.join(PKG_DIR, "csrc", "tree.cuh"),
           os.path.join(PKG_DIR, "csrc", "quantize_kernel.cuh"), os.path.join(PKG_DIR, "csrc", "bisect.cuh"), os.path.join(PKG_DIR, "csrc", "tma.cuh"), os.path.join(PKG_DIR, "csrc", "quantize_tma.cuh")]
LIB_PATH = os.path.join(PKG_DIR, "libvbq_b200.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17", "--threads", "0",
    "-Xcompiler", "-fPIC", "-shared",
]


def _nvcc():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found; vbq_b200 needs the CUDA toolkit to build libvbq_b200.so")
    return exe


def is_stale():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(p) > t for p in SOURCES + HEADERS)


def build_library(force=False, verbose=False):
    """Compile csrc/*.cu into vbq_b200/libvbq_b200.so.  Returns the library path."""
    if not force and not is_stale():
        return LIB_PATH
    cmd = [_nvcc()] + NVCC_FLAGS + ["-I", os.path.join(REPO_DIR, "include")]
    if verbose:
        cmd += ["-Xptxas", "-v"]
    if os.environ.get("VBQ_BUILD_DEFINES"):   # development switches, e.g. VBQ_BUILD_DEFINES="-DVBQ_DEV_VARIANTS"
        cmd += os.environ["VBQ_BUILD_DEFINES"].split()
    cmd += SOURCES + ["-o", LIB_PATH]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return LIB_PATH


if __name__ == "__main__":
    print(build_library(force=True, verbose=True))
