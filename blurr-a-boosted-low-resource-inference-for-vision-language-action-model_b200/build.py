"""Build the C-ABI CUDA library (`lib/libblurr_pi0.so`) in-tree with nvcc for sm_100a.

nvcc cross-compiles without a GPU, so this runs in the build container; the built `.so` is
git-ignored but travels to the GPU box with the repo snapshot.
"""

from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_DIR = os.path.join(PKG_DIR, "lib")
BUILD_DIR = os.path.join(PKG_DIR, "build")
LIB_PATH = os.path.join(LIB_DIR, "libblurr_pi0.so")
INCLUDE_DIR = os.path.join(os.path.dirname(PKG_DIR), "include")

SOURCES = ["gemm_tc.cu", "norm_consumers.cu", "attention.cu", "attention_tc.cu", "misc_kernels.cu", "engine.cu",
           "preprocess.cu", "llm_kernels.cu", "llm_engine.cu", "vit_engine.cu", "act_head.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC",
]


def _nvcc() -> str:
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: cannot build libblurr_pi0.so")
    return nvcc


def _source_digest() -> str:
    hsh = hashlib.sha256()
    names = sorted(os.listdir(CSRC)) + ["../../include/blurr_pi0.h"]
    for name in names:
        path = os.path.join(CSRC, name)
        if os.path.isfile(path):
            with open(path, "rb") as f:
                hsh.update(name.encode())
                hsh.update(f.read())
    hsh.update(" ".join(NVCC_FLAGS).encode())
    return hsh.hexdigest()


def needs_build() -> bool:
    stamp = os.path.join(LIB_DIR, "source.sha256")
    if not (os.path.isfile(LIB_PATH) and os.path.isfile(stamp)):
        return True
    with open(stamp, "r", encoding="utf-8") as f:
        return f.read().strip() != _source_digest()


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every kernel file for sm_100a and link `libblurr_pi0.so`. Returns its path."""
    if not force and not needs_build():
        return LIB_PATH
    nvcc = _nvcc()
    os.makedirs(LIB_DIR, exist_ok=True)
    os.makedirs(BUILD_DIR, exist_ok=True)

    def compile_one(src: str) -> str:
        obj = os.path.join(BUILD_DIR, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, "-I", INCLUDE_DIR, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{res.stdout}\n{res.stderr}")
        if verbose:
            sys.stderr.write(res.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as pool:
        objs = list(pool.map(compile_one, SOURCES))
    link = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB_PATH, *objs]
    res = subprocess.run(link, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError(f"link failed:\n{res.stdout}\n{res.stderr}")
    with open(os.path.join(LIB_DIR, "source.sha256"), "w", encoding="utf-8") as f:
        f.write(_source_digest())
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
