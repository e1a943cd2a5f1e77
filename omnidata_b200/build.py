"""Builds the C-ABI shared library (in-tree, sm_100a only).

`python -m omnidata_b200.build` or `__graft_entry__.build()`.  nvcc cross-compiles without a GPU.
The .so is git-ignored but travels to the GPU box with the gpurun snapshot.
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
LIB_DIR = PKG / "lib"
LIB_PATH = LIB_DIR / "libomnidata_b200.so"
SOURCES = ["api.cu", "conv_gemm.cu", "ops.cu", "attention_tc.cu", "attention_stream.cu", "fp32_path.cu", "bwd_ops.cu",
           "bgemm.cu", "bgemm_tc.cu", "loss.cu", "imageproc.cu", "optim.cu", "refocus.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC",
]
# fast-math (approximate division / sqrt / exp, denormals flushed) only where the arithmetic is bf16-bound anyway:
# the tensor-core GEMM / attention epilogues and the bf16 elementwise kernels.  The fp32 losses, the optimizer, the
# fp32 correctness mode, image resampling and the refocus blur promise reference fp32 arithmetic and are built without.
FAST_MATH_SOURCES = {"conv_gemm.cu", "ops.cu", "attention_tc.cu", "attention_stream.cu", "bgemm_tc.cu"}


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _stamp() -> str:
    h = hashlib.sha256()
    files = sorted(CSRC.glob("*")) + [PKG.parent / "include" / "omnidata_b200.h"]
    for f in files:
        if f.is_file():
            h.update(f.name.encode())
            h.update(f.read_bytes())
    h.update(" ".join(NVCC_FLAGS + sorted(FAST_MATH_SOURCES)).encode())
    return h.hexdigest()


def build_library(force: bool = False, verbose: bool = False) -> Path:
    LIB_DIR.mkdir(exist_ok=True)
    stamp_file = LIB_DIR / "build.stamp"
    stamp = _stamp()
    if not force and LIB_PATH.exists() and stamp_file.exists() and stamp_file.read_text() == stamp:
        return LIB_PATH
    objs = []
    procs = []
    obj_dir = LIB_DIR / "obj"
    obj_dir.mkdir(exist_ok=True)
    for src in SOURCES:
        if not (CSRC / src).exists():
            continue
        obj = obj_dir / (src + ".o")
        cmd = [_nvcc(), *NVCC_FLAGS, *(["--use_fast_math"] if src in FAST_MATH_SOURCES else []), "-c", str(CSRC / src),
               "-o", str(obj)]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(str(obj))
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{out}")
        if verbose and out:
            print(out)
    link = [_nvcc(), "-shared", "-o", str(LIB_PATH), *objs, "-gencode", "arch=compute_100a,code=sm_100a",
            "-Xcompiler", "-fPIC", "-lcudart"]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}")
    stamp_file.write_text(stamp)
    return LIB_PATH


if __name__ == "__main__":
    path = build_library(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(path)
