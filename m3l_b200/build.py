"""Builds the in-tree native library `m3l_b200/lib/libm3l_b200.so` for sm_100a with nvcc.

The library is a plain C-ABI shared object (include/m3l_b200.h); Python binds it with ctypes
(m3l_b200/_lib.py).  nvcc cross-compiles without a GPU, so this runs in the CPU-only container
and the built .so travels to the GPU box with the repo snapshot.
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

ROOT = Path(__file__).resolve().parent
CSRC = ROOT / "csrc"
OBJ = ROOT / "build"
LIBDIR = ROOT / "lib"
LIB = LIBDIR / "libm3l_b200.so"

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ARCH_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a"]
NVCC_FLAGS = [
    "-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC",
    "-Xcompiler", "-Wall", "-Xcompiler", "-Wno-unused-function", "--expt-relaxed-constexpr",
    "-Xptxas", "-v",
]
# --use_fast_math only where the approximate exp2 / reciprocal are the point (softmax exponentials and the GELU
# epilogues of the tensor-core kernels).  LayerNorm statistics, the MSE loss, the gradient norm and AdamW
# (elementwise.cu, optim.cu) are compiled with IEEE division / sqrt and without flush-to-zero.
FAST_MATH_SOURCES = {"gemm.cu", "gemm_gelu.cu", "attention.cu", "attention_long.cu", "attention_dh.cu",
                     "attention_dropout.cu", "rowblock.cu"}


def flags_for(src: Path) -> list[str]:
    return NVCC_FLAGS + (["--use_fast_math"] if src.name in FAST_MATH_SOURCES else [])


def _sources() -> list[Path]:
    return sorted(CSRC.glob("*.cu"))


def _deps_hash(src: Path) -> str:
    h = hashlib.sha256()
    h.update(src.read_bytes())
    for hdr in sorted(list(CSRC.glob("*.cuh")) + list(CSRC.glob("*.h")) +
                      list((ROOT.parent / "include").glob("*.h"))):
        h.update(hdr.read_bytes())
    h.update(" ".join(flags_for(src) + ARCH_FLAGS).encode())
    return h.hexdigest()


def _compile(src: Path, verbose: bool) -> Path:
    obj = OBJ / (src.stem + ".o")
    stamp = OBJ / (src.stem + ".hash")
    digest = _deps_hash(src)
    if obj.exists() and stamp.exists() and stamp.read_text() == digest:
        return obj
    cmd = [NVCC, *ARCH_FLAGS, *flags_for(src), "-c", str(src), "-o", str(obj)]
    res = subprocess.run(cmd, capture_output=True, text=True)
    log = OBJ / (src.stem + ".ptxas.log")
    log.write_text(res.stderr)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError(f"nvcc failed for {src.name}")
    if verbose:
        sys.stderr.write(f"[m3l_b200.build] compiled {src.name}\n")
    stamp.write_text(digest)
    return obj


def build(verbose: bool = True, force: bool = False) -> Path:
    OBJ.mkdir(exist_ok=True)
    LIBDIR.mkdir(exist_ok=True)
    if force:
        for f in OBJ.glob("*.hash"):
            f.unlink()
    srcs = _sources()
    with ThreadPoolExecutor(max_workers=min(8, len(srcs))) as ex:
        objs = list(ex.map(lambda s: _compile(s, verbose), srcs))
    newest = max(o.stat().st_mtime for o in objs)
    if (not LIB.exists()) or LIB.stat().st_mtime < newest:
        cmd = [NVCC, *ARCH_FLAGS, "-shared", "-o", str(LIB), *map(str, objs), "-lcudart"]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            sys.stderr.write(res.stdout + res.stderr)
            raise RuntimeError("link failed")
        if verbose:
            sys.stderr.write(f"[m3l_b200.build] linked {LIB}\n")
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv)
