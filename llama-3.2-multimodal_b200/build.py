"""Build the C-ABI shared library `libl32ffn.so` (pure CUDA, no torch headers) for sm_100a, in-tree.

The library is the only compiled artefact of the product path; the Python modules `rmsnorm` and
`swiglu_fused` (reference setup.py:11-41 names) bind it through ctypes.  Compiles in a few seconds
because no translation unit includes torch/extension.h.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
BUILD = os.path.join(HERE, "_build")
LIB = os.path.join(HERE, "libl32ffn.so")
SOURCES = ["rmsnorm.cu", "gemm_sm100.cu", "ffn_decode.cu", "elementwise.cu", "tp.cu", "lmhead.cu", "attention.cu", "attention_bwd.cu", "sampling.cu", "speculative.cu", "api.cu"]
HEADERS = ["l32_internal.cuh", "ptx_sm100.cuh", os.path.join("..", "..", "include", "l32_ffn.h")]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "--expt-relaxed-constexpr",
]


def _nvcc() -> str:
    cand = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(cand):
        raise RuntimeError("nvcc not found; the C-ABI library cannot be built")
    return cand


def _digest() -> str:
    h = hashlib.sha256()
    for name in SOURCES + HEADERS:
        with open(os.path.join(CSRC, name), "rb") as f:
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile (if sources changed) and return the path of libl32ffn.so."""
    os.makedirs(BUILD, exist_ok=True)
    stamp = os.path.join(BUILD, "digest.txt")
    digest = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read().strip() == digest:
        return LIB
    nvcc = _nvcc()
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(BUILD, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for src, p in procs:
        out, _ = p.communicate()
        if verbose and out:
            print(out)
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{out}")
    link = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC", *objs, "-o", LIB,
            "-cudart", "shared"]   # torch has already mapped libcudart.so.12; a static cudart would embed its whole symbol table
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}")
    with open(stamp, "w") as f:
        f.write(digest)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
