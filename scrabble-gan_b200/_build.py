"""Builds libsgan.so (all CUDA kernels + the C ABI) in-tree for sm_100a with nvcc.

The shared object is git-ignored but travels to the GPU box with the gpurun snapshot.  There is no JIT and no
torch extension involved: the library is a plain C-ABI .so bound with ctypes (see _abi.py)."""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
BUILD = os.path.join(HERE, "csrc", "build")
LIB = os.path.join(HERE, "libsgan.so")
SOURCES = ["ctx.cu", "ew.cu", "bn.cu", "gemm.cu", "filterbank.cu", "attention.cu", "attention_tc.cu", "nonlocal.cu", "ctc.cu", "augment.cu", "loss.cu", "optim.cu", "peer.cu",
           "conv_simt.cu", "conv_tc.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def _digest() -> str:
    h = hashlib.sha256()
    for name in sorted(os.listdir(CSRC)):
        if name.endswith((".cu", ".cuh")):
            with open(os.path.join(CSRC, name), "rb") as f:
                h.update(name.encode())
                h.update(f.read())
    with open(os.path.join(os.path.dirname(HERE), "include", "sgan.h"), "rb") as f:
        h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every .cu for sm_100a and link libsgan.so.  Returns the library path."""
    os.makedirs(BUILD, exist_ok=True)
    stamp = os.path.join(BUILD, "stamp.txt")
    digest = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read().strip() == digest:
        return LIB
    nvcc = _nvcc()

    def compile_one(src: str) -> str:
        obj = os.path.join(BUILD, src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + ["-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for {}:\n{}\n{}".format(src, r.stdout, r.stderr))
        if verbose and r.stderr.strip():
            print(r.stderr, file=sys.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n{}\n{}".format(r.stdout, r.stderr))
    with open(stamp, "w") as f:
        f.write(digest)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
