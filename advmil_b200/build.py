"""Builds libadvmil_b200.so in-tree with nvcc for sm_100a (no torch, no pybind: the library is plain C ABI).

    python -m advmil_b200.build [--force] [--verbose]
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "csrc", "_obj")
LIB = os.path.join(HERE, "libadvmil_b200.so")
SOURCES = ["api.cu", "gemm_stages.cu", "gemm_tc.cu", "seg_kernels.cu", "tail_kernels.cu", "step.cu", "esat_kernels.cu", "esat.cu", "codec.cu", "rlip_chain.cu", "esat_attn_tc.cu", "esat_attn_bwd_tc.cu", "cluster_pool.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "--use_fast_math=false",
         "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "-Xcompiler", "-O2"]
# `extern "C"` entry points must stay visible
FLAGS = [f for f in FLAGS if f != "--use_fast_math=false"]


def _digest() -> str:
    hsh = hashlib.sha256()
    for root in (CSRC, os.path.join(os.path.dirname(HERE), "include")):
        for name in sorted(os.listdir(root)):
            path = os.path.join(root, name)
            if os.path.isfile(path) and name.endswith((".cu", ".cuh", ".h")):
                hsh.update(name.encode())
                hsh.update(open(path, "rb").read())
    hsh.update(" ".join(FLAGS).encode())
    return hsh.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    stamp = os.path.join(OBJ, "digest.txt")
    dig = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read() == dig:
        return LIB

    def compile_one(src):
        obj = os.path.join(OBJ, src.replace(".cu", ".o"))
        cmd = [NVCC, *FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(12, len(SOURCES))) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    cmd = [NVCC, "-shared", "-o", LIB, *objs, "-lcudart", "-lcuda"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    open(stamp, "w").write(dig)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
