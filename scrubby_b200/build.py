"""Builds libscrubby_gpu.so (hand-written sm_100a CUDA + the C ABI) in-tree with nvcc.

    python -m scrubby_b200.build [--force]

The .so lands in scrubby_b200/lib/ (git-ignored, shipped to the GPU box by gpurun).
"""
from __future__ import annotations

import os
import shlex
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
# tuning / diagnostic builds: SGPU_VARIANT=name selects libscrubby_gpu_name.so, built with the extra nvcc
# flags in SGPU_NVCC_FLAGS (e.g. "-DSGPU_FUSED_TIMING"); the default build has no variant
VARIANT = os.environ.get("SGPU_VARIANT", "")
_SUFFIX = f"_{VARIANT}" if VARIANT else ""
OBJDIR = os.path.join(HERE, "lib", "obj" + _SUFFIX)
SO = os.path.join(LIBDIR, f"libscrubby_gpu{_SUFFIX}.so")
SOURCES = ["scan.cu", "idset.cu", "idset_build.cu", "evidence.cu", "fastq_general.cu", "fasta_general.cu", "fastq_fused.cu", "idset_route.cu", "capi.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC,-O3,-Wall", "--expt-relaxed-constexpr",
]


def _deps_mtime() -> float:
    paths = [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    paths.append(os.path.join(os.path.dirname(HERE), "include", "scrubby_gpu.h"))
    return max(os.path.getmtime(p) for p in paths)


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJDIR, exist_ok=True)
    if not force and os.path.exists(SO) and os.path.getmtime(SO) >= _deps_mtime():
        return SO
    if not os.path.exists(NVCC):
        raise RuntimeError(f"nvcc not found at {NVCC}; cannot build libscrubby_gpu.so")

    def compile_one(src: str) -> str:
        obj = os.path.join(OBJDIR, src.replace(".cu", ".o"))
        cmd = [NVCC, *FLAGS, *shlex.split(os.environ.get("SGPU_NVCC_FLAGS", "") if VARIANT else ""), "-c",
               os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    cmd = [NVCC, "-shared", "-o", SO, *objs, "-gencode", "arch=compute_100a,code=sm_100a"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return SO


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
