"""Build libqsae_b200.so (hand-written sm_100a CUDA behind the C ABI of include/qsae_b200.h).

    python -m quantizedsae_b200.build [--force] [--verbose]

nvcc cross-compiles without a GPU. The library is built in-tree (git-ignored, but it travels to
the GPU box with the repo snapshot). No fast-math: the packing kernels must evaluate the same
fp32 logistic as the reference.
"""
from __future__ import annotations

import argparse
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
BUILD = PKG / "_build"
LIB = PKG / "libqsae_b200.so"
SOURCES = ["qsae_api.cu", "encode_topk_sm100.cu", "select_topk.cu", "pack.cu", "decode.cu", "encode_dense.cu", "rescue.cu", "matryoshka.cu",
           "dense_decode_sm100.cu", "analysis.cu", "peer.cu", "train.cu", "wgrad_sm100.cu"]
# every header a source can include: an edit to any of them rebuilds every object
HEADERS = [*sorted(CSRC.glob("*.h")), *sorted(CSRC.glob("*.cuh")), PKG.parent / "include" / "qsae_b200.h"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr",
]


def nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not Path(exe).exists():
        raise RuntimeError("nvcc not found; cannot build libqsae_b200.so")
    return exe


def _stale(target: Path, deps) -> bool:
    if not target.exists():
        return True
    t = target.stat().st_mtime
    return any(Path(d).stat().st_mtime > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> Path:
    BUILD.mkdir(exist_ok=True)
    cc = nvcc()
    jobs = []
    for src in SOURCES:
        obj = BUILD / (src.replace(".cu", ".o"))
        if force or _stale(obj, [CSRC / src, *HEADERS, Path(__file__)]):
            cmd = [cc, *NVCC_FLAGS, "-c", str(CSRC / src), "-o", str(obj)]
            if verbose:
                cmd.insert(1, "-Xptxas")
                cmd.insert(2, "-v")
            jobs.append(cmd)

    def run(cmd):
        r = subprocess.run(cmd, capture_output=True, text=True)
        return cmd, r

    with ThreadPoolExecutor(max_workers=min(8, max(1, len(jobs)))) as ex:
        for cmd, r in ex.map(run, jobs):
            if verbose or r.returncode != 0:
                sys.stderr.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
            if r.returncode != 0:
                raise RuntimeError(f"nvcc failed for {cmd[-3]}")
    objs = [str(BUILD / s.replace(".cu", ".o")) for s in SOURCES]
    if force or jobs or _stale(LIB, objs):
        cmd = [cc, "-shared", "-o", str(LIB), *objs, "-gencode", "arch=compute_100a,code=sm_100a",
               "-Xcompiler", "-fPIC", "-cudart", "static"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("link failed")
    return LIB


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--force", action="store_true")
    ap.add_argument("--verbose", action="store_true")
    a = ap.parse_args()
    print(build(a.force, a.verbose))
