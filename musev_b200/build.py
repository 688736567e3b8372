"""Builds the in-tree CUDA library (sm_100a only) with a plain nvcc command line.

The .so is written next to the package (musev_b200/_lib/libmusevb200.so) so that it travels with the
repo snapshot to the GPU box; it is git-ignored.
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
LIB_DIR = os.path.join(PKG_DIR, "_lib")
LIB_PATH = os.path.join(LIB_DIR, "libmusevb200.so")
INCLUDE = os.path.join(os.path.dirname(PKG_DIR), "include")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC",
    "--expt-relaxed-constexpr",
    "-I", INCLUDE,
]


def _nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found; musev_b200 needs the CUDA toolkit to build its kernels")
    return exe


def _sources() -> list[str]:
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cu"))


def _digest() -> str:
    # names relative to the repository (not absolute paths), so that a checkout moved or copied elsewhere with its
    # built library is not rebuilt
    h = hashlib.sha256()
    repo = os.path.dirname(PKG_DIR)
    files = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC))] + [os.path.join(INCLUDE, f) for f in sorted(os.listdir(INCLUDE))]
    for p in files:
        if os.path.isfile(p):
            h.update(os.path.relpath(p, repo).encode())
            with open(p, "rb") as fh:
                h.update(fh.read())
    h.update(" ".join(f for f in NVCC_FLAGS if f != INCLUDE).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every .cu under csrc/ to one shared library. Returns its path."""
    os.makedirs(LIB_DIR, exist_ok=True)
    stamp = os.path.join(LIB_DIR, "build.stamp")
    digest = _digest()
    if not force and os.path.exists(LIB_PATH) and os.path.exists(stamp):
        with open(stamp) as fh:
            if fh.read().strip() == digest:
                return LIB_PATH
    nvcc = _nvcc()
    obj_dir = os.path.join(LIB_DIR, "obj")
    os.makedirs(obj_dir, exist_ok=True)

    def compile_one(src: str) -> str:
        obj = os.path.join(obj_dir, os.path.basename(src)[:-3] + ".o")
        cmd = [nvcc, *NVCC_FLAGS, "-c", src, "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        objs = list(ex.map(compile_one, _sources()))
    cmd = [nvcc, "-shared", "-o", LIB_PATH, *objs, "-ldl", "-lpthread"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    with open(stamp, "w") as fh:
        fh.write(digest)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
