"""Builds ``bevformer_b200/lib/libbevformer_b200.so`` with plain nvcc for sm_100a (no torch headers).

The shared library is the product's only native artefact; it is built IN-TREE so that it travels to
the GPU box with the repo snapshot (it is git-ignored through ``*.so``).
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libbevformer_b200.so")
STAMP = os.path.join(LIB_DIR, "build.stamp")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "--use_fast_math", "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
    "-shared", "-Xptxas", "-v",
]
# --use_fast_math only changes division/transcendental lowering and ftz; the sampler uses neither
# division nor transcendentals on its value path, LayerNorm/softmax use explicit intrinsics.


def sources():
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cu"))


def _digest() -> str:
    """Hash of the sources and flags.  Paths enter relative to the repository, so a built tree that is
    moved or copied elsewhere is still current and is not rebuilt (possibly read-only) where it lands."""
    root = os.path.dirname(HERE)
    h = hashlib.sha256()
    files = sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC))
    files.append(os.path.join(root, "include", "bevformer_b200.h"))
    for f in files:
        with open(f, "rb") as fh:
            h.update(os.path.relpath(f, root).encode() + b"\0" + fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def nvcc_path() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; the bevformer_b200 CUDA library cannot be built")


def build(force: bool = False, verbose: bool = False) -> str:
    digest = _digest()
    if not force and os.path.exists(LIB_PATH) and os.path.exists(STAMP):
        with open(STAMP) as f:
            if f.read().strip() == digest:
                return LIB_PATH
    os.makedirs(LIB_DIR, exist_ok=True)
    cmd = [nvcc_path(), *NVCC_FLAGS, "-o", LIB_PATH, *sources()]
    res = subprocess.run(cmd, capture_output=True, text=True)
    log = res.stdout + res.stderr
    with open(os.path.join(LIB_DIR, "build.log"), "w") as f:
        f.write(" ".join(cmd) + "\n" + log)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + log[-4000:])
    if verbose:
        print(log)
    with open(STAMP, "w") as f:
        f.write(digest)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
