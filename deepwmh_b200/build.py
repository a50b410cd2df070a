"""Build libdeepwmh_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libdeepwmh_b200.so")
STAMP = os.path.join(LIB_DIR, "libdeepwmh_b200.stamp")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared", "--expt-relaxed-constexpr",
    "-Xptxas", "-v",
]


def _sources():
    srcs = [os.path.join(CSRC, "api.cu"), os.path.join(CSRC, "stage1.cu"), os.path.join(CSRC, "resample.cu"),
            os.path.join(CSRC, "n4.cu")]
    deps = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC))] + [os.path.join(ROOT, "include", "deepwmh_b200.h")]
    return srcs, deps


def _digest(deps) -> str:
    h = hashlib.sha256()
    for d in deps:
        with open(d, "rb") as f:
            h.update(d.encode() + b"\0" + f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile the CUDA sources into deepwmh_b200/lib/libdeepwmh_b200.so; returns its path.
    Skips the compile when sources and flags are unchanged since the last build."""
    srcs, deps = _sources()
    dig = _digest(deps)
    if not force and os.path.exists(LIB_PATH) and os.path.exists(STAMP) and open(STAMP).read().strip() == dig:
        return LIB_PATH
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found; cannot build libdeepwmh_b200.so")
    os.makedirs(LIB_DIR, exist_ok=True)
    cmd = [nvcc] + NVCC_FLAGS + ["-I", os.path.join(ROOT, "include"), "-o", LIB_PATH] + srcs
    res = subprocess.run(cmd, capture_output=True, text=True)
    log = res.stdout + res.stderr
    with open(os.path.join(LIB_DIR, "build.log"), "w") as f:
        f.write(" ".join(cmd) + "\n" + log)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + log[-8000:])
    if verbose:
        print(log)
    with open(STAMP, "w") as f:
        f.write(dig)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
