"""In-tree build of the C-ABI CUDA library (``libtmc_b200.so``) for sm_100a.

nvcc cross-compiles without a GPU; the built ``.so`` is git-ignored but travels to the GPU box.
"""

from __future__ import annotations

import glob
import hashlib
import os
import subprocess

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.path.join(PKG_DIR, "libtmc_b200.so")
STAMP = LIB_PATH + ".stamp"

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
    "-DTMC_B200=1",
    "-shared",
]


def _sources():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")))


def _fingerprint() -> str:
    h = hashlib.sha256()
    for path in _sources() + sorted(glob.glob(os.path.join(CSRC, "*.cuh"))):
        h.update(path.encode())
        with open(path, "rb") as f:
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def is_current() -> bool:
    if not (os.path.exists(LIB_PATH) and os.path.exists(STAMP)):
        return False
    with open(STAMP) as f:
        return f.read().strip() == _fingerprint()


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every ``csrc/*.cu`` into ``libtmc_b200.so`` (no-op when up to date)."""
    if not force and is_current():
        return LIB_PATH
    nvcc = os.environ.get("NVCC", "nvcc")
    objs = []
    build_dir = os.path.join(PKG_DIR, "build")
    os.makedirs(build_dir, exist_ok=True)
    procs = []
    for src in _sources():
        obj = os.path.join(build_dir, os.path.basename(src)[:-3] + ".o")
        objs.append(obj)
        cmd = [nvcc, *[f for f in NVCC_FLAGS if f != "-shared"], "-c", src, "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for src, p in procs:
        out, _ = p.communicate()
        if verbose and out:
            print(out)
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{out}")
    cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB_PATH, *objs]
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if res.returncode != 0:
        raise RuntimeError(f"nvcc link failed:\n{res.stdout}")
    with open(STAMP, "w") as f:
        f.write(_fingerprint())
    return LIB_PATH


if __name__ == "__main__":
    import sys

    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
