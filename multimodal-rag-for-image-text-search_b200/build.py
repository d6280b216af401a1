"""Build libmmr_b200.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with the repo)."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from typing import List

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libmmr_b200.so")
SOURCES = ["mmr_b200.cu", "mmr_encoder.cu"]
ARCH_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a"]


def _nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: the B200 scan library cannot be built (there is no CPU fallback)")
    return exe


def _deps() -> List[str]:
    out = [os.path.join(HERE, "..", "include", "mmr_b200.h")]
    for name in os.listdir(CSRC):
        if name.endswith((".cu", ".cuh", ".h")):
            out.append(os.path.join(CSRC, name))
    return out


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(p) > t for p in _deps() if os.path.exists(p))


def build(force: bool = False, verbose: bool = False, extra: List[str] | None = None) -> str:
    """Compile csrc/*.cu -> libmmr_b200.so (one nvcc per translation unit, in parallel, then one link).  Returns the
    library path."""
    from concurrent.futures import ThreadPoolExecutor

    if not force and not needs_build():
        return LIB
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    common = [_nvcc(), *ARCH_FLAGS, "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC", *(extra or [])]

    def compile_one(src: str) -> str:
        obj = os.path.join(objdir, os.path.splitext(src)[0] + ".o")
        cmd = [*common, "-c", "-o", obj, os.path.join(CSRC, src)]
        if verbose:
            print(" ".join(cmd), file=sys.stderr)
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n" + res.stdout + res.stderr)
        if verbose and (res.stdout or res.stderr):
            print(res.stdout + res.stderr, file=sys.stderr)
        return obj

    with ThreadPoolExecutor(len(SOURCES)) as pool:
        objs = list(pool.map(compile_one, SOURCES))
    link = [_nvcc(), *ARCH_FLAGS, "-shared", "-o", LIB, *objs]
    if verbose:
        print(" ".join(link), file=sys.stderr)
    res = subprocess.run(link, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("link failed:\n" + res.stdout + res.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
