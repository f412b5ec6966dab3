"""Build the sm_100a shared library (libffb.so) in-tree with nvcc.

    python -m funscript_flow_b200.build            # build if sources are newer than the .so
    python -m funscript_flow_b200.build --force

nvcc cross-compiles for sm_100a without a GPU; the resulting .so travels to the GPU box with the
repo snapshot (it is git-ignored, not gpurun-ignored).
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libffb.so")
SOURCES = [os.path.join(CSRC, "ffb_api.cu")]
DEPS = SOURCES + [os.path.join(CSRC, "ffb_kernels.cuh"), os.path.join(CSRC, "ffb_common.h"),
                  os.path.join(ROOT, "include", "ffb.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC,-O3,-Wall,-Wno-unused-function,-pthread",
    "--expt-relaxed-constexpr",
    "-shared", "-cudart", "shared",
]


def find_nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False, extra=(), lib: str = LIB) -> str:
    """Compile the library to `lib` (default: in-tree) unless it is newer than its sources; returns its path."""
    if not force and not needs_build(lib, DEPS):
        return lib
    cmd = [find_nvcc(), *NVCC_FLAGS, *extra, "-I", os.path.join(ROOT, "include"), "-I", CSRC, "-o", lib, *SOURCES]
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
        print(" ".join(cmd))
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stdout + res.stderr)
    return lib


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
