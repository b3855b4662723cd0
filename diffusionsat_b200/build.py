"""Compile libdsat.so (sm_100a) in-tree with nvcc.  `python -m diffusionsat_b200.build`."""

from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_PATH = os.path.join(CSRC, "libdsat.so")
SOURCES = ["dsat_api.cu"]


def _headers():
    found = [f for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    return found + [os.path.join("..", "..", "include", h) for h in ("dsat.h", "dsat_debug.h")]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    built = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, s) for s in SOURCES + _headers()]
    return any(os.path.exists(d) and os.path.getmtime(d) > built for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB_PATH
    # -compress-all: the fatbin's cubin is compressed whatever its size (by default nvcc left the 8.9 MB cubin of
    # sm_100a SASS uncompressed, a 10.4 MB library instead of 3.8 MB).  No -lcuda: cuTensorMapEncodeTiled is resolved at
    # run time (cudaGetDriverEntryPoint), so the library still loads on a machine without a driver (CPU test tier)
    cmd = [_nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
           "-Xcompiler", "-fPIC", "-shared", "-Xfatbin", "-compress-all"]
    if verbose:
        cmd += ["-Xptxas", "-v"]
    cmd += os.environ.get("DSAT_NVCC_FLAGS", "").split()      # e.g. -DDSAT_ASSERT for the debug build
    cmd += ["-o", LIB_PATH] + [os.path.join(CSRC, s) for s in SOURCES]
    proc = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if verbose or proc.returncode != 0:
        sys.stderr.write(proc.stdout)
    if proc.returncode != 0:
        raise RuntimeError("nvcc failed building libdsat.so")
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
