"""In-tree nvcc build of libcsvb200.so for sm_100a (no JIT cache: the .so travels with the repo)."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SO = os.path.join(HERE, "libcsvb200.so")
SOURCES = ["api.cu", "index_build.cu", "index_build_tma.cu", "lookup.cu", "tape.cu", "materialize.cu", "stream.cu", "validate.cu", "exchange.cu"]
HEADERS = ["internal.h", "ctx.h", "slice_pool.h", "record_split.h", "bitslice.cuh", "utf8slice.cuh", "index_common.cuh", os.path.join("..", "..", "include", "csvb200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC,-O3,-Wall,-Wno-unknown-pragmas",
    "-shared",
]


def nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: libcsvb200.so cannot be built (there is no CPU fallback)")
    return exe


def is_stale() -> bool:
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS]
    return any(os.path.getmtime(d) > t for d in deps)


HOST_SO = os.path.join(HERE, "libcsvsimd_host.so")
HOST_SOURCES = [os.path.join("host", "host_capi.cpp")]
HOST_HEADERS = [os.path.join("host", "csv_simd.hpp")]


def host_is_stale() -> bool:
    if not os.path.exists(HOST_SO):
        return True
    t = os.path.getmtime(HOST_SO)
    deps = [os.path.join(CSRC, s) for s in HOST_SOURCES + HOST_HEADERS] + [SO]
    return any(os.path.getmtime(d) > t for d in deps)


def build_host(force: bool = False) -> str:
    """The C++ host mirror of the crate's API (csrc/host/csv_simd.hpp) + its flat C shim, linked against
    libcsvb200.so (rpath $ORIGIN)."""
    build(force=False)
    if not force and not host_is_stale():
        return HOST_SO
    cxx = os.environ.get("CXX") or shutil.which("g++") or "g++"
    cmd = [cxx, "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-o", HOST_SO,
           *[os.path.join(CSRC, s) for s in HOST_SOURCES], "-L" + HERE, "-lcsvb200", "-Wl,-rpath,$ORIGIN"]
    subprocess.check_call(cmd)
    return HOST_SO


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not is_stale():
        return SO
    cmd = [nvcc(), *NVCC_FLAGS, "-o", SO, *[os.path.join(CSRC, s) for s in SOURCES]]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
        print(" ".join(cmd), file=sys.stderr)
    subprocess.check_call(cmd)
    return SO


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose=True)
    build_host(force="--force" in sys.argv)
    print(SO)
    print(HOST_SO)
