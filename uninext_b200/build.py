"""In-tree build of libmsda_b200.so (the C-ABI CUDA library) with nvcc for sm_100a.

    python -m uninext_b200.build [--force] [--verbose]

The library is a plain shared object (no torch / pybind dependency): nvcc cross-compiles it in seconds without a GPU,
and it travels to the GPU box inside the repo snapshot (``uninext_b200/lib/`` is git-ignored, not gpurun-ignored).
"""
from __future__ import annotations

import argparse
import os
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_DIR = os.path.join(PKG_DIR, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libmsda_b200.so")
INCLUDE = os.path.join(os.path.dirname(PKG_DIR), "include")

SOURCES = ["msda_cabi.cu", "msda_gemm_sm100.cu"]
HEADERS = ["msda_common.cuh", "msda_tiled.cuh", "msda_slab.cuh", "msda_tmem.cuh", "msda_generic.cuh", "msda_det.cuh", "msda_module.cuh", "msda_condinst.cuh"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "--shared", "-Xcompiler", "-fPIC",
    "-Xptxas", "-v",
    "--expt-relaxed-constexpr",
]


def nvcc_path() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: cannot build libmsda_b200.so")


def is_stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    built = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.join(INCLUDE, "msda_b200.h"), __file__]
    return any(os.path.exists(d) and os.path.getmtime(d) > built for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile if sources are newer than the library. Returns the library path."""
    if not force and not is_stale():
        return LIB_PATH
    os.makedirs(LIB_DIR, exist_ok=True)
    tmp = f"{LIB_PATH}.tmp.{os.getpid()}"          # link under a private name, then rename: readers never see a partial file
    cmd = [nvcc_path()] + NVCC_FLAGS + ["-I", INCLUDE, "-o", tmp] + [os.path.join(CSRC, s) for s in SOURCES]
    proc = subprocess.run(cmd, capture_output=True, text=True)
    log = proc.stdout + proc.stderr
    with open(os.path.join(LIB_DIR, "build.log"), "w") as fh:
        fh.write(" ".join(cmd) + "\n" + log)
    if proc.returncode != 0:
        sys.stderr.write(log)
        if os.path.exists(tmp):
            os.remove(tmp)
        raise RuntimeError("nvcc failed building libmsda_b200.so (see output above)")
    os.replace(tmp, LIB_PATH)
    if verbose:
        print(log)
    return LIB_PATH


def wait_until_built(timeout_s: float = 600.0) -> str:
    """For ranks that do not build: block until another process has produced an up-to-date library."""
    import time
    t0 = time.time()
    while is_stale():
        if time.time() - t0 > timeout_s:
            raise RuntimeError(f"{LIB_PATH} was not built within {timeout_s:.0f} s")
        time.sleep(0.5)
    return LIB_PATH


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--force", action="store_true")
    ap.add_argument("--verbose", action="store_true")
    a = ap.parse_args()
    print(build(force=a.force, verbose=a.verbose))
