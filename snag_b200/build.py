"""Build recipe for libsnag_b200.so (hand-written sm_100a CUDA behind a C ABI).

nvcc cross-compiles without a GPU. The library is built IN-TREE (snag_b200/libsnag_b200.so) so that it
travels with the repo snapshot to the GPU box; it is git-ignored.

    python -m snag_b200.build [--force] [--verbose]
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
CSRC = PKG_DIR / "csrc"
BUILD_DIR = PKG_DIR / "_build"
LIB_PATH = PKG_DIR / "libsnag_b200.so"
SOURCES = ["abi.cu", "bw_kernels.cu", "sim_kernels.cu", "icl_fused.cu", "icl_fwd_sym.cu", "l1_sweep.cu"]
HEADERS = ["common.cuh", "simgemm.cuh", "snag_internal.h", "../../include/snag_b200.h"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC",
    "--expt-relaxed-constexpr",
]


def _nvcc() -> str:
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found; libsnag_b200.so cannot be built")
    return nvcc


def _source_digest() -> str:
    h = hashlib.sha256()
    for name in SOURCES + HEADERS:
        h.update(name.encode())
        h.update((CSRC / name).read_bytes())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def needs_build() -> bool:
    stamp = BUILD_DIR / "digest"
    return not (LIB_PATH.exists() and stamp.exists() and stamp.read_text() == _source_digest())


def build(force: bool = False, verbose: bool = False) -> Path:
    """Compile every CUDA source for sm_100a and link libsnag_b200.so. Returns the library path."""
    if not force and not needs_build():
        return LIB_PATH
    nvcc = _nvcc()
    BUILD_DIR.mkdir(exist_ok=True)
    objs = []
    procs = []
    for src in SOURCES:
        obj = BUILD_DIR / (Path(src).stem + ".o")
        cmd = [nvcc, *NVCC_FLAGS, "-c", str(CSRC / src), "-o", str(obj)]
        if verbose:
            cmd[1:1] = ["-Xptxas", "-v"]
            print(" ".join(cmd), flush=True)
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(str(obj))
    for src, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            print(out, flush=True)
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{out}")
    tmp = LIB_PATH.with_suffix(".so.tmp")
    cmd = [nvcc, "-shared", "-o", str(tmp), *objs, "-gencode", "arch=compute_100a,code=sm_100a"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}")
    os.replace(tmp, LIB_PATH)
    (BUILD_DIR / "digest").write_text(_source_digest())
    return LIB_PATH


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(path)
