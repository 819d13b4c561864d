"""Builds libwdx_b200.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

    python -m warpdemux_b200.build [--force] [--verbose]

The .so lands in warpdemux_b200/lib/ (git-ignored, travels with gpurun).
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libwdx_b200.so")
SOURCES = ["wdx_b200.cu", "wdx_fp.cu", "wdx_cnn.cu", "wdx_validate.cu", "wdx_vbz.cu"]
HEADERS = ["wdx_types.cuh", "fused_kernels.cuh", "dtw_band.cuh", "dtw_band_x2.cuh", "dtw_wavefront.cuh", "fingerprint_kernel.cuh", "wdx_internal.cuh", "cnn_kernels.cuh", "block_select.cuh", "cnn_tc_kernel.cuh", "validate_kernel.cuh", "llr_kernel.cuh", "vbz_kernel.cuh",
           os.path.join("..", "..", "include", "wdx_b200.h")]

NVCC_FLAGS = [
    "-O3", "-std=c++17",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo",
    "-fmad=false",          # no implicit FMA contraction: FP64 paths must round like the x86-64 CPU build;
                            # the FP32 fast path asks for FMA explicitly (__fmaf_rn)
    "-Xcompiler", "-fPIC",
    "-Xptxas", "-v",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


STAMP = os.path.join(LIBDIR, "sources.sha256")


def _source_digest() -> str:
    """Content hash of everything the library is built from (mtimes do not survive copying the tree to another box)."""
    import hashlib

    h = hashlib.sha256(" ".join(NVCC_FLAGS + [os.environ.get("WDX_NVCC_EXTRA", "")]).encode())
    for rel in SOURCES + HEADERS:
        with open(os.path.join(CSRC, rel), "rb") as fh:
            h.update(rel.encode() + b"\0" + fh.read())
    return h.hexdigest()


def needs_build() -> bool:
    if not os.path.exists(LIB) or not os.path.exists(STAMP):
        return True
    with open(STAMP) as fh:
        return fh.read().strip() != _source_digest()


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    os.makedirs(LIBDIR, exist_ok=True)
    nvcc = _nvcc()
    ccbin = ["-ccbin", "/usr/bin/g++"] if os.path.exists("/usr/bin/g++") else []  # the image's default CC may be a wrapper
    objdir = os.path.join(LIBDIR, "obj")
    os.makedirs(objdir, exist_ok=True)
    # one translation unit per process, in parallel; then one link step
    procs, objs, log = [], [], ""
    for src in SOURCES:
        obj = os.path.join(objdir, os.path.splitext(src)[0] + ".o")
        objs.append(obj)
        cmd = [nvcc] + NVCC_FLAGS + os.environ.get("WDX_NVCC_EXTRA", "").split() + ccbin + ["-c", "-o", obj, os.path.join(CSRC, src)]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    ok = True
    for cmd, pr in procs:
        out, _ = pr.communicate()
        log += " ".join(cmd) + "\n" + out
        ok = ok and pr.returncode == 0
    if ok:
        cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a"] + ccbin + ["-o", LIB] + objs
        res = subprocess.run(cmd, capture_output=True, text=True)
        log += " ".join(cmd) + "\n" + res.stdout + res.stderr
        ok = res.returncode == 0
    with open(os.path.join(LIBDIR, "build.log"), "w") as fh:
        fh.write(log)
    if not ok:
        sys.stderr.write(log)
        raise RuntimeError("nvcc failed building libwdx_b200.so")
    with open(STAMP, "w") as fh:
        fh.write(_source_digest() + "\n")
    if verbose:
        print(log)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
