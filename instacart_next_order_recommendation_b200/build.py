"""Builds libicr_b200.so in-tree with nvcc for sm_100a (no torch types, plain C ABI)."""

from __future__ import annotations

import hashlib
import os
import subprocess
import sys
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
LIB_DIR = PKG / "lib"
LIB_PATH = LIB_DIR / "libicr_b200.so"
SOURCES = ["api.cu", "prep.cu", "gemv_topk.cu", "select.cu", "select_hist.cu", "dense.cu", "mnrl.cu", "mnrl_tc.cu", "metrics.cu", "exchange.cu", "gemm_topk.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC",
    "--expt-relaxed-constexpr",
] + os.environ.get("ICR_NVCC_DEFS", "").split()  # e.g. ICR_NVCC_DEFS="-DICR_HS_WARPS=6" for tuning experiments


def _nvcc() -> str:
    cand = os.environ.get("NVCC") or "/usr/local/cuda/bin/nvcc"
    return cand if Path(cand).exists() else "nvcc"


def source_digest() -> str:
    h = hashlib.sha256()
    for p in sorted(list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cuh")) + [PKG.parent / "include" / "icr_b200.h"]):
        h.update(p.name.encode())
        h.update(p.read_bytes())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build_trace() -> Path:
    """Development build with the per-CTA %globaltimer stamps of the K1 ring kernel (benchmarks/k1_trace.py):
    lib/libicr_b200_trace.so, selected at run time with ICR_B200_LIB. Never the product library."""
    LIB_DIR.mkdir(exist_ok=True)
    out = LIB_DIR / "libicr_b200_trace.so"
    tdir = LIB_DIR / "trace_obj"
    tdir.mkdir(exist_ok=True)
    procs = []
    for src in SOURCES:
        cmd = [_nvcc(), *NVCC_FLAGS, "-DICR_TRACE", "-c", str(CSRC / src), "-o", str(tdir / (src + ".o"))]
        procs.append(subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    for p in procs:
        o, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError("nvcc failed building the trace library:\n" + o)
    subprocess.run([_nvcc(), "-shared", "-cudart", "static", "-o", str(out), *[str(tdir / (s + ".o")) for s in SOURCES]], check=True)
    return out


def build(force: bool = False, verbose: bool = False) -> Path:
    """Compile every .cu of the package into lib/libicr_b200.so (skipped when up to date)."""
    LIB_DIR.mkdir(exist_ok=True)
    stamp = LIB_DIR / "libicr_b200.digest"
    digest = source_digest()
    if not force and LIB_PATH.exists() and stamp.exists() and stamp.read_text() == digest:
        # the stamp is tracked by git: a checkout can restore it next to a library built from other sources, so the library
        # must also be newer than every source it was built from
        newest = max(p.stat().st_mtime for p in list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cuh")) + [PKG.parent / "include" / "icr_b200.h"])
        if LIB_PATH.stat().st_mtime >= newest:
            return LIB_PATH
    objs = []
    procs = []
    for src in SOURCES:
        obj = LIB_DIR / (src + ".o")
        cmd = [_nvcc(), *NVCC_FLAGS, "-c", str(CSRC / src), "-o", str(obj)]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(str(obj))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            sys.stderr.write(f"--- nvcc {src} ---\n{out}\n")
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed building libicr_b200.so")
    link = [_nvcc(), "-shared", "-cudart", "static", "-o", str(LIB_PATH), *objs]
    subprocess.run(link, check=True)
    stamp.write_text(digest)
    return LIB_PATH


if __name__ == "__main__":
    if "--trace" in sys.argv:
        print(build_trace())
        sys.exit(0)
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
