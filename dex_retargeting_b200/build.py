"""In-tree build of libdexr.so (nvcc, sm_100a only).  `python -m dex_retargeting_b200.build [--force]`"""
from __future__ import annotations

import hashlib
import shutil
import subprocess
import sys
from pathlib import Path

PKG = Path(__file__).resolve().parent
SRC = PKG / "csrc" / "dexr.cu"
DEPS = [SRC, PKG / "csrc" / "dexr_kernels.cuh", PKG.parent / "include" / "dexr.h"]
OUT = PKG / "libdexr.so"

NVCC_FLAGS = [
    "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
    "-Xptxas", "-v", "-shared", "-Xcompiler", "-fPIC",
]


def find_nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found: the CUDA library cannot be built (there is no CPU fallback)")


# Experimental builds (csrc/dexr_kernels.cuh, "Experiment switches"): one library per entry under variants/, loaded with
# DEXR_LIBRARY=<path>.  They are A/B material for tools/ab_variants.sh, never the default.
VARIANTS = {
    "fastsincos": ["-DDEXR_EXP_FASTSINCOS"],
    "multi_calls": ["-DDEXR_EXP_MULTI_CALLS"],
}


def source_id(variant: str = "") -> str:
    """16 hex digits over the library's sources and compile-time switches (what `dexr_build_id()` returns)."""
    h = hashlib.sha256()
    for d in DEPS:
        h.update(d.read_bytes())
    h.update(" ".join(VARIANTS[variant] if variant else []).encode())
    return h.hexdigest()[:16]


def build_library(force: bool = False, verbose: bool = True, variant: str = "") -> Path:
    out = PKG / "variants" / f"libdexr_{variant}.so" if variant else OUT
    log_path = PKG / "csrc" / (f"build_{variant}.log" if variant else "build.log")
    if not force and out.exists() and all(out.stat().st_mtime >= d.stat().st_mtime for d in DEPS):
        return out
    out.parent.mkdir(exist_ok=True)
    cmd = [find_nvcc(), *NVCC_FLAGS, *(VARIANTS[variant] if variant else []), f'-DDEXR_BUILD_ID="{source_id(variant)}"',
           "-o", str(out), str(SRC)]
    if verbose:
        print(" ".join(cmd), flush=True)
    res = subprocess.run(cmd, capture_output=True, text=True)
    log = (res.stdout or "") + (res.stderr or "")
    log_path.write_text(log)
    if res.returncode != 0:
        sys.stderr.write(log)
        raise RuntimeError(f"nvcc failed building {out.name}")
    if verbose:
        for line in log.splitlines():
            if "registers" in line or "spill" in line:
                print(line)
    return out


# The backward pass (include/dexr_grad.h) is a second library: libdexr.so stays the binary its build id and profiles name.
GRAD_SRC = PKG / "csrc" / "dexr_grad.cu"
GRAD_DEPS = [GRAD_SRC, PKG / "csrc" / "dexr_grad_kernels.cuh", PKG / "csrc" / "dexr_grad_seq_kernels.cuh",
             PKG / "csrc" / "dexr_kernels.cuh", PKG.parent / "include" / "dexr_grad.h", PKG.parent / "include" / "dexr.h"]
GRAD_OUT = PKG / "libdexr_grad.so"


def grad_source_id() -> str:
    """16 hex digits over the backward library's sources and the headers they include (what `dexr_grad_build_id()` returns)."""
    h = hashlib.sha256()
    for d in GRAD_DEPS:
        h.update(d.read_bytes())
    return h.hexdigest()[:16]


def build_grad_library(force: bool = False, verbose: bool = True) -> Path:
    log_path = PKG / "csrc" / "build_grad.log"
    if not force and GRAD_OUT.exists() and all(GRAD_OUT.stat().st_mtime >= d.stat().st_mtime for d in GRAD_DEPS):
        return GRAD_OUT
    cmd = [find_nvcc(), *NVCC_FLAGS, f'-DDEXR_GRAD_BUILD_ID="{grad_source_id()}"', "-o", str(GRAD_OUT), str(GRAD_SRC)]
    if verbose:
        print(" ".join(cmd), flush=True)
    res = subprocess.run(cmd, capture_output=True, text=True)
    log = (res.stdout or "") + (res.stderr or "")
    log_path.write_text(log)
    if res.returncode != 0:
        sys.stderr.write(log)
        raise RuntimeError(f"nvcc failed building {GRAD_OUT.name}")
    if verbose:
        for line in log.splitlines():
            if "registers" in line or "spill" in line or "Compiling entry" in line:
                print(line)
    return GRAD_OUT


if __name__ == "__main__":
    build_library(force="--force" in sys.argv)
    build_grad_library(force="--force" in sys.argv)
    if "--variants" in sys.argv:
        for name in VARIANTS:
            build_library(force="--force" in sys.argv, variant=name)
