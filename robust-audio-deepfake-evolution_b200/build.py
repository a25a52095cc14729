"""Build libbimamba_sm100.so in-tree with nvcc (sm_100a only; cross-compiles without a GPU).

    python robust-audio-deepfake-evolution_b200/build.py [--force]
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libbimamba_sm100.so")
SOURCES = ("api.cu", "scan_fwd.cu", "scan_fwd1.cu", "scan_fwd_split.cu", "scan_bwd1.cu", "conv.cu", "layernorm.cu", "gemm.cu", "pack.cu", "optim.cu", "head.cu", "eltwise.cu", "block.cu", "fusion.cu")
HEADERS = ("common.cuh", os.path.join("..", "..", "include", "bimamba.h"))

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-DBIMAMBA_BUILD",
]


def _nvcc() -> str:
    cand = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(cand):
        raise RuntimeError("nvcc not found; the Bi-Mamba CUDA library cannot be built")
    return cand


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + [os.path.normpath(os.path.join(CSRC, h)) for h in HEADERS]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = True, defines=(), variant: str = "") -> str:
    """Build the library.  `variant` + `defines` build an experiment copy `_variants/libbimamba_sm100_<variant>.so`
    with extra -D flags (A/B runs load it through the BIMAMBA_LIB environment variable, see _lib.py)."""
    if variant:
        return _build_variant(variant, list(defines), verbose)
    if not force and not _stale():
        return LIB
    return _compile(CSRC, LIB, [], verbose)


def _build_variant(variant: str, defines, verbose: bool) -> str:
    vdir = os.path.join(HERE, "_variants")
    odir = os.path.join(vdir, "obj_" + variant)
    os.makedirs(odir, exist_ok=True)
    return _compile(odir, os.path.join(vdir, f"libbimamba_sm100_{variant}.so"), ["-D" + d for d in defines], verbose)


def _compile(objdir: str, lib: str, extra, verbose: bool) -> str:
    nvcc = _nvcc()
    objs = []
    procs = []
    for s in SOURCES:
        obj = os.path.join(objdir, s.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + extra + ["-c", os.path.join(CSRC, s), "-o", obj]
        if verbose:
            print(" ".join(cmd), flush=True)
        procs.append((cmd, subprocess.Popen(cmd)))
        objs.append(obj)
    for cmd, p in procs:
        if p.wait() != 0:
            raise RuntimeError("nvcc failed: " + " ".join(cmd))
    cmd = [nvcc, "-shared", "-cudart", "static", "-gencode", "arch=compute_100a,code=sm_100a", "-o", lib] + objs
    if verbose:
        print(" ".join(cmd), flush=True)
    subprocess.check_call(cmd)
    return lib


if __name__ == "__main__":
    # python build.py [--force] [--variant NAME -DX=1 ...]
    argv = sys.argv[1:]
    var = argv[argv.index("--variant") + 1] if "--variant" in argv else ""
    print(build(force="--force" in argv, defines=[a[2:] for a in argv if a.startswith("-D")], variant=var))
