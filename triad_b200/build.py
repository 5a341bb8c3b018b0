"""Builds libtriad_b200.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

The library has no torch / python dependency: plain `nvcc -shared`, cudart linked statically,
the one driver entry point (cuTensorMapEncodeTiled) resolved at run time, so the .so loads on a
machine without a GPU driver (the CPU test tier checks the exported symbols there).
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIBNAME = "libtriad_b200.so"

SOURCES = ["capi.cu", "maxmean_simt.cu", "maxmean_tc.cu", "infonce.cu", "maxmean_bwd.cu", "bwd_dq_tile.cu", "bwd_dq_pipe.cu", "retrieve.cu", "dense_reg.cu", "pack.cu", "proj_head.cu", "pospair.cu", "dense_gemm.cu", "quant_e4m3.cu", "tmap.cu", "ragged.cu"]
HEADERS = ["common.cuh", "ptx.cuh", "triad_round.h", os.path.join("..", "..", "include", "triad_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC",
    "--expt-relaxed-constexpr",
    "-Xptxas", "-v",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (set NVCC=...)")


def lib_path() -> str:
    return os.path.join(LIBDIR, LIBNAME)


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(LIBDIR, exist_ok=True)
    objdir = os.path.join(LIBDIR, "obj")
    os.makedirs(objdir, exist_ok=True)
    nvcc = _nvcc()
    hdrs = [os.path.normpath(os.path.join(CSRC, h)) for h in HEADERS]
    objs = []
    procs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(objdir, src.replace(".cu", ".o"))
        objs.append(o)
        if force or _stale(o, [s] + hdrs):
            cmd = [nvcc] + NVCC_FLAGS + ["-c", s, "-o", o]
            procs.append((src, o, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, o, p in procs:
        out, _ = p.communicate()
        with open(o + ".log", "w") as f:
            f.write(out)
        if p.returncode != 0:
            failed = True
            sys.stderr.write(f"---- nvcc failed for {src} ----\n{out}\n")
        elif verbose:
            sys.stderr.write(f"---- {src} ----\n{out}\n")
    if failed:
        raise RuntimeError("nvcc compilation failed")
    target = lib_path()
    if force or procs or _stale(target, objs):
        cmd = [nvcc, "-shared", "-o", target] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static"]
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n" + r.stdout)
    return target


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
