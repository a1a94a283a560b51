"""Build libemagls_cuda.so (sm_100a) in-tree with nvcc.  No torch involved."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libemagls_cuda.so")
SOURCES = ["setup_kernels.cu", "solver_kernels.cu", "tsqr_kernels.cu", "gram_kernels.cu", "ozaki_kernels.cu", "ema_kernels.cu", "engine.cu", "generic_engine.cu", "render.cu", "tracked_render.cu", "frontend.cu", "api.cu"]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]


def _nvcc() -> str:
    for c in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found")


def _stale(target: str, deps: list[str]) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(LIBDIR, exist_ok=True)
    nvcc = _nvcc()
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(os.path.dirname(HERE), "include", "emagls_cuda.h"))
    objs = []
    procs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(LIBDIR, src.replace(".cu", ".o"))
        objs.append(o)
        if force or _stale(o, [s] + headers):
            cmd = [nvcc, *ARCH, "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC", "-c", s, "-o", o]
            if verbose:
                cmd.insert(1, "-Xptxas=-v")
            procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            failed = True
            sys.stderr.write(f"--- nvcc {src} failed ---\n{out}\n")
        elif verbose:
            print(out)
    if failed:
        raise RuntimeError("nvcc failed")
    if force or procs or _stale(LIB, objs):
        cmd = [nvcc, *ARCH, "-shared", "-o", LIB, *objs, "-lcufft", "-lcudart"]
        subprocess.run(cmd, check=True)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
