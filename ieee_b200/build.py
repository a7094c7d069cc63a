"""Build ieee_b200/libieee_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m ieee_b200.build [--force]

The library links the CUDA runtime statically and has no other dependency, so the built file
travels to the GPU box as is.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libieee_b200.so")
SOURCES = ["capi.cu", "pack.cu", "distmat_sm100.cu", "distmat_simt.cu", "rank.cu", "rerank.cu"]
HEADERS = [os.path.join(CSRC, "common.cuh"), os.path.join(os.path.dirname(HERE), "include", "ieee_b200.h")]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]


def nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.isfile(cand):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build() -> bool:
    if not os.path.isfile(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + HEADERS
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = True) -> str:
    if not force and not needs_build():
        return LIB
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    flags = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr",
             "-Xptxas", "-v" if verbose else "-O3"] + ARCH
    objs, procs = [], []
    for src in SOURCES:
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        objs.append(obj)
        cmd = [nvcc(), "-c", os.path.join(CSRC, src), "-o", obj] + flags
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            failed = True
            print(f"[build] {src} FAILED\n{out}")
        elif verbose:
            lines = [l for l in out.splitlines() if "registers" in l or "spill" in l or "warning" in l.lower()]
            print(f"[build] {src} ok" + ("".join("\n    " + l.strip() for l in lines[:40]) if lines else ""))
    if failed:
        raise RuntimeError("nvcc failed")
    subprocess.run([nvcc(), "-shared", "-o", LIB] + objs + ARCH + ["-cudart", "static"], check=True)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv))
