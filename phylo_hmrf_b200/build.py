"""In-tree build of the native libraries (nvcc cross-compiles sm_100a without a GPU).

    python -m phylo_hmrf_b200.build [--force]

* ``lib/libphmrf.so``      hand-written CUDA kernels + the C ABI of include/phmrf.h
* ``lib/libphmrf_probe.so``  pipe probes for the roofline denominators (bench/tools only; include/phmrf_probe.h)
* ``lib/libphmrf_gco.so``  host graph cut (csrc/gco.cpp, include/phmrf_gco.h): GCO v3.0's
  alpha-beta swap and alpha-expansion on a general graph
"""
from __future__ import annotations

import concurrent.futures as cf
import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "lib")
OBJ = os.path.join(PKG, "build")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
CU_SOURCES = ["api.cu", "kernels_a.cu", "kernels_b.cu", "kernels_b3.cu", "kernels_b3_d58.cu", "kernels_b3_d9c.cu", "kernels_grid.cu", "kernels_prep.cu"]


def _nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _newer(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def _run(cmd):
    p = subprocess.run(cmd, capture_output=True, text=True)
    if p.returncode != 0:
        raise RuntimeError("build failed: %s\n%s\n%s" % (" ".join(cmd), p.stdout, p.stderr))
    return p.stdout + p.stderr


def build_cuda(force=False, verbose=False):
    os.makedirs(LIB, exist_ok=True)
    os.makedirs(OBJ, exist_ok=True)
    out = os.path.join(LIB, "libphmrf.so")
    headers = [os.path.join(CSRC, "common.cuh"), os.path.join(CSRC, "estep_common.cuh"), os.path.join(CSRC, "estep_bulk.cuh"),
               os.path.join(PKG, "..", "include", "phmrf.h")]
    srcs = [os.path.join(CSRC, s) for s in CU_SOURCES]
    if not force and not _newer(out, srcs + headers):
        return out
    nvcc = _nvcc()
    objs = []

    def compile_one(src):
        obj = os.path.join(OBJ, os.path.basename(src) + ".o")
        if force or _newer(obj, [src] + headers):
            cmd = [nvcc] + ARCH + ["-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC", "-c", src, "-o", obj]
            if verbose:
                cmd.insert(1, "-Xptxas=-v")
            log = _run(cmd)
            if verbose:
                print(log)
        return obj

    with cf.ThreadPoolExecutor(max_workers=len(srcs)) as ex:
        objs = list(ex.map(compile_one, srcs))
    _run([nvcc] + ARCH + ["-shared", "-o", out] + objs)
    return out


def build_probe(force=False):
    """lib/libphmrf_probe.so: the pipe probes (csrc/probe.cu, include/phmrf_probe.h) -- a measurement tool for
    bench.py and tools/, kept out of the product library."""
    os.makedirs(LIB, exist_ok=True)
    out = os.path.join(LIB, "libphmrf_probe.so")
    src = os.path.join(CSRC, "probe.cu")
    hdr = os.path.join(PKG, "..", "include", "phmrf_probe.h")
    if not force and not _newer(out, [src, hdr]):
        return out
    _run([_nvcc()] + ARCH + ["-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC", "-shared", src, "-o", out])
    return out


def build_gco(force=False):
    os.makedirs(LIB, exist_ok=True)
    out = os.path.join(LIB, "libphmrf_gco.so")
    src = os.path.join(CSRC, "gco.cpp")
    hdr = os.path.join(PKG, "..", "include", "phmrf_gco.h")
    if not force and not _newer(out, [src, hdr]):
        return out
    _run(["g++", "-O2", "-Wall", "-fPIC", "-shared", "-std=gnu++17", "-o", out, src])
    return out


def build_all(force=False, verbose=False):
    return build_cuda(force, verbose), build_gco(force), build_probe(force)


if __name__ == "__main__":
    print(build_all(force="--force" in sys.argv, verbose="-v" in sys.argv))
