"""Builds libls_cuda.so in-tree for sm_100a (nvcc cross-compiles without a GPU).

    python -m fast_solver_lippmann_schwinger_b200.build [--force] [--verbose]
"""
from __future__ import annotations

import concurrent.futures as cf
import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
OBJDIR = os.path.join(HERE, "build")
LIB = os.path.join(LIBDIR, "libls_cuda.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr",
]


def _nvcc():
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found - libls_cuda.so cannot be built")
    return nvcc


def _sources():
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cu"))


def _digest():
    h = hashlib.sha256()
    for root in (CSRC, os.path.join(ROOT, "include")):
        for f in sorted(os.listdir(root)):
            if f.endswith((".cu", ".cuh", ".h")):
                with open(os.path.join(root, f), "rb") as fh:
                    h.update(f.encode())
                    h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(LIBDIR, exist_ok=True)
    os.makedirs(OBJDIR, exist_ok=True)
    stamp = os.path.join(LIBDIR, "libls_cuda.sha256")
    digest = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read().strip() == digest:
        return LIB
    nvcc = _nvcc()
    extra = ["-Xptxas", "-v"] if verbose else []

    def compile_one(src):
        obj = os.path.join(OBJDIR, os.path.basename(src)[:-3] + ".o")
        cmd = [nvcc] + NVCC_FLAGS + extra + ["-I", os.path.join(ROOT, "include"), "-c", src, "-o", obj]
        p = subprocess.run(cmd, capture_output=True, text=True)
        if p.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, p.stdout, p.stderr))
        if verbose:
            sys.stderr.write(p.stderr)
        return obj

    with cf.ThreadPoolExecutor(max_workers=os.cpu_count() or 4) as ex:
        objs = list(ex.map(compile_one, _sources()))
    link = [nvcc, "-shared", "--cudart", "shared", "-o", LIB] + objs
    nccl_dir = _nccl_libdir()
    if nccl_dir:
        link += ["-L" + nccl_dir, "-l:libnccl.so.2", "-Xlinker", "-rpath", "-Xlinker", nccl_dir]
    else:
        link += ["-lnccl"]
    cublas_dir = _pip_libdir("nvidia.cublas", "libcublas.so.12")      # the copy torch loads too: one cuBLAS per process
    if cublas_dir:
        link += ["-L" + cublas_dir, "-l:libcublas.so.12", "-Xlinker", "-rpath", "-Xlinker", cublas_dir]
    else:
        link += ["-lcublas"]
    cusolver_dir = _pip_libdir("nvidia.cusolver", "libcusolver.so.11")
    if cusolver_dir:
        link += ["-L" + cusolver_dir, "-l:libcusolver.so.11", "-Xlinker", "-rpath", "-Xlinker", cusolver_dir]
    else:
        link += ["-lcusolver"]
    p = subprocess.run(link, capture_output=True, text=True)
    if p.returncode != 0:
        raise RuntimeError("link failed:\n%s\n%s" % (p.stdout, p.stderr))
    with open(stamp, "w") as fh:
        fh.write(digest + "\n")
    return LIB


def _pip_libdir(module, soname):
    try:
        import importlib.util
        spec = importlib.util.find_spec(module)
        if spec and spec.submodule_search_locations:
            d = os.path.join(list(spec.submodule_search_locations)[0], "lib")
            if os.path.exists(os.path.join(d, soname)):
                return d
    except Exception:
        pass
    return None


def _nccl_libdir():
    return _pip_libdir("nvidia.nccl", "libnccl.so.2")


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
