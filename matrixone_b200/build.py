"""Build libmo_b200.so (the C-ABI library, include/mo_b200.h) with nvcc for sm_100a, in-tree.

    python -m matrixone_b200.build [--force] [--verbose]

Plain nvcc, no torch extension machinery: the library links only the CUDA runtime (static) so the Go side can load
it with cgo exactly like the reference's libmo.a + cuda.o (cgo/Makefile:15-21).
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libmo_b200.so")
OBJ = os.path.join(HERE, "build")
SOURCES = ["runtime.cu", "agg.cu", "tpch.cu", "elementwise.cu", "goelem.cu", "colops.cu", "join.cu", "strhash.cu", "kmeans.cu", "lz4.cu", "vecdecode.cu", "plan.cu", "decimal.cu", "bloom.cu", "distance.cu", "search.cu", "tcsearch.cu", "xcall.cu", "datagen.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC",
         "--expt-relaxed-constexpr", "-Xptxas", "-v"]


def _run(cmd):
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError("command failed: %s\n%s" % (" ".join(cmd), r.stdout))
    return r.stdout


def _deps_mtime():
    m = 0.0
    for root in (CSRC, os.path.join(HERE, "..", "include")):
        for f in os.listdir(root):
            if f.endswith((".cuh", ".h")):
                m = max(m, os.path.getmtime(os.path.join(root, f)))
    return m


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    hdr = _deps_mtime()
    todo, objs = [], []
    for s in SOURCES:
        src = os.path.join(CSRC, s)
        obj = os.path.join(OBJ, s.replace(".cu", ".o"))
        objs.append(obj)
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < max(os.path.getmtime(src), hdr):
            todo.append((src, obj))
    logs = {}

    def compile_one(so):
        src, obj = so
        logs[os.path.basename(src)] = _run([NVCC] + FLAGS + ["-c", src, "-o", obj])

    if todo:
        with ThreadPoolExecutor(max_workers=min(8, len(todo))) as ex:
            list(ex.map(compile_one, todo))
    if todo or not os.path.exists(OUT):
        _run([NVCC, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", OUT] + objs)
    if verbose:
        for k, v in logs.items():
            print("==", k)
            print(v)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
