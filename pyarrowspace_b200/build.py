"""Builds pyarrowspace_b200/libarrowspace_b200.so from csrc/*.cu with nvcc for sm_100a.

In-tree build (the .so travels to the GPU box with the repo snapshot).  Usage:
    python -m pyarrowspace_b200.build [--force] [--verbose] [--profiling]
"""
import concurrent.futures
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "_obj")
LIB = os.path.join(HERE, "libarrowspace_b200.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")

SOURCES = ["api.cu", "tensormap.cu", "gram.cu", "graph_select.cu", "csr.cu", "taumode.cu", "search.cu", "search_tc.cu", "knn.cu", "peer.cu", "reduce.cu", "range.cu"]
FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O2", "-ccbin", "/usr/bin/g++",
]


def _deps_mtime():
    m = 0.0
    for root in (CSRC, os.path.join(HERE, "..", "include")):
        for fn in os.listdir(root):
            if fn.endswith((".cuh", ".h")):
                m = max(m, os.path.getmtime(os.path.join(root, fn)))
    return m


def _compile(src, verbose, profiling=False):
    obj = os.path.join(OBJ, src.replace(".cu", ".o"))
    cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + (["-DASP_PROFILING"] if profiling else []) + \
        ["-c", os.path.join(CSRC, src), "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    return src, r.returncode, r.stdout + r.stderr


def build(force=False, verbose=False, profiling=False):
    """profiling=True (--profiling) compiles the diagnostic kernel variants in (ASP_TC_VARIANT: results are wrong under
    them); the default build has none.  A profiling build forces a full recompile, and so does the next default build."""
    marker = os.path.join(OBJ, ".profiling")
    if profiling or os.path.exists(marker):
        force = True
    os.makedirs(OBJ, exist_ok=True)
    hdr = _deps_mtime()
    todo = []
    for src in SOURCES:
        obj = os.path.join(OBJ, src.replace(".cu", ".o"))
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < max(hdr, os.path.getmtime(os.path.join(CSRC, src))):
            todo.append(src)
    if todo:
        with concurrent.futures.ThreadPoolExecutor(max_workers=min(8, len(todo))) as ex:
            for src, rc, out in ex.map(lambda s: _compile(s, verbose, profiling), todo):
                if verbose or rc != 0:
                    sys.stderr.write("---- %s\n%s\n" % (src, out))
                if rc != 0:
                    raise RuntimeError("nvcc failed on %s" % src)
    if profiling:
        open(marker, "w").close()
    elif os.path.exists(marker):
        os.remove(marker)
    objs = [os.path.join(OBJ, s.replace(".cu", ".o")) for s in SOURCES]
    if todo or not os.path.exists(LIB):
        cmd = [NVCC, "-shared", "-o", LIB, "-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static",
               "-ccbin", "/usr/bin/g++"] + objs
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("link failed")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv, profiling="--profiling" in sys.argv))
