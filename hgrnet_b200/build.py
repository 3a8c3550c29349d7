"""Build libhgr_b200.so (sm_100a) in-tree with nvcc.

``python -m hgrnet_b200.build [--force]``.  Objects and the shared library land in
``hgrnet_b200/lib/`` (git-ignored; they travel to the GPU box with the gpurun snapshot).
nvcc cross-compiles for sm_100a without a GPU.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libhgr_b200.so")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")

SOURCES = ["hgr_abi.cu", "aggregate_norm.cu", "topk_merge.cu", "score_simt.cu", "score_launch.cu", "score_pair.cu",
           "masked_ce.cu", "om_backward.cu", "hier_metrics.cu", "hier_mistakes.cu",
           "class_hits.cu"]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
NVCC_FLAGS = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr",
              "-Xptxas", "-v"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; set NVCC=/path/to/nvcc")


def _deps():
    out = [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    out.append(os.path.join(INCLUDE, "hgr_b200.h"))
    return out


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(p) > t for p in _deps())


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    os.makedirs(LIBDIR, exist_ok=True)
    nvcc = _nvcc()
    logs = {}

    def compile_one(src):
        obj = os.path.join(LIBDIR, src.replace(".cu", ".o"))
        cmd = [nvcc, *ARCH, *NVCC_FLAGS, *os.environ.get("HGR_NVCC_EXTRA", "").split(), "-I", INCLUDE, "-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        logs[src] = r.stdout + r.stderr
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s" % (src, logs[src]))
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    link = [nvcc, *ARCH, "-shared", "-cudart", "static", "-o", LIB, *objs]
    r = subprocess.run(link, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + r.stdout + r.stderr)
    with open(os.path.join(LIBDIR, "ptxas.log"), "w") as f:
        for src in SOURCES:
            f.write("==== %s ====\n%s\n" % (src, logs[src]))
    if verbose:
        for src in SOURCES:
            print("==== %s ====\n%s" % (src, logs[src]))
    return LIB


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(path)
