"""Build libdlrm_b200.so (sm_100a) in-tree with nvcc.  No torch, no JIT cache.

    python -m dlrm_jl_b200.csrc.build [--force] [--verbose]
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
LIB_DIR = os.path.join(os.path.dirname(HERE), "lib")
LIB_PATH = os.path.join(LIB_DIR, "libdlrm_b200.so")
SOURCES = ["api.cu", "lookup.cu", "interact.cu", "interact_warp.cu", "sort.cu", "update.cu", "loss.cu", "dense.cu", "p2p.cu", "loader.cu", "comm.cu"]
HEADERS = [os.path.join(HERE, "common.cuh"), os.path.join(HERE, "sort_small.cuh"), os.path.join(HERE, "pool_bag.cuh"), os.path.join(ROOT, "include", "dlrm_b200.h")]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC,-O3,-Wall,-Wno-unused-function",
    "-I", os.path.join(ROOT, "include"), "-I", HERE,
]


def _nvcc() -> str:
    cand = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(cand):
        raise RuntimeError("nvcc not found: libdlrm_b200.so cannot be built")
    return cand


def needs_build() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(HERE, s) for s in SOURCES] + HEADERS
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB_PATH
    os.makedirs(LIB_DIR, exist_ok=True)
    obj_dir = os.path.join(LIB_DIR, "obj")
    os.makedirs(obj_dir, exist_ok=True)
    nvcc = _nvcc()
    procs = []
    objs = []
    for src in SOURCES:
        obj = os.path.join(obj_dir, src.replace(".cu", ".o"))
        objs.append(obj)
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(HERE, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
            print(" ".join(cmd), flush=True)
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            failed = True
            sys.stderr.write(f"--- nvcc failed on {src} ---\n{out}\n")
        elif verbose or out.strip():
            sys.stderr.write(out)
    if failed:
        raise RuntimeError("nvcc compilation failed")
    cmd = [nvcc, "-shared", "-o", LIB_PATH, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-lcudart", "-ldl"]
    subprocess.run(cmd, check=True)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
