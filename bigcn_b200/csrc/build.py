"""Build libbigcn_b200.so in-tree with nvcc for sm_100a (no torch dependency)."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = ["api.cu", "graph_prep.cu", "xw.cu", "xsparse.cu", "gemm_tc.cu", "propagate.cu", "rootdense.cu", "head.cu", "loader.cu", "weighted.cu", "feeder.cu", "ebgcn.cu"]
HOST_SOURCES = ["host_compact.cpp"]      # host-only C++ (g++), linked into the same library
HEADERS = ["common.cuh", "kernels.cuh", "gather.cuh", "tc.cuh", os.path.join("..", "..", "include", "bigcn_b200.h")]
LIB = os.path.join(HERE, "..", "libbigcn_b200.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
         "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr", "-cudart", "static"]


def _stale() -> bool:
    lib = os.path.normpath(LIB)
    if not os.path.exists(lib):
        return True
    t = os.path.getmtime(lib)
    deps = [os.path.join(HERE, f) for f in SOURCES + HOST_SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    lib = os.path.normpath(LIB)
    if not force and not _stale():
        return lib
    objs = []
    procs = []
    for s in SOURCES:
        o = os.path.join(HERE, s.replace(".cu", ".o"))
        cmd = [NVCC, *FLAGS, "-c", os.path.join(HERE, s), "-o", o]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(o)
    for s in HOST_SOURCES:
        o = os.path.join(HERE, s.replace(".cpp", ".o"))
        cmd = [os.environ.get("CXX", "g++"), "-O3", "-std=c++17", "-fPIC", "-pthread", "-c", os.path.join(HERE, s), "-o", o]
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(o)
    failed = False
    for s, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            failed = True
            sys.stderr.write(f"nvcc failed on {s}:\n{out}\n")
        elif verbose or out.strip():
            sys.stderr.write(out)
    if failed:
        raise RuntimeError("nvcc compilation failed")
    subprocess.check_call([NVCC, "-shared", *FLAGS[:2], "-cudart", "static", "-Xcompiler", "-pthread", "-o", lib, *objs])
    return lib


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
