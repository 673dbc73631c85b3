"""Builds squid_b200/libsquid_b200.so in-tree: the sm_100a CUDA kernels + C ABI + C++ host twin.

    python -m squid_b200.build [--force]

nvcc cross-compiles without a GPU.  The .so is git-ignored but travels to the GPU box with the repo snapshot.
"""
from __future__ import annotations

import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "squid_b200", "csrc")
OUT = os.path.join(ROOT, "squid_b200", "libsquid_b200.so")
CU = ["sqg_api.cu", "sqg_load.cu", "sqg_bam.cu", "sqg_prepass.cu", "sqg_classify.cu", "sqg_nodes.cu", "sqg_edges.cu", "sqg_cov.cu"]
CPP = ["host/readrec.cpp", "host/chimeric.cpp", "host/prepass.cpp", "host/host_api.cpp", "host/plan.cpp", "host/bam.cpp", "host/exactbp.cpp", "host/writeio.cpp", "host/wire.cpp"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC,-fopenmp,-Wno-deprecated-declarations",
              "-Wno-deprecated-declarations", "-I", os.path.join(ROOT, "include"), "-I", CSRC]


def sources():
    out = [os.path.join(CSRC, f) for f in CU + CPP]
    for d, _, fs in os.walk(CSRC):
        out += [os.path.join(d, f) for f in fs if f.endswith((".cuh", ".h"))]
    out += [os.path.join(ROOT, "include", f) for f in os.listdir(os.path.join(ROOT, "include"))]
    return out


def up_to_date() -> bool:
    if not os.path.exists(OUT):
        return False
    t = os.path.getmtime(OUT)
    return all(os.path.getmtime(s) <= t for s in sources())


def build(force: bool = False, verbose: bool = True) -> str:
    if not force and up_to_date():
        return OUT
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    extra = os.environ.get("SQUID_NVCC_EXTRA", "").split()
    bdir = os.path.join(ROOT, "build")
    os.makedirs(bdir, exist_ok=True)
    objs = []
    procs = []
    for f in CU + CPP:
        o = os.path.join(bdir, f.replace("/", "_") + ".o")
        objs.append(o)
        cmd = [nvcc] + NVCC_FLAGS + extra + (["-x", "cu"] if f.endswith(".cu") else []) + ["-c", os.path.join(CSRC, f), "-o", o]
        if verbose:
            print(" ".join(cmd), flush=True)
        procs.append((f, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for f, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError("nvcc failed on %s:\n%s" % (f, out))
    cmd = [nvcc, "-shared", "-o", OUT] + objs + ["-lpthread", "-lgomp", "-lz"]
    if verbose:
        print(" ".join(cmd), flush=True)
    subprocess.run(cmd, check=True)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv))
