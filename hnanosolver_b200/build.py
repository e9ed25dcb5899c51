"""Builds libhns_b200.so (the product: CUDA kernels + C ABI) in-tree with nvcc for sm_100a.

    python -m hnanosolver_b200.build [--verbose] [--force]

The shared library lands next to this file so that it travels with the repository snapshot to the GPU box.
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libhns_b200.so")
SOURCES = ["topology.cu", "kernels.cu", "api.cu", "dist.cu", "nvdb_io.cu", "multigrid.cu", "advect.cu", "domain.cu", "export.cu"]
HEADERS = ["common.cuh", "kernels.cuh", "sampling.cuh", "nvdb_layout.cuh", "classify.cuh", os.path.join("..", "..", "include", "hns_b200.h")]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-Wall",
]


def _stale() -> bool:
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(verbose: bool = False, force: bool = False) -> str:
    if not force and not _stale():
        return OUT
    nvcc = os.environ.get("NVCC", "nvcc")
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(CSRC, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd[1:1] = ["-Xptxas", "-v"]
            print(" ".join(cmd), flush=True)
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write(out)
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", OUT, *objs, "-lcudart", "-ldl"]
    subprocess.check_call(cmd)
    return OUT


if __name__ == "__main__":
    print(build(verbose="--verbose" in sys.argv, force="--force" in sys.argv))
