"""In-tree nvcc build of libpynqs_b200.so for sm_100a (no JIT cache: the .so travels with the tree)."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(CSRC, "libpynqs_b200.so")
SOURCES = ["abi.cu", "enumerate.cu", "hij.cu", "lut.cu", "eloc_scan.cu", "eloc_block.cu", "hamiltonian.cu", "spmm.cu", "spin.cu", "rdm.cu", "pt2.cu", "gindex.cu", "convert.cu", "reduce_sample.cu", "compact.cu", "peer.cu", "prepare.cu", "table.cu"]
HEADERS = ["common.cuh", "lut.cuh", "tables.cuh", "prepare.cuh", "gindex.cuh", "eloc.cuh", "rederive.cuh", "enum_rows.cuh", os.path.join("..", "..", "include", "pynqs_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC",
    "-prec-sqrt=true", "-prec-div=true", "-fmad=true",
    "-Xptxas", "-v",
]


def nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: cannot build libpynqs_b200.so")
    return exe


def stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not stale():
        return LIB
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(CSRC, src.replace(".cu", ".o"))
        cmd = [nvcc(), *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    log = []
    for src, p in procs:
        out, _ = p.communicate()
        log.append(f"==== {src}\n{out}")
        if p.returncode != 0:
            sys.stderr.write("\n".join(log))
            raise RuntimeError(f"nvcc failed on {src}")
    with open(os.path.join(CSRC, "ptxas_v.log"), "w") as f:
        f.write("\n".join(log))
    subprocess.check_call([nvcc(), "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a"])
    if verbose:
        print("\n".join(log))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
