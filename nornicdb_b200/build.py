"""Build libnornic_knn.so (sm_100a) in-tree with nvcc.  No GPU is needed to build.

The library is plain CUDA C++ + cudart (no torch, no cuBLAS); it is loaded through ctypes by
nornicdb_b200._lib and is what a cgo / JNI / N-API host would link (INTEGRATION.md)."""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libnornic_knn.so")
SOURCES = ["runtime.cu", "rowops.cu", "merge.cu", "scan_simt.cu", "scan_tensor.cu", "scan_tensor_shadow.cu", "scan_tensor_pair.cu", "assign_tensor.cu", "cluster_search.cu", "kmeanspp.cu", "exchange.cu", "legacy_abi.cu", "index_api.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O2",
    "--expt-relaxed-constexpr",
    "-ccbin", "/usr/bin/g++",
]


def _stamp() -> str:
    h = hashlib.sha256()
    for root in (CSRC, os.path.join(HERE, "..", "include")):
        for name in sorted(os.listdir(root)):
            if name.endswith((".cu", ".cuh", ".h")):
                with open(os.path.join(root, name), "rb") as f:
                    h.update(name.encode())
                    h.update(f.read())
    h.update(" ".join(FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    stamp_file = OUT + ".stamp"
    stamp = _stamp()
    if not force and os.path.exists(OUT) and os.path.exists(stamp_file):
        if open(stamp_file).read().strip() == stamp:
            return OUT
    objs = []
    procs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    for src in SOURCES:
        obj = os.path.join(HERE, "build", src.replace(".cu", ".o"))
        cmd = [NVCC, *FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            failed = True
            sys.stderr.write(f"--- nvcc {src} failed ---\n{out}\n")
        elif verbose and out:
            sys.stderr.write(f"--- nvcc {src} ---\n{out}\n")
    if failed:
        raise RuntimeError("nvcc failed building libnornic_knn.so")
    link = [NVCC, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-ccbin", "/usr/bin/g++",
            "-cudart", "static", "-o", OUT, *objs]
    subprocess.run(link, check=True)
    with open(stamp_file, "w") as f:
        f.write(stamp)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
