"""Builds libdesmo_b200.so in-tree with nvcc for sm_100a (no torch / pybind dependency: plain C ABI)."""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libdesmo_b200.so")
SOURCES = ["capi.cu", "library.cu", "fused_fp32.cu", "fused_tc.cu", "gemm_path.cu", "gram_tc.cu", "preprocess.cu", "update.cu", "eval.cu", "pod.cu", "eigh.cu", "host_api.cu", "peer.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC",
              "--expt-relaxed-constexpr", "-Xptxas", "-v"]


class NvccMissing(RuntimeError):
    pass


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise NvccMissing("nvcc not found")


def _digest() -> str:
    h = hashlib.sha256()
    for root in (CSRC, os.path.join(os.path.dirname(HERE), "include")):
        for f in sorted(os.listdir(root)):
            if f.endswith((".cu", ".cuh", ".h")):
                h.update(f.encode())
                h.update(open(os.path.join(root, f), "rb").read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    stamp = LIB + ".stamp"
    dg = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read() == dg:
        return LIB
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    procs = []
    for src in SOURCES:
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [_nvcc(), *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, obj, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    objs = []
    log = []
    for src, obj, pr in procs:
        out, _ = pr.communicate()
        log.append(f"==== {src}\n{out}")
        if pr.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{out}")
        objs.append(obj)
    with open(os.path.join(objdir, "ptxas.log"), "w") as fh:
        fh.write("\n".join(log))
    if verbose:
        print("\n".join(log))
    cmd = [_nvcc(), "-shared", "-Wno-deprecated-gpu-targets", "-o", LIB, *objs, "-lcudart"]
    subprocess.run(cmd, check=True)
    with open(stamp, "w") as fh:
        fh.write(dg)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
