"""Build libtpspp.so (sm_100a) in-tree with nvcc.  ``python -m tps_pp_b200.build [--force]``.

The library is plain CUDA C++ behind a C ABI (include/tpspp.h); it links the static CUDA
runtime only -- no torch, no pybind.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libtpspp.so")
STAMP = os.path.join(HERE, ".libtpspp.stamp")
SOURCES = ["abi.cu", "warp_fwd.cu", "warp_bwd.cu", "head.cu", "head_tc.cu", "stage.cu", "conv_train.cu", "linear_train.cu", "locnet.cu", "attn_decode.cu",
           "attn_encode.cu", "ocr_prep.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
    "--expt-relaxed-constexpr",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (set NVCC=/path/to/nvcc)")


def _sources():
    return [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def _digest() -> str:
    h = hashlib.sha256()
    files = sorted(os.listdir(CSRC)) + [os.path.join("..", "..", "include", "tpspp.h")]
    for f in files:
        path = os.path.join(CSRC, f)
        if os.path.isfile(path):
            h.update(f.encode())
            with open(path, "rb") as fh:
                h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def up_to_date() -> bool:
    if not (os.path.exists(LIB) and os.path.exists(STAMP)):
        return False
    with open(STAMP) as fh:
        return fh.read().strip() == _digest()


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and up_to_date():
        return LIB
    nvcc = _nvcc()
    objs = []
    procs = []
    builddir = os.path.join(HERE, "build")
    os.makedirs(builddir, exist_ok=True)
    for src in _sources():
        obj = os.path.join(builddir, os.path.basename(src) + ".o")
        cmd = [nvcc, *NVCC_FLAGS, "-c", src, "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for cmd, pr in procs:
        out, _ = pr.communicate()
        if verbose or pr.returncode != 0:
            sys.stderr.write(out)
        if pr.returncode != 0:
            raise RuntimeError("nvcc failed: " + " ".join(cmd))
    link = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB, *objs,
            "-cudart", "static", "-Xlinker", "--exclude-libs,ALL"]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout)
        raise RuntimeError("link failed: " + " ".join(link))
    with open(STAMP, "w") as fh:
        fh.write(_digest())
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
