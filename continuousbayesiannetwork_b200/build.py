"""Build the C-ABI shared library ``libcbn_b200.so`` in-tree with nvcc for sm_100a.

``python -m continuousbayesiannetwork_b200.build`` or ``__graft_entry__.build()``.
nvcc cross-compiles without a GPU; the resulting ``.so`` is git-ignored but travels
to the GPU box with the working tree.
"""
import hashlib
import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "libcbn_b200.so")
SOURCES = ["fit.cu", "count.cu", "ve.cu", "comm.cu", "loglik.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-shared", "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
    "--cudart", "shared",
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the cbn_b200 extension cannot be built")


def _stamp():
    h = hashlib.sha256()
    for name in sorted(os.listdir(CSRC)) + ["../../include/cbn_b200.h"]:
        with open(os.path.join(CSRC, name), "rb") as f:
            h.update(name.encode())
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build_native(force: bool = False, verbose: bool = False) -> str:
    stamp_file = LIB + ".stamp"
    stamp = _stamp()
    if not force and os.path.exists(LIB) and os.path.exists(stamp_file) and open(stamp_file).read() == stamp:
        return LIB
    cmd = [_nvcc()] + NVCC_FLAGS + os.environ.get("CBN_EXTRA_NVCC", "").split() + ["-I", os.path.join(ROOT, "include"), "-I", CSRC]
    if verbose:
        cmd += ["-Xptxas", "-v"]
    cmd += [os.path.join(CSRC, s) for s in SOURCES] + ["-ldl", "-o", LIB]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("nvcc failed building libcbn_b200.so")
    if verbose:
        sys.stderr.write(res.stderr)
    with open(stamp_file, "w") as f:
        f.write(stamp)
    return LIB


if __name__ == "__main__":
    print(build_native(force="--force" in sys.argv, verbose="-v" in sys.argv))
