"""
Compile the CUDA sources of foldingdiff_b200 into an in-tree shared library (sm_100a only).

    python -m foldingdiff_b200._build        # or __graft_entry__.build()

nvcc cross-compiles without a GPU.  The .so is git-ignored but travels with the tree to
the GPU box; nothing is JIT-compiled at import time.
"""
from __future__ import annotations

import os
import subprocess
import sys

CSRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc")
LIB_PATH = os.path.join(CSRC, "libfoldingdiff_b200.so")
SOURCES = ["api.cu"]
HEADERS = ["common.cuh", "kernels_simt.cuh", "gemm_tc.cuh", "attention_mma.cuh", "attention_pool.cuh", "attention_tc.cuh", "writers.hpp", "loss.cuh", "nerf.cuh", "philox.cuh",
           os.path.join("..", "..", "include", "foldingdiff_b200.h")]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared",
]


SHA_PATH = LIB_PATH + ".src_sha"  # hash of the sources the library was built from (travels with the .so)


def source_sha() -> str:
    import hashlib
    h = hashlib.sha256()
    for f in sorted(SOURCES + HEADERS):
        p = os.path.join(CSRC, f)
        if os.path.isfile(p):
            h.update(os.path.basename(p).encode())
            with open(p, "rb") as fh:
                h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def _stale() -> bool:
    """The library is stale when it was built from other sources than the ones in the tree: decided by content hash,
    not by mtime (a checkout or a copy to the GPU box changes mtimes arbitrarily; a stale .so must never be reused)."""
    if not os.path.isfile(LIB_PATH) or not os.path.isfile(SHA_PATH):
        return True
    with open(SHA_PATH) as f:
        return f.read().strip() != source_sha()


def build(force: bool = False, verbose: bool = True) -> str:
    if not force and not _stale():
        return LIB_PATH
    nvcc = os.environ.get("NVCC", "nvcc")
    cmd = [nvcc] + NVCC_FLAGS + [os.path.join(CSRC, s) for s in SOURCES] + ["-o", LIB_PATH, "-lz"]
    if verbose:
        print("[foldingdiff_b200] " + " ".join(cmd), file=sys.stderr)
    subprocess.run(cmd, check=True, cwd=CSRC)
    with open(SHA_PATH, "w") as f:
        f.write(source_sha() + "\n")
    return LIB_PATH


if __name__ == "__main__":
    build(force="--force" in sys.argv)
    print(LIB_PATH)
