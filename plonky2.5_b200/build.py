"""Builds libgl_commit.so (all CUDA kernels + the C ABI) in-tree with nvcc for sm_100a only."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libgl_commit.so")
SOURCES = ["gl_commit.cu"]
HEADERS = ["gl_field.cuh", "poseidon.cuh", "poseidon_constants.cuh", "merkle.cuh", "ntt.cuh", "ntt2.cuh", "gates.cuh", "permutation.cuh", "poseidon2_constants.cuh", "fri.cuh", "microbench.cuh", "openings.cuh", "peer_sync.cuh"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared", "-cudart", "static"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


STAMP = os.path.join(HERE, ".libgl_commit.srchash")   # travels with the .so (git-ignored, not gpurun-ignored)


def source_hash() -> str:
    """sha256 over the flags and every source the library is built from: the build is skipped only when the .so on disk was built
    from exactly these bytes (mtimes mean nothing on a fresh checkout or a copied snapshot)."""
    import hashlib
    h = hashlib.sha256(" ".join(NVCC_FLAGS).encode())
    for d in [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.join(HERE, "..", "include", "gl_commit.h")]:
        h.update(open(d, "rb").read())
    return h.hexdigest()


def needs_build() -> bool:
    if not os.path.exists(LIB) or not os.path.exists(STAMP):
        return True
    return open(STAMP).read().strip() != source_hash()


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    cmd = [_nvcc(), *NVCC_FLAGS, "-o", LIB, *[os.path.join(CSRC, s) for s in SOURCES]]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
        print(" ".join(cmd), file=sys.stderr)
    env = dict(os.environ)
    env.pop("CC", None); env.pop("CXX", None)   # the image's CC wrapper is not a valid nvcc host compiler choice
    stamp = source_hash()                        # of the bytes nvcc reads: a source edited while it compiles must not look built
    subprocess.run(cmd, check=True, env=env)
    with open(STAMP, "w") as f:
        f.write(stamp)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
