"""Host-side OpeningSet::new for the tests and tools/opening_set_bench.py (test infrastructure only): `eval_ext` wraps
tests/cpp/eval_ext_oracle.c (OpenMP Horner in F_p^2), built on first use into a temporary directory keyed by the source's hash,
so a read-only tree works."""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "eval_ext_oracle.c")
CFLAGS = ["-O3", "-march=x86-64-v3", "-fopenmp", "-fPIC", "-shared", "-Wall", "-Wextra", "-Werror"]


def build() -> str:
    key = hashlib.sha256(open(SRC, "rb").read() + " ".join(CFLAGS).encode()).hexdigest()[:16]
    out_dir = os.path.join(tempfile.gettempdir(), f"plonky25_eval_ext_{os.getuid()}_{key}")
    lib = os.path.join(out_dir, "libeval_ext_oracle.so")
    if not os.path.exists(lib):
        os.makedirs(out_dir, exist_ok=True)
        cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"   # the image's CC wrapper lacks libgomp.spec
        tmp = lib + f".{os.getpid()}"
        subprocess.run([cc, *CFLAGS, "-o", tmp, SRC], check=True)
        os.replace(tmp, lib)
    return lib


_lib = None


def _load():
    global _lib
    if _lib is None:
        lib = ctypes.CDLL(build())
        lib.glo_eval_ext.restype = None
        lib.glo_eval_ext.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_void_p]
        lib.glo_eval_ext_threads.restype = ctypes.c_int
        _lib = lib
    return _lib


def eval_ext(polys, point) -> np.ndarray:
    """OpeningSet::new's eval_commitment on the host: polys [n_polys][N] base-field coefficients, point (a0, a1) -> [n_polys][2]"""
    f = np.ascontiguousarray(polys, dtype=np.uint64)
    if f.ndim == 1:
        f = f.reshape(1, -1)
    out = np.zeros((f.shape[0], 2), dtype=np.uint64)
    pt = np.array([int(point[0]) % (1 << 64), int(point[1]) % (1 << 64)], dtype=np.uint64)
    if f.shape[0]:
        _load().glo_eval_ext(f.ctypes.data, f.shape[0], f.shape[1], pt.ctypes.data, out.ctypes.data)
    return out


def num_threads() -> int:
    return _load().glo_eval_ext_threads()
