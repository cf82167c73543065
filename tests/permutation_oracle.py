"""ctypes wrappers of tests/cpp/permutation_oracle.c (test infrastructure only): the permutation argument's partial products, its
vanishing terms at LDE leaf rows and the quotient tail, restated in C to check the device at prover sizes.  The library is built on
first use into a temporary directory keyed by the source's hash, so a read-only tree works."""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "permutation_oracle.c")
CFLAGS = ["-O3", "-march=x86-64-v3", "-fopenmp", "-fPIC", "-shared", "-Wall", "-Wextra", "-Werror"]


def build() -> str:
    key = hashlib.sha256(open(SRC, "rb").read() + " ".join(CFLAGS).encode()).hexdigest()[:16]
    out_dir = os.path.join(tempfile.gettempdir(), f"plonky25_permutation_oracle_{os.getuid()}_{key}")
    lib = os.path.join(out_dir, "libpermutation_oracle.so")
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
        vp, u32, u64 = ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint64
        lib.glo_partial_products.restype = ctypes.c_int
        lib.glo_partial_products.argtypes = [vp, vp, u32, u32, vp, vp, vp, u32, u32, vp]
        lib.glo_vanishing_permutation.restype = ctypes.c_int
        lib.glo_vanishing_permutation.argtypes = [vp, u32, vp, u32, u32, vp, u32, u32, u32, u32, u32, vp, vp, vp, vp, u32, vp, u64, vp]
        lib.glo_quotient_chunks.restype = ctypes.c_int
        lib.glo_quotient_chunks.argtypes = [vp, u32, u32, u32, vp]
        _lib = lib
    return _lib


def partial_products(wires, sigmas, k_is, betas, gammas, degree):
    """wires_permutation_partial_products_and_zs: wires / sigmas [n_routed][N] (any words) -> [(n_ch * n_chunks)][N], Z first"""
    w = np.ascontiguousarray(wires, dtype=np.uint64)
    s = np.ascontiguousarray(sigmas, dtype=np.uint64)
    k, b, g = (np.ascontiguousarray(a, dtype=np.uint64).reshape(-1) for a in (k_is, betas, gammas))
    n_routed, n = w.shape
    assert s.shape == w.shape and k.size == n_routed and b.size == g.size
    n_chunks = -(-n_routed // degree)
    out = np.zeros((b.size * n_chunks, n), dtype=np.uint64)
    rc = _load().glo_partial_products(w.ctypes.data, s.ctypes.data, n_routed, n.bit_length() - 1, k.ctypes.data, b.ctypes.data,
                                      g.ctypes.data, b.size, degree, out.ctypes.data)
    if rc != 0:
        raise ValueError("oracle partial_products rejected the shape")
    return out


def vanishing_permutation(wires_leaves, sigmas_leaves, sigma_col0, zs_leaves, rows, log_n, rate_bits, n_routed, degree,
                          k_is, betas, gammas, alphas):
    """the alpha-reduced permutation terms at leaf rows `rows` of rate-`rate_bits` LDE leaf matrices -> [len(rows)][n_ch]"""
    w, s, z = (np.ascontiguousarray(a, dtype=np.uint64) for a in (wires_leaves, sigmas_leaves, zs_leaves))
    k, b, g, a = (np.ascontiguousarray(x, dtype=np.uint64).reshape(-1) for x in (k_is, betas, gammas, alphas))
    r = np.ascontiguousarray(rows, dtype=np.uint64).reshape(-1)
    assert w.shape[0] == s.shape[0] == z.shape[0] == 1 << (log_n + rate_bits)
    assert w.shape[1] >= n_routed and s.shape[1] >= sigma_col0 + n_routed and k.size == n_routed
    out = np.zeros((r.size, b.size), dtype=np.uint64)
    rc = _load().glo_vanishing_permutation(w.ctypes.data, w.shape[1], s.ctypes.data, s.shape[1], sigma_col0, z.ctypes.data, z.shape[1],
                                           log_n, rate_bits, n_routed, degree, k.ctypes.data, b.ctypes.data, g.ctypes.data,
                                           a.ctypes.data, b.size, r.ctypes.data, r.size, out.ctypes.data)
    if rc != 0:
        raise ValueError("oracle vanishing_permutation rejected the shape")
    return out


def quotient_chunks(acc, log_n, rate_bits):
    """compute_quotient_polys' tail: acc [n_ch][R] in leaf order -> [(n_ch << rate_bits)][N] chunk coefficients"""
    a = np.ascontiguousarray(acc, dtype=np.uint64)
    n_ch = a.shape[0]
    assert a.shape[1] == 1 << (log_n + rate_bits)
    out = np.zeros((n_ch << rate_bits, 1 << log_n), dtype=np.uint64)
    if _load().glo_quotient_chunks(a.ctypes.data, n_ch, log_n, rate_bits, out.ctypes.data) != 0:
        raise ValueError("oracle quotient_chunks rejected the shape")
    return out
