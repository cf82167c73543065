"""Shared by the transform-layer GPU tests (test_ntt_plans_gpu.py, test_stage_api_gpu.py): device buffers through the library's own
gl_dev_* calls, structured input columns, and the reference coset LDE (C oracle per column, plus Python-integer evaluation) compared
with device matrices chunk by chunk, so that 2^24-point cases stay within about a gigabyte of host memory."""
import ctypes
from concurrent.futures import ThreadPoolExecutor

import numpy as np

import gl_oracle as o
from oracle_c import P, splitmix_columns

SENTINEL = 2**64 - 1          # never a canonical word: a store the kernels skipped shows up in any comparison
COSET_SHIFT = 7
CHUNK_WORDS = 1 << 24         # host staging of uploads / fills / downloads (128 MB)


def edge_words():
    """the adversarial words of the field-primitive tests: carry and wrap corners, non-canonical representatives"""
    return [0, 1, 2, 0xFFFFFFFE, 0xFFFFFFFF, 1 << 32, (1 << 32) + 1, P - 2, P - 1, P, P + 1, 2**64 - 2, 2**64 - 1, 0xFFFFFFFF << 32,
            (0xFFFFFFFF << 32) | 1, 1 << 63, (1 << 63) - 1, 0xFFFFFFFE00000001, 0xFFFFFFFE00000002, 0x00000001FFFFFFFF, 0xFFFFFF, 1 << 40]


# Column kinds.  Random data reaches the carry-save butterflies' and the folds' corners with probability ~2^-32; these reach them directly.
KINDS = ("random", "noncanonical", "const_p_minus_1", "impulse_first", "impulse_last", "alternating", "edge_words", "all_ones")


def make_column(kind, n, seed):
    if kind == "random":
        return splitmix_columns(seed, 1, n)[0]
    if kind == "noncanonical":            # every word in [p, 2^64): the same residues as words below 2^32 - 1
        return np.uint64(P) + splitmix_columns(seed, 1, n, canonical=False)[0] % np.uint64(2**64 - P)
    if kind == "const_p_minus_1":
        return np.full(n, P - 1, dtype=np.uint64)
    if kind == "impulse_first":
        c = np.zeros(n, dtype=np.uint64); c[0] = P - 1
        return c
    if kind == "impulse_last":
        c = np.zeros(n, dtype=np.uint64); c[-1] = P - 1
        return c
    if kind == "alternating":
        c = np.zeros(n, dtype=np.uint64); c[1::2] = P - 1
        return c
    if kind == "edge_words":
        e = np.array(edge_words(), dtype=np.uint64)
        return e[splitmix_columns(seed, 1, n, canonical=False)[0] % np.uint64(len(e))]
    if kind == "all_ones":
        return np.full(n, 2**64 - 1, dtype=np.uint64)
    raise ValueError(kind)


def make_columns(n_cols, n, seed, stride=None):
    """[n_cols][stride] (stride >= n words apart; the gap holds SENTINEL), column j of kind KINDS[(seed + j) % len(KINDS)]"""
    stride = n if stride is None else stride
    cols = np.full((n_cols, stride), SENTINEL, dtype=np.uint64)
    for j in range(n_cols):
        cols[j, :n] = make_column(KINDS[(seed + j) % len(KINDS)], n, seed * 131 + j)
    return cols


def canon(a):
    a = np.asarray(a, dtype=np.uint64)
    return np.where(a >= np.uint64(P), a - np.uint64(P), a)


def bitrev(idx, bits):
    idx = np.asarray(idx, dtype=np.uint64)
    r = np.zeros_like(idx)
    for b in range(bits):
        r |= ((idx >> np.uint64(b)) & np.uint64(1)) << np.uint64(bits - 1 - b)
    return r


def reference_lde(oc, cols, n, rate_bits, is_coeffs):
    """(coefficients [n_cols][N] natural order, LDE values [n_cols][N 2^rate_bits] in NATURAL point order) from the C oracle, one column
    at a time: the iFFT (unless the inputs are coefficients), then coset_fft(coefficients zero-padded to R, 7).  Leaf row i of the
    product is the value at point bitrev_R(i)."""
    R = n << rate_bits
    coeffs = np.zeros((len(cols), n), dtype=np.uint64)
    values = np.zeros((len(cols), R), dtype=np.uint64)

    def one(j):
        coeffs[j] = canon(cols[j][:n])
        if not is_coeffs:
            oc.lib.glo_ifft(coeffs[j].ctypes.data, n.bit_length() - 1)                      # in place
        values[j, :n] = coeffs[j]
        oc.lib.glo_coset_fft(values[j].ctypes.data, R.bit_length() - 1, COSET_SHIFT)      # in place (R words of scratch)

    # ctypes releases the GIL during the oracle calls; fewer threads at large R keep the oracle's scratch within a few hundred MB
    with ThreadPoolExecutor(max_workers=max(1, min(len(cols), 8, (1 << 25) // R))) as ex:
        list(ex.map(one, range(len(cols))))
    return coeffs, values


def horner(coeffs, x):
    """sum_k coeffs[k] x^k in Python integers"""
    acc = 0
    rev = np.asarray(coeffs, dtype=np.uint64)[::-1]
    for k in range(0, len(rev), 1 << 16):
        for c in rev[k:k + (1 << 16)].tolist():
            acc = (acc * x + c) % P
    return acc


def eval_points(coeffs, xs):
    """[sum_k coeffs[k] x^k for x in xs] in Python integers, vectorised over the points (the O(N * len(xs)) DFT)"""
    xs = np.array([int(x) for x in xs], dtype=object)
    acc = np.zeros(len(xs), dtype=object)
    for c in np.asarray(coeffs, dtype=np.uint64)[::-1].tolist():
        acc = (acc * xs + c) % P
    return [int(v) for v in acc]


def leaf_point(i, bits):
    """the LDE point of leaf row i: 7 * w_R^bitrev_R(i)"""
    return COSET_SHIFT * pow(o.primitive_root_of_unity(bits), o.reverse_bits(i, bits), P) % P


class DeviceBuffers:
    """device memory of one test through the library's own gl_dev_* calls; freed on exit"""

    def __init__(self, ctx):
        self.lib, self.h = ctx.lib, ctx.handle
        self._live = []

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        for p, ipc in reversed(self._live):
            (self.lib.gl_dev_ipc_free if ipc else self.lib.gl_dev_free)(self.h, p)
        self._live.clear()

    def alloc(self, words, fill=SENTINEL, ipc=False):
        """words (>= 1) of device memory; ipc: exported by gl_dev_ipc_alloc, i.e. a buffer the context knows as its own"""
        p = ctypes.c_void_p()
        if ipc:
            handle = (ctypes.c_uint8 * 64)()
            rc = self.lib.gl_dev_ipc_alloc(self.h, max(int(words), 1), ctypes.byref(p), handle)
        else:
            rc = self.lib.gl_dev_alloc(self.h, max(int(words), 1), ctypes.byref(p))
        assert rc == 0, self.lib.gl_ctx_last_error(self.h).decode()
        self._live.append((p.value, ipc))
        if fill is not None:
            self.fill(p.value, words, fill)
        return p.value

    def upload(self, ptr, arr, offset=0):
        a = np.ascontiguousarray(arr, dtype=np.uint64).reshape(-1)
        for k in range(0, a.size, CHUNK_WORDS):
            part = a[k:k + CHUNK_WORDS]
            assert self.lib.gl_dev_upload(self.h, part.ctypes.data, ptr + 8 * (offset + k), part.size) == 0

    def fill(self, ptr, words, value):
        block = np.full(min(int(words), CHUNK_WORDS), value, dtype=np.uint64)
        for k in range(0, int(words), CHUNK_WORDS):
            m = min(CHUNK_WORDS, int(words) - k)
            assert self.lib.gl_dev_upload(self.h, block.ctypes.data, ptr + 8 * k, m) == 0

    def download(self, ptr, words, offset=0):
        out = np.empty(int(words), dtype=np.uint64)
        assert self.lib.gl_dev_download(self.h, ptr + 8 * offset, out.ctypes.data, out.size) == 0
        return out

    def rows(self, ptr, row0, n_rows, pitch):
        return self.download(ptr, n_rows * pitch, row0 * pitch).reshape(n_rows, pitch)


def _first_mismatch(got, want):
    bad = np.argwhere(got != want)[0]
    return tuple(int(b) for b in bad), int(got[tuple(bad)]), int(want[tuple(bad)])


def check_leaves(bufs, ptr, pitch, col_off, values, rate_bits, what="leaves", row0=0, n_rows=None):
    """device rows [row0, row0 + n_rows) of a [..][pitch] leaf matrix, columns [col_off, col_off + n_cols), against the reference's
    natural-order values (leaf row i = point bitrev_R(i)); downloaded in chunks"""
    n_cols, R = values.shape
    bits = R.bit_length() - 1
    n_rows = R - row0 if n_rows is None else n_rows
    step = max(1, CHUNK_WORDS // max(pitch, 1))
    for a in range(0, n_rows, step):
        m = min(step, n_rows - a)
        got = bufs.rows(ptr, a, m, pitch)[:, col_off:col_off + n_cols]
        want = values[:, bitrev(np.arange(row0 + a, row0 + a + m), bits)].T
        if not np.array_equal(got, want):
            (r, c), g, w = _first_mismatch(got, want)
            raise AssertionError(f"{what}: row {row0 + a + r} column {c}: got {g:#x}, want {w:#x}")


def check_coeffs(bufs, ptr, pitch, coeffs, what="coefficients"):
    """device [N][pitch] coefficients (natural order, canonical), columns [0, n_cols), against the reference"""
    n_cols, n = coeffs.shape
    step = max(1, CHUNK_WORDS // pitch)
    for a in range(0, n, step):
        m = min(step, n - a)
        got = bufs.rows(ptr, a, m, pitch)[:, :n_cols]
        want = coeffs[:, a:a + m].T
        if not np.array_equal(got, want):
            (r, c), g, w = _first_mismatch(got, want)
            raise AssertionError(f"{what}: row {a + r} column {c}: got {g:#x}, want {w:#x}")
