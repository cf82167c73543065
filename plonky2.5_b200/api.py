"""Host-side mirror of the plonky2 operator interface for the commitment hot path, on top of the C ABI.

The reference's toolchain (Rust) is absent from this image, so the host layer above ``include/gl_commit.h`` is
written in Python with the SAME names, argument meaning and error behaviour as the upstream items the reference
drives from /root/reference/src/p3/mod.rs:250 (``builder.build``) and :260 (``data.prove``):

    plonky2 fri/oracle.rs        PolynomialBatch::from_values / from_coeffs / get_lde_values
    plonky2 hash/merkle_tree.rs  MerkleTree::new / get / prove,  MerkleCap
    plonky2 fri/prover.rs        fri_committed_trees
    plonky2 iop/challenger.rs    Challenger (observe_* / get_challenge / get_extension_challenge)

Upstream ``assert!`` panics become ``ValueError`` (GL_ERR_INVALID) here.  Field elements are ``numpy.uint64``;
outputs are canonical.  All compute happens in libgl_commit.so on the GPU — there is no CPU path in this module.
"""
from __future__ import annotations

import ctypes
from ctypes import byref, c_uint64, c_void_p
from typing import List, Optional, Sequence, Tuple

import numpy as np

from . import _lib

P = 0xFFFF_FFFF_0000_0001
SPONGE_RATE = 8
SPONGE_WIDTH = 12


class GlError(RuntimeError):
    pass


def _check(ctx: "Context", rc: int):
    if rc == _lib.GL_OK:
        return
    msg = ctx.lib.gl_ctx_last_error(ctx.handle).decode() if ctx.handle else ""
    text = f"{ctx.lib.gl_strerror(rc).decode()}: {msg}"
    if rc == _lib.GL_ERR_INVALID:
        raise ValueError(text)
    if rc == _lib.GL_ERR_OOM:
        raise MemoryError(text)
    raise GlError(text)


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(c_void_p)


class Context:
    """One CUDA device + stream + cached twiddle tables (gl_ctx)."""

    def __init__(self, device: int = 0):
        self.lib = _lib.load()
        self.handle = c_void_p()
        rc = self.lib.gl_ctx_create(byref(self.handle), device)
        if rc != _lib.GL_OK:
            self.handle = None
            raise GlError(f"gl_ctx_create(device={device}) failed: {self.lib.gl_strerror(rc).decode()} "
                          "(libgl_commit has no CPU fallback; a CUDA device is required)")
        self.device = device

    def close(self):
        if self.handle:
            self.lib.gl_ctx_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def stream(self) -> int:
        return int(self.lib.gl_ctx_stream(self.handle))

    def stage_times(self) -> Tuple[dict, dict]:
        ms = (ctypes.c_float * len(_lib.STAGES))()
        ln = (ctypes.c_uint32 * len(_lib.STAGES))()
        _check(self, self.lib.gl_ctx_stage_times(self.handle, ms, ln))
        return dict(zip(_lib.STAGES, map(float, ms))), dict(zip(_lib.STAGES, map(int, ln)))

    def microbench(self, which: int, iters: int = 2000) -> float:
        out = ctypes.c_double()
        _check(self, self.lib.gl_microbench(self.handle, which, iters, byref(out)))
        return out.value

    def field_op(self, op: int, a: np.ndarray, b: Optional[np.ndarray] = None) -> np.ndarray:
        """Element-wise field primitive exactly as the kernels use it (include/gl_commit.h · GL_FOP_*)."""
        a = np.ascontiguousarray(a, dtype=np.uint64).reshape(-1)
        b = a if b is None else np.ascontiguousarray(b, dtype=np.uint64).reshape(-1)
        out = np.zeros_like(a)
        _check(self, self.lib.gl_field_op(self.handle, op, _ptr(a), _ptr(b), _ptr(out), a.size))
        return out

    def poseidon_permute(self, states: np.ndarray) -> np.ndarray:
        s = np.ascontiguousarray(states, dtype=np.uint64).reshape(-1, SPONGE_WIDTH).copy()
        _check(self, self.lib.gl_poseidon_permute(self.handle, _ptr(s), s.shape[0]))
        return s


_default_ctx: Optional[Context] = None


def default_context() -> Context:
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context(0)
    return _default_ctx


class MerkleCap:
    def __init__(self, hashes: np.ndarray):
        self.hashes = hashes.reshape(-1, 4)

    def height(self) -> int:
        return int(self.hashes.shape[0]).bit_length() - 1

    def flatten(self) -> np.ndarray:
        return self.hashes.reshape(-1)

    def __len__(self):
        return self.hashes.shape[0]


class MerkleTree:
    """plonky2 hash/merkle_tree.rs · MerkleTree { leaves, digests, cap } — device resident, host views on demand."""

    def __init__(self, ctx: Context, handle: int, cap: np.ndarray, leaves=None, digests=None):
        self.ctx = ctx
        self._h = handle
        self.cap = MerkleCap(cap)
        info = _lib.TreeInfo()
        _check(ctx, ctx.lib.gl_tree_info(ctx.handle, handle, byref(info)))
        self.n_leaves, self.leaf_len, self.cap_height = int(info.n_leaves), int(info.leaf_len), int(info.cap_height)
        self.degree_log, self.rate_bits = int(info.degree_log), int(info.rate_bits)
        self._leaves, self._digests = leaves, digests

    @classmethod
    def new(cls, leaves, cap_height: int, ctx: Optional[Context] = None, copy_back: bool = False) -> "MerkleTree":
        ctx = ctx or default_context()
        lv = np.ascontiguousarray(leaves, dtype=np.uint64)
        if lv.ndim != 2:
            raise ValueError("leaves must be a 2-D array [n_leaves][leaf_len]")
        n, ll = lv.shape
        if n == 0 or cap_height > n.bit_length() - 1:   # upstream's assert, checked BEFORE sizing the cap buffer by 2^cap_height
            raise ValueError(f"cap_height={cap_height} should be at most log2(leaves.len())={max(n.bit_length() - 1, 0)}")
        cap = np.zeros(4 << cap_height, dtype=np.uint64)
        dig = None
        if copy_back and n >= (1 << cap_height):
            dig = np.zeros((2 * (n - (1 << cap_height)), 4), dtype=np.uint64)
        h = c_uint64()
        _check(ctx, ctx.lib.gl_merkle_new(ctx.handle, _ptr(lv), n, ll, cap_height, _ptr(dig), _ptr(cap), byref(h)))
        return cls(ctx, h.value, cap, leaves=lv if copy_back else None, digests=dig)

    @property
    def leaves(self) -> np.ndarray:
        if self._leaves is None:
            out = np.zeros((self.n_leaves, self.leaf_len), dtype=np.uint64)
            _check(self.ctx, self.ctx.lib.gl_tree_read(self.ctx.handle, self._h, _lib.GL_PART_LEAVES, _ptr(out)))
            self._leaves = out
        return self._leaves

    @property
    def digests(self) -> np.ndarray:
        if self._digests is None:
            out = np.zeros((2 * (self.n_leaves - (1 << self.cap_height)), 4), dtype=np.uint64)
            _check(self.ctx, self.ctx.lib.gl_tree_read(self.ctx.handle, self._h, _lib.GL_PART_DIGESTS, _ptr(out)))
            self._digests = out
        return self._digests

    def get(self, i: int) -> np.ndarray:
        out = np.zeros(self.leaf_len, dtype=np.uint64)
        _check(self.ctx, self.ctx.lib.gl_tree_get(self.ctx.handle, self._h, i, _ptr(out)))
        return out

    def prove(self, leaf_index: int) -> np.ndarray:
        """MerkleProof::siblings, bottom-up, shape [log2(n_leaves) - cap_height][4]."""
        depth = self.n_leaves.bit_length() - 1 - self.cap_height
        out = np.zeros((depth, 4), dtype=np.uint64)
        _check(self.ctx, self.ctx.lib.gl_tree_prove(self.ctx.handle, self._h, leaf_index, _ptr(out)))
        return out

    def open_batch(self, indices) -> Tuple[np.ndarray, np.ndarray]:
        """(get(i), prove(i)) for every i of `indices` in one device round trip: ([n][leaf_len], [n][depth][4])."""
        idx = np.ascontiguousarray(indices, dtype=np.uint64).reshape(-1)
        depth = self.n_leaves.bit_length() - 1 - self.cap_height
        rows = np.zeros((idx.size, self.leaf_len), dtype=np.uint64)
        sib = np.zeros((idx.size, depth, 4), dtype=np.uint64)
        _check(self.ctx, self.ctx.lib.gl_tree_open_batch(self.ctx.handle, self._h, _ptr(idx) if idx.size else None, idx.size,
                                                         _ptr(rows), _ptr(sib)))
        return rows, sib

    def free(self):
        if self._h and self.ctx.handle:
            self.ctx.lib.gl_tree_free(self.ctx.handle, self._h)
        self._h = 0

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class PolynomialBatch:
    """plonky2 fri/oracle.rs · PolynomialBatch { polynomials, merkle_tree, degree_log, rate_bits, blinding }."""

    def __init__(self, ctx, tree: MerkleTree, n_cols: int, polynomials=None):
        self.ctx = ctx
        self.merkle_tree = tree
        self.degree_log = tree.degree_log
        self.rate_bits = tree.rate_bits
        self.blinding = False
        self._n_cols = n_cols
        self._polys = polynomials

    @staticmethod
    def _cols(values) -> Tuple[List[np.ndarray], int]:
        cols = [np.ascontiguousarray(v, dtype=np.uint64) for v in values]
        if not cols:
            raise ValueError("empty polynomial batch")
        n = cols[0].shape[0]
        if any(c.ndim != 1 or c.shape[0] != n for c in cols):
            raise ValueError("Polynomial degrees inconsistent")
        if n == 0 or n & (n - 1):
            raise ValueError("polynomial length must be a power of two")
        return cols, n.bit_length() - 1

    @classmethod
    def _commit(cls, values, rate_bits, blinding, cap_height, is_coeffs, ctx, copy_back):
        if blinding:
            raise ValueError("blinding (zero_knowledge) is not on the GPU path: the reference runs with zk off "
                             "(/root/reference/src/p3/mod.rs:231)")
        ctx = ctx or default_context()
        cols, log_n = cls._cols(values)
        n_cols, n = len(cols), 1 << log_n
        rows = n << rate_bits
        ptrs = (c_void_p * n_cols)(*[c.ctypes.data for c in cols])
        if cap_height > log_n + rate_bits:               # upstream's assert, checked BEFORE sizing the cap buffer by 2^cap_height
            raise ValueError(f"cap_height={cap_height} should be at most log2(leaves.len())={log_n + rate_bits}")
        cap = np.zeros(4 << cap_height, dtype=np.uint64)
        oc = ol = od = None
        if copy_back:
            oc = np.zeros((n_cols, n), dtype=np.uint64)
            ol = np.zeros((rows, n_cols), dtype=np.uint64)
            od = np.zeros((max(2 * (rows - (1 << cap_height)), 0), 4), dtype=np.uint64)
        h = c_uint64()
        _check(ctx, ctx.lib.gl_commit(ctx.handle, ptrs, n_cols, log_n, rate_bits, cap_height, int(is_coeffs),
                                      _ptr(oc), _ptr(ol), _ptr(od), _ptr(cap), byref(h)))
        tree = MerkleTree(ctx, h.value, cap, leaves=ol, digests=od)
        return cls(ctx, tree, n_cols, polynomials=oc)

    @classmethod
    def from_values(cls, values, rate_bits: int, blinding: bool, cap_height: int, timing=None, fft_root_table=None,
                    ctx: Optional[Context] = None, copy_back: bool = False) -> "PolynomialBatch":
        """values: Vec<PolynomialValues<F>> — sequence of equal-length 1-D uint64 arrays (one per column)."""
        return cls._commit(values, rate_bits, blinding, cap_height, False, ctx, copy_back)

    @classmethod
    def from_coeffs(cls, polynomials, rate_bits: int, blinding: bool, cap_height: int, timing=None, fft_root_table=None,
                    ctx: Optional[Context] = None, copy_back: bool = False) -> "PolynomialBatch":
        return cls._commit(polynomials, rate_bits, blinding, cap_height, True, ctx, copy_back)

    @property
    def polynomials(self) -> np.ndarray:
        """[n_cols][N] canonical coefficients."""
        if self._polys is None:
            out = np.zeros((self._n_cols, 1 << self.degree_log), dtype=np.uint64)
            t = self.merkle_tree
            _check(self.ctx, self.ctx.lib.gl_tree_read(self.ctx.handle, t._h, _lib.GL_PART_COEFFS, _ptr(out)))
            self._polys = out
        return self._polys

    def get_lde_values(self, index: int, step: int) -> np.ndarray:
        t = self.merkle_tree
        out = np.zeros(t.leaf_len, dtype=np.uint64)
        _check(self.ctx, self.ctx.lib.gl_tree_get_lde_values(self.ctx.handle, t._h, index, step, _ptr(out)))
        return out


def commit_multi(ctxs: Sequence[Context], values, rate_bits: int, cap_height: int, is_coeffs: bool = False) -> Tuple[MerkleCap, List[MerkleTree]]:
    """PolynomialBatch::from_values / from_coeffs on several GPUs from one process (gl_commit_multi): one Context per device, columns
    sharded for the LDE, leaf ranges hashed per context.  Returns (cap, shard trees); leaf row i of the batch lives in
    trees[i // (R // len(ctxs))] at local index i % (R // len(ctxs)), and `.prove` there is MerkleTree::prove(i)."""
    cols, log_n = PolynomialBatch._cols(values)
    if cap_height > log_n + rate_bits:
        raise ValueError(f"cap_height={cap_height} should be at most log2(leaves.len())={log_n + rate_bits}")
    lib = ctxs[0].lib
    hs = (c_void_p * len(ctxs))(*[c.handle for c in ctxs])
    ptrs = (c_void_p * len(cols))(*[c.ctypes.data for c in cols])
    cap = np.zeros(4 << cap_height, dtype=np.uint64)
    trees = (c_uint64 * len(ctxs))()
    _check(ctxs[0], lib.gl_commit_multi(hs, len(ctxs), ptrs, len(cols), log_n, rate_bits, cap_height, int(is_coeffs), _ptr(cap), trees))
    per = (4 << cap_height) // len(ctxs)
    return MerkleCap(cap), [MerkleTree(c, int(t), cap[g * per:(g + 1) * per].copy()) for g, (c, t) in enumerate(zip(ctxs, trees))]


class Challenger:
    """plonky2 iop/challenger.rs · Challenger<F, PoseidonHash>: duplex sponge; the permutation runs on the GPU."""

    def __init__(self, ctx: Optional[Context] = None):
        self.ctx = ctx or default_context()
        self.sponge_state = np.zeros(SPONGE_WIDTH, dtype=np.uint64)
        self.input_buffer: List[int] = []
        self.output_buffer: List[int] = []

    def observe_element(self, e: int):
        self.output_buffer = []
        self.input_buffer.append(int(e) % P)
        if len(self.input_buffer) == SPONGE_RATE:
            self._duplexing()

    def observe_elements(self, es):
        """observe_element for every element — with the duplexing of all FULL groups of 8 done in one device call (gl_poseidon_absorb):
        the chain of permutations is sequential anyway, so a Merkle cap costs one launch and one round trip instead of eight"""
        vals = [int(e) % P for e in np.asarray(es, dtype=np.uint64).reshape(-1).tolist()]
        if not vals:
            return
        self.output_buffer = []
        buf = self.input_buffer + vals
        n_full = len(buf) // SPONGE_RATE
        if n_full:
            groups = np.array(buf[:n_full * SPONGE_RATE], dtype=np.uint64)
            st = np.ascontiguousarray(self.sponge_state, dtype=np.uint64)
            _check(self.ctx, self.ctx.lib.gl_poseidon_absorb(self.ctx.handle, _ptr(st), _ptr(groups), n_full))
            self.sponge_state = st
            self.output_buffer = [int(x) for x in st[:SPONGE_RATE]]
        self.input_buffer = buf[n_full * SPONGE_RATE:]
        if self.input_buffer:
            self.output_buffer = []       # an element observed after the last duplexing invalidates the buffered outputs

    def observe_hash(self, h):
        self.observe_elements(h)

    def observe_cap(self, cap):
        self.observe_elements(cap.flatten() if isinstance(cap, MerkleCap) else cap)

    def observe_extension_element(self, e):
        self.observe_elements(e)

    def observe_extension_elements(self, es):
        self.observe_elements(es)

    def observe_openings(self, fri_openings: "FriOpenings"):
        """every batch's values, in order, as extension elements (upstream: observe_openings(&openings.to_fri_openings()))"""
        for batch in fri_openings.batches:
            self.observe_extension_elements(batch.values)

    def get_challenge(self) -> int:
        if self.input_buffer or not self.output_buffer:
            self._duplexing()
        return self.output_buffer.pop()

    def get_extension_challenge(self) -> Tuple[int, int]:
        c0 = self.get_challenge()
        c1 = self.get_challenge()
        return (c0, c1)

    def _duplexing(self):
        for i, v in enumerate(self.input_buffer):
            self.sponge_state[i] = v
        self.input_buffer = []
        self.sponge_state = self.ctx.poseidon_permute(self.sponge_state)[0]
        self.output_buffer = [int(x) for x in self.sponge_state[:SPONGE_RATE]]


def fri_proof_of_work(challenger: Challenger, min_leading_zeros: int, ctx: Optional[Context] = None) -> int:
    """plonky2 fri/prover.rs · fri_proof_of_work: grind on the GPU for the smallest witness, then advance the transcript
    exactly as upstream (observe the witness, draw the response and check its leading zeros)."""
    ctx = ctx or challenger.ctx
    st = np.ascontiguousarray(challenger.sponge_state, dtype=np.uint64)
    buf = np.array(challenger.input_buffer, dtype=np.uint64)
    w = c_uint64()
    _check(ctx, ctx.lib.gl_fri_pow(ctx.handle, _ptr(st), _ptr(buf) if buf.size else None, buf.size, min_leading_zeros, byref(w)))
    challenger.observe_element(w.value)
    resp = challenger.get_challenge()
    if 64 - int(resp).bit_length() < min_leading_zeros:
        raise GlError("proof-of-work response does not have the required leading zeros")
    return w.value


class FriParams:
    """The fields of plonky2 fri/mod.rs · FriParams that fri_committed_trees reads."""

    def __init__(self, rate_bits: int, cap_height: int, reduction_arity_bits: Sequence[int]):
        self.rate_bits = rate_bits
        self.cap_height = cap_height
        self.reduction_arity_bits = list(reduction_arity_bits)


def reduction_arity_bits(degree_bits: int, rate_bits: int, cap_height: int, arity_bits: int = 4, final_poly_bits: int = 5) -> List[int]:
    """plonky2 fri/reduction_strategies.rs · FriReductionStrategy::ConstantArityBits(arity_bits, final_poly_bits).reduction_arity_bits
    (standard_recursion_config uses (4, 5): the wrapper circuit, degree_bits 16, folds 4, 4, 4 down to 16 coefficients)."""
    out = []
    while degree_bits > final_poly_bits and degree_bits + rate_bits - arity_bits >= cap_height:
        out.append(arity_bits)
        if degree_bits < arity_bits:
            raise ValueError("assertion failed: degree_bits >= *arity_bits")
        degree_bits -= arity_bits
    return out


def _fri_commit_phase(ctx: Context, fh: int, challenger, fri_params: FriParams):
    """the per-layer loop of fri_committed_trees on a device-resident FRI state (gl_fri handle)"""
    lib = ctx.lib
    trees = []
    cur = c_uint64()
    _check(ctx, lib.gl_fri_read(ctx.handle, fh, None, None, byref(cur)))
    cur = int(cur.value)
    for arity_bits in fri_params.reduction_arity_bits:
        cur >>= arity_bits                      # leaves of this layer; MerkleTree::new's assert before the cap is sized
        if fri_params.cap_height > (cur.bit_length() - 1 if cur else 31):   # cur == 0: the library reports "arity larger than the codeword"
            raise ValueError(f"cap_height={fri_params.cap_height} should be at most log2(leaves.len())={max(cur.bit_length() - 1, 0)}")
        cap = np.zeros(4 << fri_params.cap_height, dtype=np.uint64)
        th = c_uint64()
        _check(ctx, lib.gl_fri_commit_layer(ctx.handle, fh, arity_bits, None, None, _ptr(cap), byref(th)))
        tree = MerkleTree(ctx, th.value, cap)
        challenger.observe_cap(tree.cap.flatten())
        trees.append(tree)
        beta = challenger.get_extension_challenge()
        b = np.array([int(beta[0]), int(beta[1])], dtype=np.uint64)
        _check(ctx, lib.gl_fri_fold(ctx.handle, fh, _ptr(b)))
    n = c_uint64()
    _check(ctx, lib.gl_fri_final_poly(ctx.handle, fh, None, byref(n)))
    final = np.zeros((n.value, 2), dtype=np.uint64)
    _check(ctx, lib.gl_fri_final_poly(ctx.handle, fh, _ptr(final), byref(n)))
    challenger.observe_extension_elements(final)
    return trees, final


def fri_committed_trees(polynomial_coeffs, polynomial_values, challenger, fri_params: FriParams,
                        ctx: Optional[Context] = None):
    """plonky2 fri/prover.rs · fri_committed_trees.

    polynomial_coeffs / polynomial_values: [len][2] extension elements (values = coset_fft(coeffs, 7), natural order).
    `challenger` is the caller's Fiat–Shamir transcript (any object with observe_cap / get_extension_challenge /
    observe_extension_elements).  Returns (trees, final_poly_coeffs[len_final][2]).
    """
    ctx = ctx or default_context()
    co = np.ascontiguousarray(polynomial_coeffs, dtype=np.uint64).reshape(-1, 2)
    va = np.ascontiguousarray(polynomial_values, dtype=np.uint64).reshape(-1, 2)
    if co.shape != va.shape:
        raise ValueError("coeffs and values must have the same length")
    fh = c_uint64()
    _check(ctx, ctx.lib.gl_fri_begin(ctx.handle, _ptr(co), _ptr(va), co.shape[0], fri_params.rate_bits, fri_params.cap_height,
                                     byref(fh)))
    try:
        return _fri_commit_phase(ctx, fh.value, challenger, fri_params)
    finally:
        ctx.lib.gl_fri_end(ctx.handle, fh.value)


class FriBatchInfo:
    """plonky2 fri/structure.rs · FriBatchInfo { point, polynomials: Vec<FriPolynomialInfo { oracle_index, polynomial_index }> }"""

    def __init__(self, point: Tuple[int, int], polynomials: Sequence[Tuple[int, int]]):
        self.point = (int(point[0]), int(point[1]))
        self.polynomials = [(int(o), int(i)) for (o, i) in polynomials]


def eval_commitment(batch: "PolynomialBatch", points) -> np.ndarray:
    """OpeningSet::new's eval_commitment closure: every polynomial of `batch` at each of 1 or 2 extension points (a0, a1), on the
    device (gl_batch_eval); the coefficients stay in HBM.  Returns [n_points][num_polys][2] canonical words."""
    pts = np.array([[int(p[0]), int(p[1])] for p in points], dtype=np.uint64)
    t = batch.merkle_tree
    out = np.zeros((len(pts), t.leaf_len, 2), dtype=np.uint64)
    _check(batch.ctx, batch.ctx.lib.gl_batch_eval(batch.ctx.handle, t._h, _ptr(pts) if pts.size else None, len(pts), _ptr(out)))
    return out


class FriOpeningBatch:
    """plonky2 fri/structure.rs · FriOpeningBatch { values: Vec<F::Extension> } — [n][2] words"""

    def __init__(self, values):
        self.values = np.ascontiguousarray(values, dtype=np.uint64).reshape(-1, 2)


class FriOpenings:
    """plonky2 fri/structure.rs · FriOpenings { batches: Vec<FriOpeningBatch> }"""

    def __init__(self, batches: Sequence[FriOpeningBatch]):
        self.batches = list(batches)


class OpeningSet:
    """plonky2 plonk/proof.rs · OpeningSet without lookups (the reference's circuits use none); every field is [n][2] words."""

    def __init__(self, constants, plonk_sigmas, wires, plonk_zs, plonk_zs_next, partial_products, quotient_polys):
        self.constants, self.plonk_sigmas, self.wires = constants, plonk_sigmas, wires
        self.plonk_zs, self.plonk_zs_next, self.partial_products = plonk_zs, plonk_zs_next, partial_products
        self.quotient_polys = quotient_polys

    @classmethod
    def new(cls, zeta, g, constants_sigmas: "PolynomialBatch", wires: "PolynomialBatch", zs_partial_products: "PolynomialBatch",
            quotient: "PolynomialBatch", num_constants: int, num_challenges: int) -> "OpeningSet":
        """OpeningSet::new: the four commits at zeta, the Z/partial-products commit also at g * zeta (one device call for both points).
        Commit #0 holds the constants first, then the sigmas; commit #2 the Z polynomial of every challenge first (gl_partial_products'
        order), then the partial products.  g: the subgroup generator, a base element or an extension element (a0, a1)."""
        z = (int(zeta[0]) % P, int(zeta[1]) % P)
        g0, g1 = (int(g), 0) if np.isscalar(g) else (int(g[0]), int(g[1]))
        gz = ((g0 * z[0] + 7 * g1 * z[1]) % P, (g0 * z[1] + g1 * z[0]) % P)
        if num_constants > constants_sigmas.merkle_tree.leaf_len or num_challenges > zs_partial_products.merkle_tree.leaf_len:
            raise ValueError("num_constants / num_challenges exceed the width of their commit")
        cs = eval_commitment(constants_sigmas, [z])[0]
        zs = eval_commitment(zs_partial_products, [z, gz])
        return cls(constants=cs[:num_constants], plonk_sigmas=cs[num_constants:], wires=eval_commitment(wires, [z])[0],
                   plonk_zs=zs[0][:num_challenges], plonk_zs_next=zs[1][:num_challenges], partial_products=zs[0][num_challenges:],
                   quotient_polys=eval_commitment(quotient, [z])[0])

    def to_fri_openings(self) -> FriOpenings:
        """the zeta batch (constants, sigmas, wires, zs, partial products, quotient) and the g * zeta batch (zs_next)"""
        zeta_batch = np.concatenate([self.constants, self.plonk_sigmas, self.wires, self.plonk_zs, self.partial_products,
                                     self.quotient_polys])
        return FriOpenings([FriOpeningBatch(zeta_batch), FriOpeningBatch(self.plonk_zs_next)])


class FriProofHead:
    """What prove_openings produces before the query rounds: FriProof { commit_phase_merkle_caps, final_poly, pow_witness };
    `trees` are the commit-phase MerkleTrees the query rounds read with .get/.prove."""

    def __init__(self, trees, final_poly, pow_witness, lde_final_len):
        self.trees = trees
        self.commit_phase_merkle_caps = [t.cap for t in trees]
        self.final_poly = final_poly
        self.pow_witness = pow_witness
        self.lde_final_len = lde_final_len


def prove_openings(instance: Sequence[FriBatchInfo], oracles: Sequence["PolynomialBatch"], challenger, fri_params: FriParams,
                   proof_of_work_bits: Optional[int] = None, ctx: Optional[Context] = None, debug: Optional[dict] = None) -> FriProofHead:
    """plonky2 fri/oracle.rs · PolynomialBatch::prove_openings up to (not including) the query rounds, on the device:
    alpha <- challenger; per batch reduce_polys_base + divide_by_linear + shift_poly; final_poly.lde(rate_bits).coset_fft(7);
    fri_committed_trees; fri_proof_of_work (if proof_of_work_bits is given).  The coefficient matrices of `oracles` never
    leave HBM.  `debug` (a dict) receives final_poly / quotients / lde arrays for tests."""
    ctx = ctx or default_context()
    lib = ctx.lib
    if not oracles:
        raise ValueError("no oracles")
    log_n = oracles[0].degree_log
    alpha = challenger.get_extension_challenge()
    al = np.array([int(alpha[0]), int(alpha[1])], dtype=np.uint64)
    oh = c_uint64()
    _check(ctx, lib.gl_openings_begin(ctx.handle, log_n, byref(oh)))
    fh = c_uint64()
    try:
        for batch in instance:
            hs = np.array([oracles[o].merkle_tree._h for (o, _) in batch.polynomials], dtype=np.uint64)
            cs = np.array([i for (_, i) in batch.polynomials], dtype=np.uint32)
            pt = np.array(batch.point, dtype=np.uint64)
            q = np.zeros((1 << log_n, 2), dtype=np.uint64) if debug is not None else None
            _check(ctx, lib.gl_openings_add_batch(ctx.handle, oh.value, _ptr(hs) if hs.size else None, _ptr(cs) if cs.size else None,
                                                  hs.size, _ptr(al), _ptr(pt), _ptr(q)))
            if debug is not None:
                debug.setdefault("quotients", []).append(q)
        if debug is not None:
            fp = np.zeros((1 << log_n, 2), dtype=np.uint64)
            _check(ctx, lib.gl_openings_final_poly(ctx.handle, oh.value, _ptr(fp)))
            debug["final_poly"] = fp
        _check(ctx, lib.gl_openings_lde(ctx.handle, oh.value, fri_params.rate_bits, fri_params.cap_height, byref(fh)))
    finally:
        lib.gl_openings_end(ctx.handle, oh.value)
    try:
        n = c_uint64()
        _check(ctx, lib.gl_fri_read(ctx.handle, fh.value, None, None, byref(n)))
        if debug is not None:
            co = np.zeros((n.value, 2), dtype=np.uint64)
            va = np.zeros((n.value, 2), dtype=np.uint64)
            _check(ctx, lib.gl_fri_read(ctx.handle, fh.value, _ptr(co), _ptr(va), byref(n)))
            debug["lde_final_poly"], debug["lde_final_values_bitrev"] = co, va
        trees, final = _fri_commit_phase(ctx, fh.value, challenger, fri_params)
    finally:
        lib.gl_fri_end(ctx.handle, fh.value)
    w = fri_proof_of_work(challenger, proof_of_work_bits, ctx) if proof_of_work_bits is not None else None
    return FriProofHead(trees, final, w, int(n.value))


def fri_prover_query_rounds(initial_merkle_trees: Sequence[MerkleTree], trees: Sequence[MerkleTree], challenger, n_query_rounds: int,
                            fri_params: FriParams, lde_size: Optional[int] = None) -> List[dict]:
    """plonky2 fri/prover.rs · fri_prover_query_rounds / fri_prover_query_round: per round x_index = challenge mod lde_size;
    initial_trees_proof = [(tree.get(x), tree.prove(x))] for every initial oracle; per commit-phase layer the coset evaluations
    (the whole leaf x >> arity_bits = `arity` extension elements, as upstream's FriQueryStep holds them) and its Merkle proof.  All indices of a tree are
    opened in one gl_tree_open_batch call.  Returns one dict per round:
    {"x_index", "initial_trees_proof": [(row, siblings)], "steps": [{"evals": [arity][2], "merkle_proof": siblings}]}."""
    n = int(lde_size if lde_size is not None else initial_merkle_trees[0].n_leaves)
    xs = [int(challenger.get_challenge()) % n for _ in range(n_query_rounds)]
    init = [t.open_batch(xs) for t in initial_merkle_trees]
    steps = []
    cur = list(xs)
    for arity_bits, t in zip(fri_params.reduction_arity_bits, trees):
        rows, sib = t.open_batch([x >> arity_bits for x in cur])
        steps.append((arity_bits, rows, sib, list(cur)))
        cur = [x >> arity_bits for x in cur]
    out = []
    for q, x in enumerate(xs):
        rnd = {"x_index": x, "initial_trees_proof": [(rows[q], sib[q]) for rows, sib in init], "steps": []}
        for arity_bits, rows, sib, idx in steps:
            # evals = unflatten(tree.get(x_index >> arity_bits)): all `arity` elements of the coset (only FriProof::compress drops
            # the queried one; the verifier reads evals[x_index & (arity - 1)] and Merkle-verifies flatten(evals))
            rnd["steps"].append({"evals": rows[q].reshape(-1, 2).copy(), "merkle_proof": sib[q]})
        out.append(rnd)
    return out


# ---- SURVEY §8(f) ranks 3-4: gate constraints over the resident LDE rows, partial products / Z, witness rows -------------------------
GATE_POSEIDON2, GATE_U32_ARITHMETIC, GATE_U32_ADD_MANY, GATE_U32_SUBTRACTION, GATE_U32_RANGE_CHECK = 0, 1, 2, 3, 4
GATE_U32_INTERLEAVE, GATE_UNINTERLEAVE_TO_U32, GATE_UNINTERLEAVE_TO_B32, GATE_COMPARISON = 5, 6, 7, 8
# plonky2's core gates: NoopGate, ConstantGate { num_consts }, PublicInputGate, ArithmeticGate { num_ops }, BaseSumGate<B> (num_limbs | B << 8)
GATE_NOOP, GATE_CONSTANT, GATE_PUBLIC_INPUT, GATE_ARITHMETIC, GATE_BASE_SUM = 9, 10, 11, 12, 13
# PoseidonGate (param 0), ExponentiationGate { num_power_bits }, RandomAccessGate (bits | num_copies << 8 | num_extra_constants << 16)
GATE_POSEIDON, GATE_EXPONENTIATION, GATE_RANDOM_ACCESS = 15, 16, 17


def random_access_params(bits: int, num_wires: int = 135, num_routed: int = 80, num_constants: int = 2) -> int:
    """plonky2 gates/random_access.rs · RandomAccessGate::new_from_config as a GATE_RANDOM_ACCESS param: as many copies as the routed
    and total wires allow, and the routed wires left over (at most num_constants) as extra constants"""
    v = 1 << bits
    copies = min(num_routed // (2 + v), num_wires // (2 + v + bits))
    extras = min(num_routed - (2 + v) * copies, num_constants)
    return bits | copies << 8 | extras << 16


def gate_shape(kind: int, param: int = 0) -> Tuple[int, int]:
    """(num_wires, num_constraints) of a gate (Gate::num_wires / num_constraints); ValueError for an unknown kind or parameter"""
    lib = _lib.load()
    nw, nc = lib.gl_gate_num_wires(kind, param), lib.gl_gate_num_constraints(kind, param)
    if nw < 0 or nc < 0:
        raise ValueError(f"unknown gate kind {kind} / parameter {param}")
    return nw, nc


def evaluate_gate_constraints(kind: int, param: int, rows, ctx: Optional[Context] = None, constants=None,
                              public_inputs_hash=None) -> np.ndarray:
    """Gate::eval_unfiltered_base_batch for host rows [n][num_wires]: every constraint value, uncombined ([n][num_constraints]).
    Gates that read gate constants or the public-inputs hash (GATE_CONSTANT, GATE_ARITHMETIC, GATE_PUBLIC_INPUT) take `constants`
    ([n][num_constants], the row's local constants after the selectors) and `public_inputs_hash` (4 words)."""
    ctx = ctx or default_context()
    nw, nc = gate_shape(kind, param)
    r = np.ascontiguousarray(rows, dtype=np.uint64)
    if r.ndim != 2 or r.shape[1] != nw:
        raise ValueError(f"rows must be [n][{nw}]")
    out = np.zeros((r.shape[0], nc), dtype=np.uint64)
    if constants is None and public_inputs_hash is None:
        _check(ctx, ctx.lib.gl_gate_eval_rows(ctx.handle, kind, param, _ptr(r), r.shape[0], _ptr(out)))
        return out
    nk = ctx.lib.gl_gate_num_constants(kind, param)
    k = np.ascontiguousarray(np.zeros((r.shape[0], 0)) if constants is None else constants, dtype=np.uint64)
    if k.shape != (r.shape[0], nk):
        raise ValueError(f"constants must be [n][{nk}]")
    pi = np.ascontiguousarray(np.zeros(4) if public_inputs_hash is None else public_inputs_hash, dtype=np.uint64).reshape(-1)
    if pi.size != 4:
        raise ValueError("public_inputs_hash must be 4 words")
    _check(ctx, ctx.lib.gl_gate_eval_rows_with_constants(ctx.handle, kind, param, _ptr(r), _ptr(k) if nk else None, _ptr(pi), r.shape[0],
                                                         _ptr(out)))
    return out


class SelectorsInfo:
    """plonky2 gates/selectors.rs · SelectorsInfo { selector_indices, groups }: gate i is filtered by selector column
    selector_indices[i], whose group is the gate range groups[selector_indices[i]] = (start, end)."""

    def __init__(self, selector_indices: Sequence[int], groups: Sequence[Tuple[int, int]]):
        self.selector_indices = [int(i) for i in selector_indices]
        self.groups = [(int(a), int(b)) for a, b in groups]

    def num_selectors(self) -> int:
        return len(self.groups)


class Quotient:
    """The gate part of plonky2 plonk/prover.rs · compute_quotient_polys on the device: for every LDE row of the committed wires batch,
    acc[k] += filter * sum_i alpha_k^(offset + i) * constraint_i (evaluate_gate_constraints_base_batch + reduce_with_powers), then
    `commit` = divide by Z_H on the coset, coset_ifft, split into 2^rate_bits chunks, PolynomialBatch::from_coeffs."""

    def __init__(self, wires: "PolynomialBatch", n_challenges: int, ctx: Optional[Context] = None):
        self.ctx = ctx or wires.ctx
        self.wires, self.n_challenges = wires, n_challenges
        h = c_uint64()
        _check(self.ctx, self.ctx.lib.gl_quotient_begin(self.ctx.handle, wires.merkle_tree._h, n_challenges, byref(h)))
        self._h = h.value

    def add_gate(self, kind: int, param: int, alphas, constraint_offset: int = 0, filter: Optional[Tuple["PolynomialBatch", int]] = None) -> float:
        """returns the kernel time in ms (CUDA events)"""
        a = np.ascontiguousarray(alphas, dtype=np.uint64).reshape(-1)
        if a.size != self.n_challenges:
            raise ValueError("one alpha per challenge expected")
        fb, fc = (filter[0].merkle_tree._h, int(filter[1])) if filter is not None else (0, 0)
        _check(self.ctx, self.ctx.lib.gl_quotient_add_gate(self.ctx.handle, self._h, kind, param, _ptr(a), constraint_offset, fb, fc))
        ms = ctypes.c_float()
        self.ctx.lib.gl_ctx_aux_ms(self.ctx.handle, byref(ms))
        return float(ms.value)

    def add_gates(self, gates: Sequence[Tuple[int, int]], selectors_info: SelectorsInfo, constants_sigmas: "PolynomialBatch", num_constants: int,
                  public_inputs_hash, alphas, constraint_offset: int = 0, num_lookup_selectors: int = 0) -> float:
        """plonk/vanishing_poly.rs · evaluate_gate_constraints_base_batch over the LDE rows: gates = CommonCircuitData::gates as
        (kind, param) pairs; every gate's constraints times compute_filter(i, group, s(x), num_selectors > 1), with s the gate's selector
        column of `constants_sigmas` (commit #0) and the gate constants its columns after the selectors.  Every gate's constraint c is
        weighted by alpha_k^(constraint_offset + c).  Returns the kernel time in ms (CUDA events, first launch to last)."""
        a = np.ascontiguousarray(alphas, dtype=np.uint64).reshape(-1)
        if a.size != self.n_challenges:
            raise ValueError("one alpha per challenge expected")
        pi = np.ascontiguousarray(public_inputs_hash, dtype=np.uint64).reshape(-1)
        if pi.size != 4:
            raise ValueError("public_inputs_hash must be 4 words")
        kinds = np.array([int(g[0]) for g in gates], dtype=np.int32)
        params = np.array([int(g[1]) for g in gates], dtype=np.uint32)
        sel = np.array(selectors_info.selector_indices, dtype=np.uint32)
        if sel.size != kinds.size:
            raise ValueError("SelectorsInfo must have one selector index per gate")
        grp = np.array(selectors_info.groups, dtype=np.uint32).reshape(-1)
        _check(self.ctx, self.ctx.lib.gl_quotient_add_gates(self.ctx.handle, self._h, _ptr(kinds), _ptr(params), kinds.size, _ptr(sel), _ptr(grp),
                                                            selectors_info.num_selectors(), num_lookup_selectors, constants_sigmas.merkle_tree._h,
                                                            num_constants, _ptr(pi), _ptr(a), constraint_offset))
        ms = ctypes.c_float()
        self.ctx.lib.gl_ctx_aux_ms(self.ctx.handle, byref(ms))
        return float(ms.value)

    def add_permutation(self, sigmas: "PolynomialBatch", sigma_col0: int, zs_partial_products: "PolynomialBatch", n_routed: int, degree: int,
                        k_is, betas, gammas, alphas) -> float:
        """the permutation-argument terms of eval_vanishing_poly_base_batch — L_0(x)(Z_i(x) - 1) for every challenge, then
        check_partial_products of every challenge: vanishing_terms[0 .. n_ch * (1 + n_chunks)); gates follow from that offset.
        `sigmas`: the constants+sigmas commit (sigma polynomials at columns [sigma_col0, sigma_col0 + n_routed));
        `zs_partial_products`: the commit of partial_products_and_zs' columns.  Returns the kernel time in ms."""
        arrs = [np.ascontiguousarray(a, dtype=np.uint64).reshape(-1) for a in (k_is, betas, gammas, alphas)]
        if arrs[0].size != n_routed or any(a.size != self.n_challenges for a in arrs[1:]):
            raise ValueError("k_is: one per routed wire; betas / gammas / alphas: one per challenge")
        _check(self.ctx, self.ctx.lib.gl_quotient_add_permutation(self.ctx.handle, self._h, sigmas.merkle_tree._h, sigma_col0,
                                                                  zs_partial_products.merkle_tree._h, n_routed, degree, *[_ptr(a) for a in arrs]))
        ms = ctypes.c_float()
        self.ctx.lib.gl_ctx_aux_ms(self.ctx.handle, byref(ms))
        return float(ms.value)

    def values(self) -> np.ndarray:
        """[n_challenges][R] accumulated values, row order = the leaves' (row i = LDE point bitrev(i))"""
        out = np.zeros((self.n_challenges, self.wires.merkle_tree.n_leaves), dtype=np.uint64)
        _check(self.ctx, self.ctx.lib.gl_quotient_read(self.ctx.handle, self._h, _ptr(out)))
        return out

    def commit(self, cap_height: int) -> "PolynomialBatch":
        """quotient_polys_commitment: n_challenges * 2^rate_bits chunk polynomials of N coefficients, committed with from_coeffs"""
        t = self.wires.merkle_tree
        if cap_height > t.degree_log + t.rate_bits:
            raise ValueError(f"cap_height={cap_height} should be at most log2(leaves.len())={t.degree_log + t.rate_bits}")
        cap = np.zeros(4 << cap_height, dtype=np.uint64)
        h = c_uint64()
        _check(self.ctx, self.ctx.lib.gl_quotient_commit(self.ctx.handle, self._h, cap_height, _ptr(cap), byref(h)))
        return PolynomialBatch(self.ctx, MerkleTree(self.ctx, h.value, cap), self.n_challenges << t.rate_bits)

    def free(self):
        if self._h and self.ctx.handle:
            self.ctx.lib.gl_quotient_end(self.ctx.handle, self._h)
        self._h = 0

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def poseidon_gate_witness(inputs, ctx: Optional[Context] = None) -> np.ndarray:
    """plonky2 gates/poseidon.rs · PoseidonGenerator::run_once for a batch of PoseidonGate rows: inputs [n][13] = 12 state inputs + swap
    flag -> [n][135] wires (the shape of poseidon2_gate_witness)"""
    ctx = ctx or default_context()
    x = np.ascontiguousarray(inputs, dtype=np.uint64)
    if x.ndim != 2 or x.shape[1] != 13:
        raise ValueError("inputs must be [n][13]")
    out = np.zeros((x.shape[0], 135), dtype=np.uint64)
    _check(ctx, ctx.lib.gl_poseidon_gate_witness(ctx.handle, _ptr(x), x.shape[0], _ptr(out)))
    return out


def partial_products_and_zs(wire_cols, sigma_cols, k_is, betas, gammas, degree: int, ctx: Optional[Context] = None) -> np.ndarray:
    """plonky2 plonk/prover.rs · all_wires_permutation_partial_products with prove()'s "Z first" order: wire_cols / sigma_cols are the
    routed wires' witness values and the sigma polynomials' values on the subgroup ([n_routed][N]); returns [(n_ch * n_chunks)][N]."""
    ctx = ctx or default_context()
    w, log_n = PolynomialBatch._cols(wire_cols)
    s, log_s = PolynomialBatch._cols(sigma_cols)
    if len(w) != len(s) or log_n != log_s:
        raise ValueError("wires and sigmas must have the same shape")
    k = np.ascontiguousarray(k_is, dtype=np.uint64).reshape(-1)
    b = np.ascontiguousarray(betas, dtype=np.uint64).reshape(-1)
    g = np.ascontiguousarray(gammas, dtype=np.uint64).reshape(-1)
    if k.size != len(w) or b.size != g.size or b.size == 0:
        raise ValueError("k_is must have one entry per routed wire; betas and gammas one per challenge")
    n_chunks = -(-len(w) // degree)
    out = np.zeros((b.size * n_chunks, 1 << log_n), dtype=np.uint64)
    wp = (c_void_p * len(w))(*[c.ctypes.data for c in w])
    sp = (c_void_p * len(s))(*[c.ctypes.data for c in s])
    _check(ctx, ctx.lib.gl_partial_products(ctx.handle, wp, sp, len(w), log_n, _ptr(k), _ptr(b), _ptr(g), b.size, degree, _ptr(out)))
    return out


def poseidon2_gate_witness(inputs, ctx: Optional[Context] = None) -> np.ndarray:
    """Poseidon2Generator::run_once (/root/reference/src/common/poseidon2/poseidon2_gate.rs:447-523) for a batch of gate rows:
    inputs [n][13] = 12 state inputs + swap flag -> [n][135] wires"""
    ctx = ctx or default_context()
    x = np.ascontiguousarray(inputs, dtype=np.uint64)
    if x.ndim != 2 or x.shape[1] != 13:
        raise ValueError("inputs must be [n][13]")
    out = np.zeros((x.shape[0], 135), dtype=np.uint64)
    _check(ctx, ctx.lib.gl_poseidon2_gate_witness(ctx.handle, _ptr(x), x.shape[0], _ptr(out)))
    return out
