"""Lifecycle of the objects a context hands out (trees, FRI states, openings, quotients), through the C ABI: release, use after
release, a handle of one kind passed where another kind is expected, and destroying a context that still holds objects."""
from ctypes import byref, c_uint64, c_void_p

import numpy as np
import pytest

from oracle_c import splitmix_columns

pytestmark = pytest.mark.gpu

LOG_N, N_COLS, RATE_BITS, CAP_HEIGHT = 4, 17, 1, 1   # 17 wires: one GL_GATE_U32_RANGE_CHECK op (param 1)
GL_GATE_U32_RANGE_CHECK = 4


def _lib():
    from plonky25_b200 import _lib
    return _lib


def _ptr(a):
    return a.ctypes.data_as(c_void_p)


@pytest.fixture
def hctx():
    import plonky25_b200 as g
    c = g.Context(0)
    yield c
    c.close()


def _ok(ctx, rc):
    assert rc == _lib().GL_OK, ctx.lib.gl_ctx_last_error(ctx.handle).decode()


def _commit(ctx):
    cols = splitmix_columns(7, N_COLS, 1 << LOG_N)
    ptrs = (c_void_p * N_COLS)(*[c.ctypes.data for c in cols])
    cap = np.zeros(4 << CAP_HEIGHT, dtype=np.uint64)
    h = c_uint64()
    _ok(ctx, ctx.lib.gl_commit(ctx.handle, ptrs, N_COLS, LOG_N, RATE_BITS, CAP_HEIGHT, 0, None, None, None, _ptr(cap), byref(h)))
    return h.value


def _merkle_new(ctx):
    leaves = splitmix_columns(8, 16, 5)
    cap = np.zeros(4 << CAP_HEIGHT, dtype=np.uint64)
    h = c_uint64()
    _ok(ctx, ctx.lib.gl_merkle_new(ctx.handle, _ptr(leaves), 16, 5, CAP_HEIGHT, None, _ptr(cap), byref(h)))
    return h.value


def _fri_begin(ctx):
    coeffs, values = splitmix_columns(9, 2, 32)
    h = c_uint64()
    _ok(ctx, ctx.lib.gl_fri_begin(ctx.handle, _ptr(coeffs), _ptr(values), 16, RATE_BITS, CAP_HEIGHT, byref(h)))
    return h.value


def _openings_begin(ctx):
    h = c_uint64()
    _ok(ctx, ctx.lib.gl_openings_begin(ctx.handle, LOG_N, byref(h)))
    return h.value


def _openings_lde(ctx, oh):
    h = c_uint64()
    _ok(ctx, ctx.lib.gl_openings_lde(ctx.handle, oh, RATE_BITS, CAP_HEIGHT, byref(h)))
    return h.value


def _quotient_begin(ctx, wires):
    h = c_uint64()
    _ok(ctx, ctx.lib.gl_quotient_begin(ctx.handle, wires, 1, byref(h)))
    return h.value


# the read call and the release call of each kind; _OUT is large enough for any object this file creates
_OUT = np.zeros(1 << 12, dtype=np.uint64)
READ = {
    "tree": lambda ctx, h: ctx.lib.gl_tree_info(ctx.handle, h, byref(_lib().TreeInfo())),
    "fri": lambda ctx, h: ctx.lib.gl_fri_read(ctx.handle, h, None, None, byref(c_uint64())),
    "openings": lambda ctx, h: ctx.lib.gl_openings_final_poly(ctx.handle, h, _ptr(_OUT)),
    "quotient": lambda ctx, h: ctx.lib.gl_quotient_read(ctx.handle, h, _ptr(_OUT)),
}
RELEASE = {
    "tree": lambda ctx, h: ctx.lib.gl_tree_free(ctx.handle, h),
    "fri": lambda ctx, h: ctx.lib.gl_fri_end(ctx.handle, h),
    "openings": lambda ctx, h: ctx.lib.gl_openings_end(ctx.handle, h),
    "quotient": lambda ctx, h: ctx.lib.gl_quotient_end(ctx.handle, h),
}


def _one_of_each(ctx):
    """(kind, handle) for every entry point that creates an object"""
    wires = _commit(ctx)
    oh = _openings_begin(ctx)
    return [("tree", _merkle_new(ctx)), ("tree", wires), ("fri", _fri_begin(ctx)), ("fri", _openings_lde(ctx, oh)),
            ("openings", oh), ("quotient", _quotient_begin(ctx, wires))]


def test_release_once_then_unknown(hctx):
    objs = _one_of_each(hctx)
    for kind, h in objs:
        _ok(hctx, READ[kind](hctx, h))
        assert RELEASE[kind](hctx, h) == _lib().GL_OK
        assert RELEASE[kind](hctx, h) == _lib().GL_ERR_HANDLE
        assert READ[kind](hctx, h) == _lib().GL_ERR_HANDLE
        assert f"unknown {kind} handle" in hctx.lib.gl_ctx_last_error(hctx.handle).decode()


def test_handle_of_one_kind_is_no_other_kind(hctx):
    objs = _one_of_each(hctx)
    assert len({h for _, h in objs}) == len(objs)
    for kind, h in objs:
        for other in READ:
            if other == kind:
                continue
            assert READ[other](hctx, h) == _lib().GL_ERR_HANDLE, (kind, other)
            assert f"unknown {other} handle" in hctx.lib.gl_ctx_last_error(hctx.handle).decode()
        _ok(hctx, READ[kind](hctx, h))   # a failed lookup leaves the object alone
    for kind, h in reversed(objs):
        _ok(hctx, RELEASE[kind](hctx, h))


def test_quotient_outliving_its_wires(hctx):
    wires = _commit(hctx)
    q = _quotient_begin(hctx, wires)
    _ok(hctx, hctx.lib.gl_tree_free(hctx.handle, wires))
    alphas = np.array([3], dtype=np.uint64)
    rc = hctx.lib.gl_quotient_add_gate(hctx.handle, q, GL_GATE_U32_RANGE_CHECK, 1, _ptr(alphas), 0, 0, 0)
    assert rc == _lib().GL_ERR_HANDLE
    assert "unknown tree handle" in hctx.lib.gl_ctx_last_error(hctx.handle).decode()
    _ok(hctx, READ["quotient"](hctx, q))
    _ok(hctx, hctx.lib.gl_quotient_end(hctx.handle, q))


def test_destroy_with_live_objects_then_fresh_context(oc):
    import plonky25_b200 as g
    c = g.Context(0)
    objs = _one_of_each(c)
    assert {k for k, _ in objs} == set(READ)
    c.close()   # gl_ctx_destroy with every object still alive
    c = g.Context(0)
    try:
        log_n, n_cols, r, h = 4, 9, 3, 4   # one of test_gpu_parity's COMMIT_SHAPES
        cols = splitmix_columns(1000 + log_n * 13 + n_cols, n_cols, 1 << log_n, canonical=(log_n % 2 == 0))
        ref = oc.commit(cols, r, h)
        pb = g.PolynomialBatch.from_values(list(cols), r, False, h, ctx=c, copy_back=True)
        assert np.array_equal(pb.polynomials, ref["coeffs"])
        assert np.array_equal(pb.merkle_tree.leaves, ref["leaves"])
        assert np.array_equal(pb.merkle_tree.digests, ref["digests"])
        assert np.array_equal(pb.merkle_tree.cap.hashes, ref["cap"])
        pb.merkle_tree.free()
    finally:
        c.close()
