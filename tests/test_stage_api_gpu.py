"""The device-pointer stage API of the sharded commit plans (include/gl_commit.h) on ONE device, against the oracle.

plonky2.5_b200/sharded.py runs these calls one process per GPU; here the "peer" leaf buffers are simply more buffers on the same GPU, so
every store path is reached without a second device:
  * gl_dev_lde_scatter / gl_lde_scatter: the last NTT pass storing straight into the owner's buffer (store_mode 2, including its scalar
    stores for an odd col_off or leaf_pitch, and the tiny kernel's scatter branch at log_n < 3), the copy-engine shipment of cosets that
    belong to other owners (ship_coset, one 2-D copy per owner when a coset spans several), first_coset rotation, and the scatter_ncols
    guard that keeps padding columns out of the neighbours' columns: every word outside [col_off, col_off + n_cols) must keep its
    sentinel;
  * gl_dev_intt / gl_intt_host, then gl_dev_lde_own_cosets with columns dealt as ShardPlan deals them (uneven counts, pitches that force
    4-column groups), run once for every rank and assembled;
  * gl_dev_repack, gl_dev_merkle and gl_dev_commit at the shapes the sharded plans and their callers use them."""
import ctypes

import numpy as np
import pytest

from lde_reference import SENTINEL, DeviceBuffers, bitrev, canon, check_coeffs, make_columns, reference_lde
from oracle_c import splitmix_columns

pytestmark = pytest.mark.gpu

GL_ERR_INVALID = -1


def round_up(x, m):
    return (x + m - 1) // m * m


def _u32(*v):
    return (ctypes.c_uint32 * len(v))(*v)


def _ptrs(v):
    return (ctypes.c_void_p * len(v))(*v)


def _err(ctx):
    return ctx.lib.gl_ctx_last_error(ctx.handle).decode()


def _leaf_matrix(values):
    """[R][n_cols]: leaf row i = LDE point bitrev_R(i)"""
    R = values.shape[1]
    return values[:, bitrev(np.arange(R), R.bit_length() - 1)].T


# ---- gl_dev_lde_scatter / gl_lde_scatter ----------------------------------------------------------------------------------------------

def _scatter_cases():
    """(log_n, rate_bits, n_peers, n_cols, col_off, leaf_pitch, first_coset, own): own = the owner whose buffer comes from
    gl_dev_ipc_alloc (stored by the NTT itself when a whole coset is its), n_peers = none (every coset shipped)"""
    cases = []
    i = 0
    for log_n in (0, 2, 7, 12, 17):
        for n_peers in (1, 2, 4, 8):
            r = (1, 2, 3)[i % 3]
            while (1 << (log_n + r)) < n_peers:
                r += 1
            n_cols = (5, 4, 13, 1)[(i // 2) % 4]
            col_off = (0, 3, 8)[(i // 4) % 3]
            odd = i % 2
            leaf_pitch = round_up(col_off + n_cols, 2) + (3 if odd else 4)
            first_coset = (0, 1, (1 << r) - 1)[(i // 3) % 3]
            own = i % (n_peers + 1) if log_n >= 3 else 0          # log_n < 3: the tiny kernel's own scatter stores
            cases.append((log_n, r, n_peers, n_cols, col_off, leaf_pitch, first_coset, own))
            i += 1
    return cases


SCATTER_CASES = _scatter_cases()
# the host variant: more than 8 columns, so that several host chunks (8, 16, 24, ... columns) run
HOST_SCATTER_CASES = [(2, 2, 4, 13, 3, 19, 1, 0), (7, 1, 4, 20, 8, 32, 0, 4), (12, 3, 2, 13, 0, 16, 7, 1), (12, 2, 8, 20, 3, 27, 3, 2),
                      (17, 1, 2, 29, 8, 40, 1, 0)]


def _scatter_ids(c):
    return "logn%d_r%d_peers%d_c%d_off%d_lp%d_first%d_own%d" % c


def _run_scatter(ctx, oc, case, host):
    log_n, r, n_peers, n_cols, col_off, leaf_pitch, first_coset, own = case
    n = 1 << log_n
    R = n << r
    rpp = R // n_peers
    is_coeffs = (log_n + n_cols) % 2
    coeff_pitch = round_up(n_cols, 8) + 4 * (col_off == 3)
    cols = make_columns(n_cols, n, 3000 + log_n * 17 + n_peers, n + 5)
    with DeviceBuffers(ctx) as bufs:
        owners = [bufs.alloc(rpp * leaf_pitch, ipc=(q == own)) for q in range(n_peers)]
        coefs = bufs.alloc(n * coeff_pitch)
        if host:
            host_cols = [np.ascontiguousarray(cols[j, :n]) for j in range(n_cols)]
            rc = ctx.lib.gl_lde_scatter(ctx.handle, _ptrs([c.ctypes.data for c in host_cols]), n_cols, log_n, r, is_coeffs, _ptrs(owners),
                                        n_peers, leaf_pitch, col_off, coefs, coeff_pitch, first_coset)
        else:
            d_cols = bufs.alloc(cols.size, fill=None)
            bufs.upload(d_cols, cols)
            rc = ctx.lib.gl_dev_lde_scatter(ctx.handle, d_cols, cols.shape[1], n_cols, log_n, r, is_coeffs, _ptrs(owners), n_peers,
                                            leaf_pitch, col_off, coefs, coeff_pitch, first_coset)
        assert rc == 0, _err(ctx)
        ref_coeffs, ref_values = reference_lde(oc, cols, n, r, is_coeffs)
        check_coeffs(bufs, coefs, coeff_pitch, ref_coeffs)
        leaves = _leaf_matrix(ref_values)
        for q in range(n_peers):
            want = np.full((rpp, leaf_pitch), SENTINEL, dtype=np.uint64)
            want[:, col_off:col_off + n_cols] = leaves[q * rpp:(q + 1) * rpp]
            got = bufs.rows(owners[q], 0, rpp, leaf_pitch)
            if not np.array_equal(got, want):
                row, col = (int(v) for v in np.argwhere(got != want)[0])
                raise AssertionError(f"owner {q}: row {row} column {col}: got {int(got[row, col]):#x}, want {int(want[row, col]):#x} "
                                     f"(columns [{col_off}, {col_off + n_cols}) are this call's, the rest must keep the sentinel)")


def test_scatter_cases_cover_the_store_paths():
    """the case table reaches both coset placements, odd and even pitches, every col_off and both ends of the rotation"""
    spans = {n_peers > (1 << r) for _, r, n_peers, *_ in SCATTER_CASES}
    assert spans == {True, False}
    assert {lp % 2 for *_, lp, _, _ in SCATTER_CASES} == {0, 1}
    assert {c[4] for c in SCATTER_CASES} == {0, 3, 8}
    assert {c[6] for c in SCATTER_CASES} >= {0, 1, 3, 7}
    assert any(c[0] < 3 and c[7] < c[2] and c[2] <= 1 << c[1] for c in SCATTER_CASES)     # tiny kernel, store_mode 2


@pytest.mark.parametrize("case", SCATTER_CASES, ids=_scatter_ids)
def test_dev_lde_scatter(ctx, oc, case):
    _run_scatter(ctx, oc, case, host=False)


@pytest.mark.parametrize("case", HOST_SCATTER_CASES, ids=_scatter_ids)
def test_lde_scatter_host_columns(ctx, oc, case):
    _run_scatter(ctx, oc, case, host=True)


# ---- gl_dev_intt / gl_intt_host, then gl_dev_lde_own_cosets ---------------------------------------------------------------------------

OWN_COSET_CASES = [  # (log_n, rate_bits, n_peers, n_cols, leaf_pitch extra words beyond round_up(n_cols, 8), input_is_coeffs)
    (3, 1, 1, 5, 0, 0), (9, 2, 1, 13, 4, 1), (10, 1, 2, 37, 0, 0), (12, 2, 4, 37, 4, 1), (7, 3, 8, 37, 0, 0), (11, 3, 8, 70, 4, 0),
    (14, 2, 2, 21, 0, 1), (17, 3, 4, 45, 0, 0), (2, 3, 8, 37, 4, 1)]


@pytest.mark.parametrize("case", OWN_COSET_CASES, ids=lambda c: "logn%d_r%d_peers%d_c%d_lp+%d_%s" % (*c[:5], "coeffs" if c[5] else "values"))
def test_intt_then_lde_own_cosets(ctx, oc, case):
    """every rank's iNTT block (device and host columns agree), then every rank's own cosets from all blocks; the assembled leaf rows
    equal the oracle's and nothing lands beyond column round_up(n_cols, 4) of a leaf row"""
    from plonky25_b200.sharded import ShardPlan
    log_n, r, n_peers, n_cols, extra, is_coeffs = case
    n = 1 << log_n
    plan = ShardPlan(n_cols, log_n, r, 3, n_peers)
    leaf_pitch = plan.leaf_pitch + extra
    rpp = plan.rows_per_rank
    lib, h = ctx.lib, ctx.handle
    cols = make_columns(n_cols, n, 5000 + log_n + n_peers)
    ref_coeffs, ref_values = reference_lde(oc, cols, n, r, is_coeffs)
    leaves = _leaf_matrix(ref_values)
    with DeviceBuffers(ctx) as bufs:
        blocks = []
        for q in range(n_peers):
            c0, c1 = plan.col_range(q)
            cnt, pitch = c1 - c0, plan.pitches[q]
            d_cols = bufs.alloc(cnt * n, fill=None)
            bufs.upload(d_cols, cols[c0:c1])
            blk = bufs.alloc(n * pitch)
            assert lib.gl_dev_intt(h, d_cols, n, cnt, log_n, is_coeffs, blk, pitch) == 0, _err(ctx)
            check_coeffs(bufs, blk, pitch, ref_coeffs[c0:c1], what=f"rank {q} coefficient block")
            from_host = bufs.alloc(n * pitch)
            host_cols = [np.ascontiguousarray(cols[j]) for j in range(c0, c1)]
            assert lib.gl_intt_host(h, _ptrs([c.ctypes.data for c in host_cols]), cnt, log_n, is_coeffs, from_host, pitch) == 0, _err(ctx)
            assert np.array_equal(bufs.download(from_host, n * pitch), bufs.download(blk, n * pitch)), f"rank {q}: gl_intt_host != gl_dev_intt"
            blocks.append(blk)
        for me in range(n_peers):
            stage = [0 if q == me else bufs.alloc(n * plan.pitches[q], fill=None) for q in range(n_peers)]
            out = bufs.alloc(rpp * leaf_pitch)
            rc = lib.gl_dev_lde_own_cosets(h, _ptrs(blocks), _ptrs(stage), _u32(*plan.pitches), _u32(*plan.col_counts),
                                           _u32(*plan.col_offsets), n_peers, me, log_n, r, out, leaf_pitch)
            assert rc == 0, _err(ctx)
            got = bufs.rows(out, 0, rpp, leaf_pitch)
            want = leaves[me * rpp:(me + 1) * rpp]
            if not np.array_equal(got[:, :n_cols], want):
                row, col = (int(v) for v in np.argwhere(got[:, :n_cols] != want)[0])
                raise AssertionError(f"rank {me}: leaf row {me * rpp + row} column {col}: got {int(got[row, col]):#x}, want {int(want[row, col]):#x}")
            assert (got[:, round_up(n_cols, 4):] == SENTINEL).all(), f"rank {me}: stores beyond the last column group"


def test_lde_own_cosets_refuses_a_pitch_of_partial_groups(ctx):
    """leaf_pitch = 13 with one 13-column block of pitch 16 would store columns 13..15 of every row into the next row (and past the end of
    d_leaves): refused before anything runs.  The buffers are large enough that even an accepted call stays inside them."""
    lib, h = ctx.lib, ctx.handle
    log_n, n = 6, 64
    with DeviceBuffers(ctx) as bufs:
        blk = bufs.alloc(n * 16, fill=0)
        out_words = 2 * n * 24                          # 2N leaf rows of up to 24 words: room for any of the pitches below
        out = bufs.alloc(out_words)
        for leaf_pitch, offset, message in ((13, 0, "leaf_pitch must be a multiple of 4"), (14, 0, "leaf_pitch must be a multiple of 4"),
                                            (15, 0, "leaf_pitch must be a multiple of 4"), (20, 2, "bad column layout")):
            rc = lib.gl_dev_lde_own_cosets(h, _ptrs([blk]), _ptrs([0]), _u32(16), _u32(13), _u32(offset), 1, 0, log_n, 1, out, leaf_pitch)
            assert rc == GL_ERR_INVALID and message in _err(ctx), (leaf_pitch, offset, _err(ctx))
        assert (bufs.download(out, out_words) == SENTINEL).all()
        # the same block at pitch 16 is accepted
        assert lib.gl_dev_lde_own_cosets(h, _ptrs([blk]), _ptrs([0]), _u32(16), _u32(13), _u32(0), 1, 0, log_n, 1, out, 16) == 0, _err(ctx)


# ---- gl_dev_repack, gl_dev_merkle, gl_dev_commit ---------------------------------------------------------------------------------------

@pytest.mark.parametrize("shape", [(1000, 12, 5, 16, 3), (257, 8, 8, 24, 16), (64, 4, 1, 8, 7), (0, 8, 5, 8, 0)])
def test_dev_repack(ctx, shape):
    """the first src_cols columns of [n_rows][src_pitch] land canonical in columns [off, off + src_cols) of [n_rows][dst_pitch]; every
    other word keeps its sentinel (n_rows = 0: nothing is written)"""
    n_rows, src_pitch, src_cols, dst_pitch, off = shape
    src = make_columns(max(n_rows, 1), src_pitch, 31 + n_rows)          # non-canonical and edge words among them
    with DeviceBuffers(ctx) as bufs:
        d_src = bufs.alloc(src.size, fill=None)
        bufs.upload(d_src, src)
        rows = max(n_rows, 1)
        d_dst = bufs.alloc(rows * dst_pitch)
        assert ctx.lib.gl_dev_repack(ctx.handle, d_src, src_pitch, src_cols, n_rows, d_dst, dst_pitch, off) == 0, _err(ctx)
        want = np.full((rows, dst_pitch), SENTINEL, dtype=np.uint64)
        if n_rows:
            want[:, off:off + src_cols] = canon(src[:, :src_cols])
        assert np.array_equal(bufs.rows(d_dst, 0, rows, dst_pitch), want)


@pytest.mark.parametrize("shape", [(256, 12, 16, 0), (256, 12, 16, 8), (64, 4, 8, 2), (32, 1, 8, 5), (128, 3, 8, 7), (8, 135, 136, 3),
                                   (1, 7, 8, 0)])
def test_dev_merkle(ctx, oc, shape):
    """leaf rows with a pitch beyond leaf_len and non-canonical words; cap_height 0 and log2(n_leaves); leaf_len <= 4 (hash_or_noop: the
    leaf is its own digest, no permutation)"""
    n_leaves, leaf_len, pitch, cap_height = shape
    rows = make_columns(n_leaves, pitch, 41 + leaf_len)
    dig, cap = oc.merkle_new(canon(rows[:, :leaf_len]), cap_height)
    with DeviceBuffers(ctx) as bufs:
        d_rows = bufs.alloc(rows.size, fill=None)
        bufs.upload(d_rows, rows)
        n_dig = 2 * (n_leaves - (1 << cap_height)) * 4
        d_dig = bufs.alloc(n_dig) if n_dig else 0
        out_cap = np.zeros(4 << cap_height, dtype=np.uint64)
        rc = ctx.lib.gl_dev_merkle(ctx.handle, d_rows, n_leaves, leaf_len, pitch, cap_height, d_dig or None, out_cap.ctypes.data)
        assert rc == 0, _err(ctx)
        assert np.array_equal(out_cap.reshape(-1, 4), cap)
        if n_dig:
            assert np.array_equal(bufs.download(d_dig, n_dig).reshape(-1, 4), dig)


@pytest.mark.parametrize("n_cols", range(1, 41))
def test_dev_commit_widths(ctx, oc, n_cols):
    """gl_dev_commit (column group from column_group, one leaf_hash_kernel sweep) at every width 1..40 with columns further apart than N,
    against the oracle's commit: cap, and the batch's coefficients, leaves and digests"""
    log_n, r = 3 + n_cols % 7, 1 + n_cols % 3
    h = min(n_cols % 5, log_n + r)
    n, R = 1 << log_n, 1 << (log_n + r)
    is_coeffs = n_cols % 2
    cols = make_columns(n_cols, n, 7000 + n_cols, n + 7)
    ref = oc.commit([canon(c[:n]) for c in cols], r, h, is_coeffs=bool(is_coeffs))
    lib = ctx.lib
    with DeviceBuffers(ctx) as bufs:
        d_cols = bufs.alloc(cols.size, fill=None)
        bufs.upload(d_cols, cols)
        cap = np.zeros(4 << h, dtype=np.uint64)
        batch = ctypes.c_uint64()
        assert lib.gl_dev_commit(ctx.handle, d_cols, n + 7, n_cols, log_n, r, h, is_coeffs, cap.ctypes.data, ctypes.byref(batch)) == 0, _err(ctx)
        try:
            assert np.array_equal(cap.reshape(-1, 4), ref["cap"])
            parts = {0: np.zeros(n * n_cols, dtype=np.uint64), 1: np.zeros(R * n_cols, dtype=np.uint64),
                     2: np.zeros(max(ref["digests"].size, 1), dtype=np.uint64)}
            for part, buf in parts.items():
                if part == 2 and not ref["digests"].size:
                    continue
                assert lib.gl_tree_read(ctx.handle, batch.value, part, buf.ctypes.data) == 0, _err(ctx)
            assert np.array_equal(parts[0].reshape(n_cols, n), ref["coeffs"])
            assert np.array_equal(parts[1].reshape(R, n_cols), ref["leaves"])
            if ref["digests"].size:
                assert np.array_equal(parts[2].reshape(-1, 4), ref["digests"])
        finally:
            lib.gl_tree_free(ctx.handle, batch.value)
