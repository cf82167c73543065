"""Every NTT pass plan of the transform layer against the oracle on one GPU (include/gl_commit.h · gl_dev_lde).

gl_commit.cu · plan_passes splits log_n into shared-memory passes; each plan runs different instantiations of the pass kernels
(csrc/ntt2.cuh, and csrc/ntt.cuh for outputs that are not 16-byte aligned), with different epilogues (radix-8 or radix-16 last round,
with or without the inter-pass twiddle).  The sweep below runs every log_n from 0 to 24 with both column groups (G = 4 when
n_cols % 8 is 1..4, else G = 8), values and coefficient inputs, non-canonical and structured words, a column stride larger than N and
an output pitch larger than needed, and compares the coefficients and the whole leaf matrix bit for bit with the C oracle, plus an
O(N^2) Python-integer DFT up to 2^10 and Horner evaluations of sampled leaf rows at every size.  The outputs are pre-filled with a
non-canonical sentinel, so that a row or column the kernels never wrote cannot pass."""
import random

import numpy as np
import pytest

import gl_oracle as o
from lde_reference import (SENTINEL, DeviceBuffers, canon, check_coeffs, check_leaves, eval_points, horner, leaf_point, make_columns,
                           reference_lde)
from oracle_c import P

pytestmark = pytest.mark.gpu


def plan_passes(log_n, max_a=10):
    """mirror of gl_commit.cu · plan_passes: log_n stages in ceil(log_n / 10) passes as even as possible, larger passes first;
    [] = the tiny kernel (log_n < 3)"""
    if log_n < 3:
        return []
    k = (log_n + max_a - 1) // max_a
    base, rem = divmod(log_n, k)
    return [base + (1 if i < rem else 0) for i in range(k)]


# The plans this file was written against.  If gl_commit.cu's plan changes, test_pass_plans_match_the_sweep fails and names the
# sizes whose new plans the sweep (and its choice of sizes) must be revisited for.
SWEPT_PLANS = {0: [], 1: [], 2: [], 3: [3], 4: [4], 5: [5], 6: [6], 7: [7], 8: [8], 9: [9], 10: [10], 11: [6, 5], 12: [6, 6],
               13: [7, 6], 14: [7, 7], 15: [8, 7], 16: [8, 8], 17: [9, 8], 18: [9, 9], 19: [10, 9], 20: [10, 10], 21: [7, 7, 7],
               22: [8, 7, 7], 23: [8, 8, 7], 24: [8, 8, 8]}

WIDTHS = (1, 4, 5, 8, 13)   # G = 4, 4, 8, 8, 8


def group(n_cols):
    return 4 if (-n_cols) % 8 >= 4 else 8


def round_up(x, m):
    return (x + m - 1) // m * m


def _cases():
    """(log_n, rate_bits, n_cols, input_is_coeffs, extra pitch words)"""
    cases = []
    for log_n in range(14):
        cases.append((log_n, 1 + log_n % 4, WIDTHS[log_n % 5], 0, 4 * (log_n % 2)))
        cases.append((log_n, 1 + (log_n + 2) % 4, WIDTHS[(log_n + 2) % 5], 1, 4 * (1 - log_n % 2)))
    # 2^14 (7+7), 2^17 (9+8: the A = 9 radix-8 epilogue with an inter-pass twiddle), 2^18 (9+9), 2^19 (10+9): every width
    for log_n in (14, 17, 18, 19):
        for k, w in enumerate(WIDTHS):
            r = 1 + (log_n + k) % (4 if log_n < 19 else 2)
            cases.append((log_n, r, w, k % 2, 4 * (k % 2)))
    cases += [(15, 2, 5, 0, 4), (15, 1, 4, 1, 0), (16, 3, 13, 1, 0), (16, 1, 1, 0, 4), (20, 1, 5, 0, 0), (20, 2, 4, 1, 0),
              (21, 2, 4, 0, 0), (21, 1, 5, 1, 0), (22, 1, 5, 0, 0), (22, 1, 1, 1, 0),
              (23, 1, 1, 0, 0), (23, 1, 4, 1, 0), (23, 1, 5, 0, 0), (24, 1, 1, 0, 0), (24, 1, 1, 1, 0)]
    return cases


def _launches(ctx):
    return ctx.stage_times()[1]


def _check_plan(ctx, log_n, rate_bits, is_coeffs):
    passes = max(len(plan_passes(log_n)), 1)          # the tiny kernel is one launch
    ln = _launches(ctx)
    assert ln["intt"] == (0 if is_coeffs else passes), (log_n, ln)
    assert ln["lde"] == passes << rate_bits, (log_n, ln)


def _run_lde(ctx, bufs, cols, n, n_cols, rate_bits, is_coeffs, pitch, misalign=0):
    """gl_dev_lde of the uploaded columns into sentinel-filled outputs; misalign = word offset of both output bases"""
    R = n << rate_bits
    stride = cols.shape[1]
    d_cols = bufs.alloc(cols.size, fill=None)
    bufs.upload(d_cols, cols)
    rows_buf = bufs.alloc(R * pitch + 2 * misalign)
    coef_buf = bufs.alloc(n * pitch + 2 * misalign)
    rows, coefs = rows_buf + 8 * misalign, coef_buf + 8 * misalign
    rc = ctx.lib.gl_dev_lde(ctx.handle, d_cols, stride, n_cols, n.bit_length() - 1, rate_bits, is_coeffs, rows, pitch, coefs)
    assert rc == 0, ctx.lib.gl_ctx_last_error(ctx.handle).decode()
    return rows_buf, coef_buf, rows, coefs


def _independent_checks(bufs, coeffs, pitch, cols, n, n_cols, rate_bits, is_coeffs, rows, rng):
    """Python integers only (no oracle): up to 2^10 the coefficients interpolate the inputs (O(N^2) DFT) and, when N * R <= 2^20, every
    leaf row is the DFT of the coefficients; otherwise sampled rows are Horner evaluations at 7 * w_R^bitrev(i).  coeffs: the device's
    coefficients (already found equal to the oracle's)."""
    R, bits = n << rate_bits, (n << rate_bits).bit_length() - 1
    for j in sorted({0, n_cols - 1}):
        c = coeffs[j]
        if n <= 1 << 10 and not is_coeffs:
            w = o.primitive_root_of_unity(n.bit_length() - 1)
            assert eval_points(c, [pow(w, k, P) for k in range(n)]) == [int(v) for v in canon(cols[j][:n])], f"column {j}"
        if n * R <= 1 << 20:
            idx = list(range(R))
        else:
            idx = sorted({0, 1, R - 1, rng.randrange(R)}) if n <= 1 << 20 else [rng.randrange(R)]
        want = eval_points(c, [leaf_point(i, bits) for i in idx]) if len(idx) > 8 else [horner(c, leaf_point(i, bits)) for i in idx]
        got = [int(bufs.rows(rows, i, 1, pitch)[0, j]) for i in idx]
        assert got == want, f"column {j}: leaf rows {idx}"


@pytest.mark.parametrize("case", _cases(), ids=lambda c: "logn%d_r%d_c%d_%s_p+%d" % (c[0], c[1], c[2], "coeffs" if c[3] else "values", c[4]))
def test_lde_plan_sweep(ctx, oc, case):
    log_n, r, n_cols, is_coeffs, extra = case
    n = 1 << log_n
    pitch = round_up(n_cols, group(n_cols)) + extra
    stride = n + 3 if log_n < 21 else n                  # columns further apart than N (an odd number of words)
    seed = 1000 * log_n + 10 * n_cols + is_coeffs
    cols = make_columns(n_cols, n, seed, stride)
    rng = random.Random(seed)
    with DeviceBuffers(ctx) as bufs:
        _, _, rows, coefs = _run_lde(ctx, bufs, cols, n, n_cols, r, is_coeffs, pitch)
        _check_plan(ctx, log_n, r, is_coeffs)
        ref_coeffs, ref_values = reference_lde(oc, cols, n, r, is_coeffs)
        if n > 1 << 10:
            cols = None                                  # host memory: the inputs are needed again only by the O(N^2) check
        check_coeffs(bufs, coefs, pitch, ref_coeffs)
        check_leaves(bufs, rows, pitch, 0, ref_values, r)
        del ref_values
        _independent_checks(bufs, ref_coeffs, pitch, cols, n, n_cols, r, is_coeffs, rows, rng)


@pytest.mark.parametrize("log_n", [3, 4, 5, 6, 7, 8, 9, 10, 12])
def test_lde_misaligned_outputs(ctx, oc, log_n):
    """d_out_rows and d_out_coeffs one word past a 16-byte boundary (a legal slice of a caller's buffer): every pass runs the
    first-generation <4, A> / <8, A> kernels, which access memory one word at a time.  The words just outside both outputs stay
    untouched."""
    n_cols = (5, 4, 13)[log_n % 3]
    r = 1 + log_n % 3
    is_coeffs = log_n % 2
    n, pitch = 1 << log_n, round_up(n_cols, group(n_cols))
    R = n << r
    cols = make_columns(n_cols, n, 77 + log_n)
    with DeviceBuffers(ctx) as bufs:
        rows_buf, coef_buf, rows, coefs = _run_lde(ctx, bufs, cols, n, n_cols, r, is_coeffs, pitch, misalign=1)
        _check_plan(ctx, log_n, r, is_coeffs)
        ref_coeffs, ref_values = reference_lde(oc, cols, n, r, is_coeffs)
        check_coeffs(bufs, coefs, pitch, ref_coeffs)
        check_leaves(bufs, rows, pitch, 0, ref_values, r)
        for buf, words in ((rows_buf, R * pitch), (coef_buf, n * pitch)):
            assert bufs.download(buf, 1)[0] == SENTINEL and bufs.download(buf, 1, words + 1)[0] == SENTINEL


def test_pass_plans_match_the_sweep(ctx):
    """The plans the sweep assumes are the plans the library runs: the Python mirror of plan_passes gives the table above, and the launch
    counts of gl_dev_intt and gl_dev_lde (gl_ctx_stage_times) at every log_n match it.  A mismatch names the sizes to revisit."""
    stale = [k for k in SWEPT_PLANS if plan_passes(k) != SWEPT_PLANS[k]]
    assert not stale, f"plan_passes mirror differs from the swept plans at log_n {stale}"
    lib, h = ctx.lib, ctx.handle
    wrong = {}
    for log_n in range(25):
        with DeviceBuffers(ctx) as bufs:
            n = 1 << log_n
            d_cols = bufs.alloc(n, fill=1)
            out = bufs.alloc(4 * (n << 1), fill=None)
            coef = bufs.alloc(4 * n, fill=None)
            assert lib.gl_dev_intt(h, d_cols, n, 1, log_n, 0, coef, 4) == 0, lib.gl_ctx_last_error(h).decode()
            intt = _launches(ctx)["intt"]
            assert lib.gl_dev_lde(h, d_cols, n, 1, log_n, 1, 0, out, 4, coef) == 0, lib.gl_ctx_last_error(h).decode()
            lde = _launches(ctx)["lde"] // 2
            want = max(len(SWEPT_PLANS[log_n]), 1)
            if (intt, lde) != (want, want):
                wrong[log_n] = (intt, lde, want)
    assert not wrong, f"pass counts (iNTT, LDE per coset, swept) differ at log_n {wrong}: revisit the sweep's sizes for the new plan"
