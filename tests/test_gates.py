"""§8(f) ranks 3-4: the reference's own gates on the GPU — constraint evaluation over the resident LDE rows (what
compute_quotient_polys does per gate) and Poseidon2Gate witness generation — against oracle/gates_oracle.py, a line-by-line
restatement of Rust that IS in the reference tree (/root/reference/src/common/poseidon2/poseidon2_gate.rs:233-310, :447-523;
/root/reference/src/common/u32/gates/arithmetic_u32.rs:103-166)."""
import ctypes
import json
import os
import random

import numpy as np
import pytest

import gates_oracle as go
from oracle_c import splitmix_columns

P = go.P
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------------------------------------ CPU: the oracle itself
def test_poseidon2_constants_match_the_reference_source():
    """tests/golden/poseidon2_constants.json holds the constants as parsed out of the reference's poseidon2_goldilocks.rs
    (tools/gen_poseidon2_constants.py); the oracle's and the device's tables must be those numbers."""
    fix = json.load(open(os.path.join(ROOT, "tests", "golden", "poseidon2_constants.json")))
    assert fix["MAT_DIAG_M_1"] == go.MAT_DIAG_M_1 and fix["RC"] == go.RC and fix["RC_MID"] == go.RC_MID
    assert all(0 <= x < P for row in go.RC for x in row) and all(0 <= x < P for x in go.RC_MID)
    cuh = open(os.path.join(ROOT, "plonky2.5_b200", "csrc", "poseidon2_constants.cuh")).read()
    for x in go.RC_MID + go.RC[3] + [d - 1 for d in go.MAT_DIAG_M_1]:
        assert "0x%016xULL" % x in cuh


def test_gate_oracle_consistency():
    """rows filled by the generators satisfy every constraint; outputs are the permutation; tampering any wire breaks a constraint"""
    rnd = random.Random(5)
    assert go.POSEIDON2_NUM_WIRES == 135 and go.POSEIDON2_NUM_CONSTRAINTS == 123
    for swap in (0, 1):
        x = [rnd.randrange(P) for _ in range(12)]
        w = go.poseidon2_gate_witness(x, swap)
        assert not any(go.poseidon2_gate_eval(w))
        assert w[12:24] == go.poseidon2(x[4:8] + x[0:4] + x[8:12] if swap else x)
        for i in rnd.sample(range(135), 20):
            t = list(w)
            t[i] = (t[i] + 1) % P
            assert any(go.poseidon2_gate_eval(t)), i
    assert go.u32_arith_num_ops() == 3
    ops = [(0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF), (0, 5, 7), (rnd.getrandbits(32), rnd.getrandbits(32), rnd.getrandbits(32))]
    w = go.u32_arithmetic_witness(ops)
    assert len(go.u32_arithmetic_eval(w)) == 108 and not any(go.u32_arithmetic_eval(w))
    w[3] ^= 1
    assert any(go.u32_arithmetic_eval(w))


# ------------------------------------------------------------------------------------------------ GPU
def _rows(kind, n, seed):
    """n x 135 rows: valid gate rows, valid rows with one wire tampered, and arbitrary field elements (incl. non-canonical words)"""
    rnd = random.Random(seed)
    rows = []
    for r in range(n):
        m = r % 3
        if kind == 0:
            w = go.poseidon2_gate_witness([rnd.randrange(P) for _ in range(12)], rnd.randrange(2))
        else:
            w = go.u32_arithmetic_witness([(rnd.getrandbits(32), rnd.getrandbits(32), rnd.getrandbits(32)) for _ in range(3)])
        if m == 1:
            w[rnd.randrange(len(w))] = rnd.randrange(P)
        if m == 2:
            w = [rnd.getrandbits(64) for _ in range(135)]
        rows.append(w)
    return np.array(rows, dtype=np.uint64)


def _other_gate_case(kind, param, rnd):
    """(valid witness row, oracle evaluator) for the u32 / b32 gates 2..8"""
    u = lambda: rnd.getrandbits(32)
    lo, hi = param & 0xFF, param >> 8
    if kind == 2:
        return go.add_many_witness([([u() for _ in range(lo)], rnd.randrange(4)) for _ in range(hi)], lo), lambda w: go.add_many_eval(w, lo, hi)
    if kind == 3:
        return go.subtraction_witness([(u(), u(), rnd.randrange(2)) for _ in range(param)]), lambda w: go.subtraction_eval(w, param)
    if kind == 4:
        return go.range_check_witness([u() for _ in range(param)]), lambda w: go.range_check_eval(w, param)
    if kind == 5:
        return go.interleave_witness([u() for _ in range(param)]), lambda w: go.interleave_eval(w, param)
    if kind in (6, 7):
        return go.uninterleave_witness([rnd.getrandbits(63) for _ in range(param)], kind == 7), lambda w: go.uninterleave_eval(w, param, kind == 7)
    a, b = (u(), u()) if rnd.random() < 0.7 else (7, 7)
    return go.comparison_witness(a & ((1 << lo) - 1), b & ((1 << lo) - 1), lo, hi), lambda w: go.comparison_eval(w, lo, hi)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,param", [(2, 5 | 5 << 8), (2, 24 | 1 << 8), (3, 6), (3, 1), (4, 7), (5, 3), (6, 2), (7, 2), (7, 1), (8, 32 | 16 << 8),
                                        (8, 10 | 2 << 8)])
def test_other_u32_gates_match_oracle(ctx, kind, param):
    """the reference's remaining gates (src/common/u32/gates/{add_many_u32,subtraction_u32,range_check_u32,interleave_u32,
    uninterleave_to_u32,uninterleave_to_b32,comparison}.rs): every constraint of valid, tampered and arbitrary rows"""
    lib, rnd = ctx.lib, random.Random(1000 * kind + param)
    nw, nc = lib.gl_gate_num_wires(kind, param), lib.gl_gate_num_constraints(kind, param)
    rows, evalf = [], None
    for r in range(48):
        w, evalf = _other_gate_case(kind, param, rnd)
        w = w[:nw]
        assert not any(evalf(w)), "the oracle's own witness must satisfy the gate"
        if r % 3 == 1:
            w[rnd.randrange(nw)] = rnd.randrange(P)
        if r % 3 == 2:
            w = [rnd.getrandbits(64) for _ in range(nw)]
        rows.append(w)
    rows = np.array(rows, dtype=np.uint64)
    assert len(evalf(rows[0].tolist())) == nc
    out = np.zeros((rows.shape[0], nc), dtype=np.uint64)
    assert lib.gl_gate_eval_rows(ctx.handle, kind, param, rows.ctypes.data, rows.shape[0], out.ctypes.data) == 0
    for r in range(rows.shape[0]):
        assert out[r].tolist() == evalf(rows[r].tolist()), r
    assert lib.gl_gate_num_wires(kind, 0) == -1 or kind == 0


@pytest.mark.gpu
@pytest.mark.parametrize("kind,param", [(0, 0), (1, 3), (1, 1)])
def test_gate_constraints_match_oracle(ctx, kind, param):
    lib = ctx.lib
    nw, nc = lib.gl_gate_num_wires(kind, param), lib.gl_gate_num_constraints(kind, param)
    assert (nw, nc) == ((135, 123) if kind == 0 else (38 * param, 36 * param))
    rows = _rows(kind, 96, 40 + kind)[:, :nw].copy()
    if kind == 1 and param == 1:
        rows = np.array([go.u32_arithmetic_witness([(7, 9, 11)], num_wires=38), [random.Random(3).getrandbits(64) for _ in range(38)]], dtype=np.uint64)
    out = np.zeros((rows.shape[0], nc), dtype=np.uint64)
    assert lib.gl_gate_eval_rows(ctx.handle, kind, param, rows.ctypes.data, rows.shape[0], out.ctypes.data) == 0
    for r in range(rows.shape[0]):
        want = go.poseidon2_gate_eval(rows[r].tolist()) if kind == 0 else go.u32_arithmetic_eval(rows[r].tolist(), num_ops=param)
        assert out[r].tolist() == want, r


@pytest.mark.gpu
def test_poseidon2_gate_witness_matches_generator(ctx):
    rnd = random.Random(9)
    inp = np.array([[rnd.randrange(P) for _ in range(12)] + [rnd.randrange(2)] for _ in range(64)], dtype=np.uint64)
    inp[5, :12] = np.uint64(P - 1)
    inp[6, :12] = 0
    import plonky25_b200 as g
    out = g.poseidon2_gate_witness(inp, ctx=ctx)
    for r in range(64):
        assert out[r].tolist() == go.poseidon2_gate_witness(inp[r, :12].tolist(), int(inp[r, 12])), r
    # and the generated rows satisfy the gate on the device
    assert not g.evaluate_gate_constraints(g.GATE_POSEIDON2, 0, out, ctx=ctx).any()


@pytest.mark.gpu
@pytest.mark.parametrize("log_n,n_ch", [(5, 2), (9, 2), (7, 1)])
def test_quotient_accumulation_over_resident_lde_rows(ctx, log_n, n_ch):
    """commit a wires batch, then accumulate both gates' alpha-combined constraints over its R = 8N LDE rows (with a filter column for
    the second gate): every row equals reduce_with_powers of the oracle's constraint values of that leaf row."""
    import plonky25_b200 as g
    lib, r = ctx.lib, 3
    n = 1 << log_n
    wires = g.PolynomialBatch.from_values(list(splitmix_columns(70 + log_n, 135, n)), r, False, 0, ctx=ctx)
    consts = g.PolynomialBatch.from_values(list(splitmix_columns(71 + log_n, 4, n)), r, False, 0, ctx=ctx)
    R = n << r
    alphas = np.array([0x123456789ABCDEF % P, P - 2, 5, 0][:n_ch], dtype=np.uint64)
    q = ctypes.c_uint64()
    assert lib.gl_quotient_begin(ctx.handle, wires.merkle_tree._h, n_ch, ctypes.byref(q)) == 0
    assert lib.gl_quotient_add_gate(ctx.handle, q.value, 0, 0, alphas.ctypes.data, 0, 0, 0) == 0
    assert lib.gl_quotient_add_gate(ctx.handle, q.value, 1, 3, alphas.ctypes.data, 123, consts.merkle_tree._h, 2) == 0
    out = np.zeros((n_ch, R), dtype=np.uint64)
    assert lib.gl_quotient_read(ctx.handle, q.value, out.ctypes.data) == 0
    assert lib.gl_quotient_end(ctx.handle, q.value) == 0
    rnd = random.Random(log_n)
    rows = sorted(set([0, 1, R - 1] + [rnd.randrange(R) for _ in range(24)]))
    lw, lc = wires.merkle_tree.open_batch(rows)[0], consts.merkle_tree.open_batch(rows)[0]
    for j, row in enumerate(rows):
        c0 = go.poseidon2_gate_eval(lw[j].tolist())
        c1 = go.u32_arithmetic_eval(lw[j].tolist()[:114], num_ops=3)
        f = int(lc[j][2])
        for k in range(n_ch):
            a = int(alphas[k])
            want = (go.reduce_with_powers(c0, a) + f * go.reduce_with_powers(c1, a, start_power=123)) % P
            assert int(out[k, row]) == want, (row, k)
    with pytest.raises(Exception):
        assert lib.gl_quotient_add_gate(ctx.handle, 12345, 0, 0, alphas.ctypes.data, 0, 0, 0) == 0
    wires.merkle_tree.free(); consts.merkle_tree.free()


@pytest.mark.gpu
@pytest.mark.parametrize("log_n,n_routed,degree,n_ch", [(4, 80, 8, 2), (6, 80, 8, 2), (5, 13, 4, 1), (3, 8, 8, 3)])
def test_partial_products_and_zs_match_oracle(ctx, log_n, n_routed, degree, n_ch):
    """gl_partial_products against the restated wires_permutation_partial_products_and_zs; and the argument's own identity: when the
    wires satisfy a copy permutation sigma, the running product closes (Z(x_0) = 1 and the product over all rows is 1 again)."""
    rnd = random.Random(100 + log_n)
    n = 1 << log_n
    w = pow(1753635133440165772, 1 << (32 - log_n), P)
    xs = [pow(w, i, P) for i in range(n)]
    k_is = [pow(7, j, P) for j in range(n_routed)]
    # a copy permutation on the (column, row) grid made of a few cycles; wires constant on every cycle
    cells = [(j, i) for j in range(n_routed) for i in range(n)]
    perm = list(range(len(cells)))
    rnd.shuffle(perm)
    sigma_of = {}
    wires = [[0] * n for _ in range(n_routed)]
    cycle_len = 5
    for c0 in range(0, len(perm), cycle_len):
        cyc = [cells[t] for t in perm[c0:c0 + cycle_len]]
        v = rnd.randrange(P)
        for a, b in zip(cyc, cyc[1:] + cyc[:1]):
            sigma_of[a] = b
            wires[a[0]][a[1]] = v
    sigmas = [[k_is[sigma_of[(j, i)][0]] * xs[sigma_of[(j, i)][1]] % P for i in range(n)] for j in range(n_routed)]
    betas = [rnd.randrange(P) for _ in range(n_ch)]
    gammas = [rnd.randrange(P) for _ in range(n_ch)]
    want = go.partial_products_and_zs(wires, sigmas, k_is, betas, gammas, degree, log_n)
    n_chunks = -(-n_routed // degree)
    W, S = np.array(wires, dtype=np.uint64), np.array(sigmas, dtype=np.uint64)
    W[0, 0] += np.uint64(P) if int(W[0, 0]) < 2**32 - 1 else np.uint64(0)     # a non-canonical input word
    import plonky25_b200 as g
    out = g.partial_products_and_zs(list(W), list(S), k_is, betas, gammas, degree, ctx=ctx)
    assert out.shape == (n_ch * n_chunks, n)
    assert out.tolist() == want
    # the permutation argument closes: Z(x_0) = 1 and Z(x_{n-1}) * (last row's chunk products) = 1
    for c in range(n_ch):
        assert int(out[c, 0]) == 1
        last = int(out[c, n - 1])
        acc = last
        for j in range(n_routed):
            num = (wires[j][n - 1] + betas[c] * k_is[j] % P * xs[n - 1] + gammas[c]) % P
            den = (wires[j][n - 1] + betas[c] * sigmas[j][n - 1] + gammas[c]) % P
            acc = acc * num % P * pow(den, P - 2, P) % P
        assert acc == 1


@pytest.mark.gpu
@pytest.mark.parametrize("log_n", [4, 8])
def test_quotient_commit_tail(ctx, oc, log_n):
    """gl_quotient_commit: acc / Z_H on the coset -> coset iFFT -> 2^r chunks of N coefficients -> from_coeffs commit.  Checked (a) against
    the oracle's ifft + commit on the same accumulator values and (b) by the defining identity at sampled LDE points:
    Z_H(x) * sum_c x^(cN) chunk_c(x) == acc(x)."""
    import plonky25_b200 as g
    lib, r, h, n_ch = ctx.lib, 3, 2, 2
    n, R, bits = 1 << log_n, 1 << (log_n + 3), log_n + 3
    wires = g.PolynomialBatch.from_values(list(splitmix_columns(90 + log_n, 135, n)), r, False, h, ctx=ctx)
    alphas = np.array([11, 0xABCDEF0123456789 % P], dtype=np.uint64)
    quot = g.Quotient(wires, n_ch, ctx=ctx)                     # the Python mirror of the reference-facing interface
    quot.add_gate(g.GATE_POSEIDON2, 0, alphas)
    acc = quot.values()
    batch = quot.commit(h)
    quot.free()
    cap = batch.merkle_tree.cap.hashes
    chunks = batch.polynomials                                  # [16][N] coefficients
    # (a) oracle: divide by Z_H, interpolate on the coset, split
    rev = np.array([int(format(i, "0%db" % bits)[::-1], 2) for i in range(R)])
    w_r = pow(1753635133440165772, 1 << (32 - 3), P)
    zh_inv = [pow((pow(7, n, P) * pow(w_r, j, P) - 1) % P, P - 2, P) for j in range(8)]
    inv7 = pow(7, P - 2, P)
    want = []
    for k in range(n_ch):
        vals = [int(acc[k, rev[i]]) * zh_inv[i % 8] % P for i in range(R)]
        co = [int(c) * pow(inv7, j, P) % P for j, c in enumerate(oc.ifft(np.array(vals, dtype=np.uint64)))]
        want += [co[c * n:(c + 1) * n] for c in range(8)]
    assert chunks.tolist() == want
    ref = oc.commit(np.array(want, dtype=np.uint64), r, h, is_coeffs=True, want=())
    assert np.array_equal(cap, ref["cap"])
    # (b) identity at sampled points of the LDE coset
    w_R = pow(1753635133440165772, 1 << (32 - bits), P)
    for i in (0, 1, R // 3, R - 1):
        x = 7 * pow(w_R, i, P) % P
        zh = (pow(x, n, P) - 1) % P
        for k in range(n_ch):
            tot = 0
            for c in reversed(range(8)):
                ev = 0
                for cf in reversed(chunks[k * 8 + c].tolist()):
                    ev = (ev * x + cf) % P
                tot = (tot * pow(x, n, P) + ev) % P
            assert tot * zh % P == int(acc[k, rev[i]])
    batch.merkle_tree.free(); wires.merkle_tree.free()


def _eval_poly(coeffs, x):
    acc = 0
    for c in reversed(coeffs):
        acc = (acc * x + int(c)) % P
    return acc


@pytest.mark.gpu
@pytest.mark.parametrize("log_n,n_routed,degree", [(4, 80, 8), (5, 12, 4)])
def test_permutation_argument_end_to_end(ctx, log_n, n_routed, degree):
    """wires with a copy permutation -> gl_partial_products (Z, partial products) -> three commits -> gl_quotient_add_permutation over the
    LDE rows (+ a gate, to exercise the offset) -> gl_quotient_commit.  Checked (a) row by row against the restated vanishing terms and
    (b) the way the VERIFIER checks a proof: at a random point zeta outside the domain, Z_H(zeta) * sum_c zeta^(cN) t_c(zeta) must equal
    the alpha-combination of the terms computed from the opened polynomial values — which only holds if Z really closes the argument."""
    import plonky25_b200 as g
    rnd = random.Random(77 + log_n)
    n, r, n_ch, n_wires = 1 << log_n, 3, 2, 135
    w_n = pow(1753635133440165772, 1 << (32 - log_n), P)
    xs = [pow(w_n, i, P) for i in range(n)]
    k_is = [pow(7, j, P) for j in range(n_routed)]
    cells = [(j, i) for j in range(n_routed) for i in range(n)]
    perm = list(range(len(cells)))
    rnd.shuffle(perm)
    sigma_of, wires = {}, [[rnd.randrange(P) for _ in range(n)] for _ in range(n_wires)]
    for c0 in range(0, len(perm), 3):
        cyc = [cells[t] for t in perm[c0:c0 + 3]]
        v = rnd.randrange(P)
        for a_, b_ in zip(cyc, cyc[1:] + cyc[:1]):
            sigma_of[a_] = b_
            wires[a_[0]][a_[1]] = v
    sigmas = [[k_is[sigma_of[(j, i)][0]] * xs[sigma_of[(j, i)][1]] % P for i in range(n)] for j in range(n_routed)]
    betas, gammas = [rnd.randrange(P) for _ in range(n_ch)], [rnd.randrange(P) for _ in range(n_ch)]
    alphas = [rnd.randrange(P) for _ in range(n_ch)]
    W = np.array(wires, dtype=np.uint64)
    S = np.array(sigmas, dtype=np.uint64)
    zs = g.partial_products_and_zs(list(W[:n_routed]), list(S), k_is, betas, gammas, degree, ctx=ctx)
    n_chunks = -(-n_routed // degree)
    consts = np.array([[rnd.randrange(P) for _ in range(n)] for _ in range(3)], dtype=np.uint64)
    wires_b = g.PolynomialBatch.from_values(list(W), r, False, 2, ctx=ctx)
    sig_b = g.PolynomialBatch.from_values(list(consts) + list(S), r, False, 2, ctx=ctx)       # sigma polynomials at columns [3, 3 + n_routed)
    zs_b = g.PolynomialBatch.from_values(list(zs), r, False, 2, ctx=ctx)
    quot = g.Quotient(wires_b, n_ch, ctx=ctx)
    al = np.array(alphas, dtype=np.uint64)
    quot.add_permutation(sig_b, 3, zs_b, n_routed, degree, k_is, betas, gammas, alphas)
    n_terms = n_ch * (1 + n_chunks)
    acc = quot.values()
    # (a) sampled LDE rows against the restated terms
    bits, R = log_n + r, n << r
    w_R = pow(1753635133440165772, 1 << (32 - bits), P)
    rev = lambda i: int(format(i, "0%db" % bits)[::-1], 2)
    for row in [0, 1, R - 1] + [rnd.randrange(R) for _ in range(5)]:
        idx = rev(row)
        row_next = rev((idx + (1 << r)) % R)
        x = 7 * pow(w_R, idx, P) % P
        lw, ls = wires_b.merkle_tree.get(row).tolist(), sig_b.merkle_tree.get(row).tolist()
        lz, lzn = zs_b.merkle_tree.get(row).tolist(), zs_b.merkle_tree.get(row_next).tolist()
        terms = go.vanishing_permutation_terms(lw[:n_routed], ls[3:3 + n_routed], lz, lzn, x, k_is, betas, gammas, degree, log_n)
        assert len(terms) == n_terms
        for c in range(n_ch):
            assert int(acc[c, row]) == go.reduce_with_powers(terms, alphas[c]), (row, c)
    # a gate on top, at the offset the terms above leave
    quot.add_gate(g.GATE_U32_ARITHMETIC, 3, al, constraint_offset=n_terms)
    tq = quot.commit(2)
    quot.free()
    # (b) the verifier's identity at a random zeta
    zeta = rnd.randrange(2, P)
    gz = zeta * w_n % P
    cw, cs, cz = wires_b.polynomials, sig_b.polynomials, zs_b.polynomials
    ew = [_eval_poly(cw[j], zeta) for j in range(n_wires)]
    es = [_eval_poly(cs[3 + j], zeta) for j in range(n_routed)]
    ez = [_eval_poly(cz[j], zeta) for j in range(n_ch * n_chunks)]
    ezn = [_eval_poly(cz[j], gz) for j in range(n_ch * n_chunks)]
    terms = go.vanishing_permutation_terms(ew[:n_routed], es, ez, ezn, zeta, k_is, betas, gammas, degree, log_n)
    z_h = (pow(zeta, n, P) - 1) % P
    # (the u32 gate's constraints do not vanish on H for these random wires, so the identity is checked on a second accumulator that
    # holds the permutation terms alone; `tq` above only exercises the gate offset and the commit)
    assert tq.polynomials.shape == (n_ch * 8, n)
    quot2 = g.Quotient(wires_b, n_ch, ctx=ctx)
    quot2.add_permutation(sig_b, 3, zs_b, n_routed, degree, k_is, betas, gammas, alphas)
    t2 = quot2.commit(2)
    quot2.free()
    ch2 = t2.polynomials
    perm_terms = terms[:n_terms]
    for c in range(n_ch):
        t_zeta = 0
        for ch in reversed(range(8)):
            t_zeta = (t_zeta * pow(zeta, n, P) + _eval_poly(ch2[c * 8 + ch], zeta)) % P
        assert z_h * t_zeta % P == go.reduce_with_powers(perm_terms, alphas[c]), "Z_H(zeta) t(zeta) != vanishing(zeta): the argument does not close"
    for b_ in (wires_b, sig_b, zs_b, tq, t2):
        b_.merkle_tree.free()
