"""Selector filters and gate constants read from the constants/sigmas commit (gl_quotient_add_gates), and plonky2's core gates (NoopGate,
ConstantGate, PublicInputGate, ArithmeticGate, BaseSumGate).  CPU: the restated oracle's own consistency, compute_filter on H, and a small
circuit whose filtered constraint sum vanishes on H.  GPU: the gates bit for bit against the oracle, gl_quotient_add_gates row by row, the
verifier's identity Z_H(zeta) t(zeta) = vanishing(zeta) for whole circuits (and its failure when the witness, the selector groups or a
committed constant is wrong), every error path, and the C++ mirror on the real library."""
import os
import random
import subprocess

import numpy as np
import pytest

import gates_oracle as go
import plonky2_gates_oracle as pgo

P = pgo.P
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W32 = 1753635133440165772   # 2^32nd root of unity
N_ROUTED, N_WIRES, DEGREE = 80, 135, 8

POSEIDON2, U32_ARITH = 0, 1
BASE_SUM_2 = 63 | 2 << 8            # split_le's BaseSumGate<2> (63 limbs)
BASE_SUM_4 = 32 | 4 << 8
# the wrapper circuit's gate list in miniature: [Poseidon2] [U32Arithmetic(3), Arithmetic(20), Constant(2), PublicInput] [BaseSum<2>, Noop]
CIRCUIT_GATES = [(POSEIDON2, 0), (U32_ARITH, 3), (pgo.ARITHMETIC, 20), (pgo.CONSTANT, 2), (pgo.PUBLIC_INPUT, 0), (pgo.BASE_SUM, BASE_SUM_2),
                 (pgo.NOOP, 0)]
CIRCUIT_GROUPS = [(0, 1), (1, 5), (5, 7)]          # degree + (group size - 1) + 1 <= 8 for every gate
CIRCUIT_SELECTORS = [0, 1, 1, 1, 1, 2, 2]
NUM_GATE_CONSTANTS = 2


def constraints(kind, param, w, k, pi):
    """eval_unfiltered of any gate the tests use: the reference's own (gates_oracle.py) and plonky2's core gates (plonky2_gates_oracle.py)"""
    if kind == POSEIDON2:
        return go.poseidon2_gate_eval(w)
    if kind == U32_ARITH:
        return go.u32_arithmetic_eval(w, num_ops=param)
    return pgo.gate_eval(kind, param, w, k, pi)


def _core_case(kind, param, rnd):
    """(valid wires, constants, pi_hash) of one row of a core gate"""
    pi = [rnd.randrange(P) for _ in range(4)]
    if kind == pgo.CONSTANT:
        k = [rnd.randrange(P) for _ in range(param)]
        return pgo.constant_witness(k), k, pi
    if kind == pgo.PUBLIC_INPUT:
        return pgo.public_input_witness(pi), [], pi
    if kind == pgo.ARITHMETIC:
        k = [rnd.randrange(P), rnd.randrange(P)]
        return pgo.arithmetic_witness([(rnd.randrange(P), rnd.randrange(P), rnd.randrange(P)) for _ in range(param)], *k), k, pi
    if kind == pgo.BASE_SUM:
        n, b = param & 0xFF, param >> 8
        return pgo.base_sum_witness(rnd.randrange(b ** n), n, b), [], pi
    return [], [], pi


# ------------------------------------------------------------------------------------------------ a circuit
def build_circuit(log_n, seed, poseidon2_witness):
    """A circuit of N rows with CIRCUIT_GATES, valid witnesses and the identity copy permutation.  Returns the wire columns [135][N], the
    constants/sigmas columns in plonky2's order (selectors, gate constants, sigmas) and everything the quotient needs."""
    rnd = random.Random(seed)
    n = 1 << log_n
    m = n // 16
    counts = {0: 2 * m, 1: 2 * m, 2: 3 * m, 3: 2 * m, 4: 1, 5: 2 * m}
    row_gate = [g for g, c in counts.items() for _ in range(c)]
    row_gate += [6] * (n - len(row_gate))
    rnd.shuffle(row_gate)
    p2_rows = [r for r in range(n) if row_gate[r] == 0]
    p2 = poseidon2_witness([[rnd.randrange(P) for _ in range(12)] + [rnd.randrange(2)] for _ in p2_rows])
    wires = [[rnd.randrange(P) for _ in range(N_WIRES)] for _ in range(n)]     # unused wires of a row stay random
    gconsts = [[0] * NUM_GATE_CONSTANTS for _ in range(n)]
    pi = [rnd.randrange(P) for _ in range(4)]
    for r in range(n):
        kind, param = CIRCUIT_GATES[row_gate[r]]
        if kind == POSEIDON2:
            w, k = list(p2[p2_rows.index(r)]), []
        elif kind == U32_ARITH:
            w, k = go.u32_arithmetic_witness([(rnd.getrandbits(32), rnd.getrandbits(32), rnd.getrandbits(32)) for _ in range(3)]), []
        elif kind == pgo.PUBLIC_INPUT:
            w, k = pgo.public_input_witness(pi), []
        else:
            w, k, _ = _core_case(kind, param, rnd)
        wires[r][:len(w)] = [int(x) for x in w]
        gconsts[r][:len(k)] = k
    nsel = len(CIRCUIT_GROUPS)
    sel_cols = [[row_gate[r] if CIRCUIT_SELECTORS[row_gate[r]] == j else pgo.UNUSED_SELECTOR for r in range(n)] for j in range(nsel)]
    w_n = pow(W32, 1 << (32 - log_n), P)
    xs = [pow(w_n, i, P) for i in range(n)]
    k_is = [pow(7, j, P) for j in range(N_ROUTED)]
    sigmas = [[k_is[j] * xs[i] % P for i in range(n)] for j in range(N_ROUTED)]     # identity copy permutation: Z = 1
    const_cols = sel_cols + [[gconsts[r][j] for r in range(n)] for j in range(NUM_GATE_CONSTANTS)]
    return {"n": n, "log_n": log_n, "row_gate": row_gate, "wires": np.array(wires, dtype=np.uint64).T.copy(),
            "consts": np.array(const_cols, dtype=np.uint64), "sigmas": np.array(sigmas, dtype=np.uint64), "pi": pi, "k_is": k_is,
            "num_constants": nsel + NUM_GATE_CONSTANTS}


def eval_filtered(gates, selectors, groups, consts_row, wires_row, pi, num_lookup_selectors=0):
    return pgo.eval_filtered(gates, selectors, groups, consts_row, wires_row, pi, num_lookup_selectors, constraints)


# ------------------------------------------------------------------------------------------------ CPU
def test_core_gate_oracle_consistency():
    """witness rows satisfy every constraint; a tampered wire, constant or hash word breaks one"""
    rnd = random.Random(3)
    for kind, param in [(pgo.CONSTANT, 1), (pgo.CONSTANT, 8), (pgo.PUBLIC_INPUT, 0), (pgo.ARITHMETIC, 20), (pgo.ARITHMETIC, 1),
                        (pgo.BASE_SUM, BASE_SUM_2), (pgo.BASE_SUM, BASE_SUM_4), (pgo.BASE_SUM, 1 | 16 << 8)]:
        nw, nc, nk = pgo.shape(kind, param)
        for _ in range(3):
            w, k, pi = _core_case(kind, param, rnd)
            assert len(w) == nw and len(k) == nk
            c = pgo.gate_eval(kind, param, w, k, pi)
            assert len(c) == nc and not any(c), (kind, param)
            i = rnd.randrange(nw)
            t = list(w)
            t[i] = (t[i] + 1) % P
            assert any(pgo.gate_eval(kind, param, t, k, pi)), (kind, param, i)
            if nk:
                t = list(k)
                t[rnd.randrange(nk)] ^= 1
                assert any(pgo.gate_eval(kind, param, w, t, pi)), (kind, param)
            if kind == pgo.PUBLIC_INPUT:
                t = list(pi)
                t[rnd.randrange(4)] ^= 1
                assert any(pgo.gate_eval(kind, param, w, k, t))
    assert pgo.shape(pgo.NOOP, 0) == (0, 0, 0) and pgo.gate_eval(pgo.NOOP, 0, []) == []
    with pytest.raises(AssertionError):
        pgo.base_sum_witness(4, 2, 2)


def test_compute_filter_on_H():
    for group in [(0, 1), (2, 7), (5, 6), (0, 9)]:
        for many in (False, True):
            for i in range(*group):
                assert pgo.compute_filter(i, group, i, many) != 0
                for j in range(*group):
                    if j != i:
                        assert pgo.compute_filter(i, group, j, many) == 0, (group, i, j)
                assert (pgo.compute_filter(i, group, pgo.UNUSED_SELECTOR, many) == 0) == many
    # by definition: prod over the other indices, then the unused selector
    assert pgo.compute_filter(1, (0, 3), 10, True) == (0 - 10) * (2 - 10) * (pgo.UNUSED_SELECTOR - 10) % P


@pytest.mark.parametrize("log_n", [4, 5, 6])
def test_small_circuit_filtered_constraints_vanish_on_H(log_n):
    c = build_circuit(log_n, 10 + log_n, lambda ins: [go.poseidon2_gate_witness(x[:12], x[12]) for x in ins])
    n = c["n"]

    def at(r, wires):
        return eval_filtered(CIRCUIT_GATES, CIRCUIT_SELECTORS, CIRCUIT_GROUPS, c["consts"][:, r].tolist(), wires[:, r].tolist(), c["pi"])
    for r in range(n):
        assert not any(at(r, c["wires"])), r
    rnd = random.Random(log_n)
    for _ in range(3):
        r = rnd.randrange(n)
        kind, param = CIRCUIT_GATES[c["row_gate"][r]]
        nw = go.POSEIDON2_NUM_WIRES if kind == POSEIDON2 else 38 * 3 if kind == U32_ARITH else pgo.shape(kind, param)[0]
        if nw == 0:
            continue
        t = c["wires"].copy()
        t[rnd.randrange(nw), r] = (int(t[0, r]) + 12345) % P
        assert any(at(r, t)), (r, kind)


# ------------------------------------------------------------------------------------------------ GPU
def _eval_rows(ctx, kind, param, rows, consts, pi):
    lib = ctx.lib
    nc = lib.gl_gate_num_constraints(kind, param)
    out = np.zeros((rows.shape[0], nc), dtype=np.uint64)
    pi_a = np.array(pi, dtype=np.uint64)
    k = consts if consts.size else None
    assert lib.gl_gate_eval_rows_with_constants(ctx.handle, kind, param, rows.ctypes.data, None if k is None else k.ctypes.data,
                                                pi_a.ctypes.data, rows.shape[0], out.ctypes.data) == 0, lib.gl_ctx_last_error(ctx.handle)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("kind,param", [(pgo.NOOP, 0), (pgo.CONSTANT, 2), (pgo.CONSTANT, 8), (pgo.PUBLIC_INPUT, 0), (pgo.ARITHMETIC, 20),
                                        (pgo.ARITHMETIC, 33), (pgo.BASE_SUM, BASE_SUM_2), (pgo.BASE_SUM, BASE_SUM_4), (pgo.BASE_SUM, 7 | 16 << 8)])
def test_core_gates_match_oracle(ctx, kind, param):
    """valid, tampered and arbitrary rows (non-canonical words included) against the oracle, bit for bit"""
    import plonky25_b200 as g
    lib, rnd = ctx.lib, random.Random(100 * kind + param)
    nw, nc, nk = pgo.shape(kind, param)
    assert (lib.gl_gate_num_wires(kind, param), lib.gl_gate_num_constraints(kind, param), lib.gl_gate_num_constants(kind, param)) == (nw, nc, nk)
    pi = [rnd.getrandbits(64) for _ in range(4)]
    rows, consts = [], []
    for r in range(60):
        w, k, _ = _core_case(kind, param, rnd)
        if kind == pgo.PUBLIC_INPUT:
            w = [x % P for x in pi]
        if r % 3 == 1 and nw:
            w[rnd.randrange(nw)] = rnd.randrange(P)
        if r % 3 == 2:
            w, k = [rnd.getrandbits(64) for _ in range(nw)], [rnd.getrandbits(64) for _ in range(nk)]
        rows.append(w)
        consts.append(k)
    rows = np.array(rows, dtype=np.uint64).reshape(60, nw)
    consts = np.array(consts, dtype=np.uint64).reshape(60, nk)
    out = _eval_rows(ctx, kind, param, rows, consts, pi)
    for r in range(60):
        assert out[r].tolist() == pgo.gate_eval(kind, param, rows[r].tolist(), consts[r].tolist(), pi), r
    if nk == 0 and kind != pgo.PUBLIC_INPUT:      # the old entry point takes the gates that read neither
        assert np.array_equal(g.evaluate_gate_constraints(kind, param, rows, ctx=ctx), out)
    else:
        assert np.array_equal(g.evaluate_gate_constraints(kind, param, rows, ctx=ctx, constants=consts, public_inputs_hash=pi), out)


def _rows_at(batch, rows):
    return batch.merkle_tree.open_batch(rows)[0]


@pytest.mark.gpu
@pytest.mark.parametrize("groups,selectors,n_lookup,n_ch", [
    ([(0, 2), (2, 5), (5, 8)], [0, 0, 1, 1, 1, 2, 2, 2], 0, 2),
    ([(0, 3), (3, 8)], [0, 0, 0, 1, 1, 1, 1, 1], 1, 4),
    ([(0, 8)], [0] * 8, 0, 1),
    ([(0, 1), (1, 2), (2, 7), (7, 8)], [0, 1, 2, 2, 2, 2, 2, 3], 2, 3)])
def test_add_gates_row_by_row(ctx, groups, selectors, n_lookup, n_ch):
    """random wires and constants/sigmas columns (so the selector values are arbitrary field elements at the LDE points): every sampled
    row of the accumulator is sum_i compute_filter(i, group, s(row)) * reduce_with_powers(c_i(row), alpha_k, offset)"""
    import plonky25_b200 as g
    from oracle_c import splitmix_columns
    gates = [(POSEIDON2, 0), (U32_ARITH, 3), (pgo.ARITHMETIC, 20), (pgo.CONSTANT, 2), (pgo.PUBLIC_INPUT, 0), (pgo.BASE_SUM, BASE_SUM_4),
             (pgo.NOOP, 0), (pgo.CONSTANT, 1)]
    log_n, r = 6, 3
    n, R = 1 << log_n, 1 << (log_n + r)
    nsel = len(groups)
    num_constants = nsel + n_lookup + 2
    wires = g.PolynomialBatch.from_values(list(splitmix_columns(500 + n_ch, N_WIRES, n)), r, False, 1, ctx=ctx)
    cs = g.PolynomialBatch.from_values(list(splitmix_columns(600 + n_ch, num_constants + 7, n)), r, False, 1, ctx=ctx)
    rnd = random.Random(n_ch)
    alphas = [rnd.randrange(P) for _ in range(n_ch)]
    pi = [rnd.getrandbits(64) for _ in range(4)]
    offset = 17
    q = g.Quotient(wires, n_ch, ctx=ctx)
    ms = q.add_gates(gates, g.SelectorsInfo(selectors, groups), cs, num_constants, pi, alphas, constraint_offset=offset,
                     num_lookup_selectors=n_lookup)
    assert ms > 0
    acc = q.values()
    q.free()
    rows = sorted(set([0, 1, R - 1] + [rnd.randrange(R) for _ in range(20)]))
    lw, lc = _rows_at(wires, rows), _rows_at(cs, rows)
    for j, row in enumerate(rows):
        w, k = lw[j].tolist(), lc[j].tolist()
        want = [0] * n_ch
        for i, (kind, param) in enumerate(gates):
            f = pgo.compute_filter(i, groups[selectors[i]], k[selectors[i]], nsel > 1)
            c = constraints(kind, param, w, k[nsel + n_lookup:num_constants], [x % P for x in pi])
            for ch in range(n_ch):
                want[ch] = (want[ch] + f * pgo.reduce_with_powers(c, alphas[ch], offset)) % P
        assert [int(acc[ch, row]) for ch in range(n_ch)] == want, row
    wires.merkle_tree.free(); cs.merkle_tree.free()


def _eval_poly(coeffs, x):
    acc = 0
    for c in reversed(coeffs):
        acc = (acc * x + int(c)) % P
    return acc


def _prove_quotient(g, ctx, c, wires_cols, const_cols, selectors, groups, alphas, betas, gammas, n_ch=2, r=3):
    """commit constants+sigmas, wires and Z/partial products; add_permutation, add_gates at offset n_ch (1 + n_chunks); commit the
    quotient.  Returns the three batches, the quotient batch and the offset."""
    sig = g.PolynomialBatch.from_values(list(const_cols) + list(c["sigmas"]), r, False, 2, ctx=ctx)
    wires = g.PolynomialBatch.from_values(list(wires_cols), r, False, 2, ctx=ctx)
    zs = g.partial_products_and_zs(list(wires_cols[:N_ROUTED]), list(c["sigmas"]), c["k_is"], betas, gammas, DEGREE, ctx=ctx)
    zs_b = g.PolynomialBatch.from_values(list(zs), r, False, 2, ctx=ctx)
    n_chunks = -(-N_ROUTED // DEGREE)
    offset = n_ch * (1 + n_chunks)
    q = g.Quotient(wires, n_ch, ctx=ctx)
    q.add_permutation(sig, c["num_constants"], zs_b, N_ROUTED, DEGREE, c["k_is"], betas, gammas, alphas)
    q.add_gates(CIRCUIT_GATES, g.SelectorsInfo(selectors, groups), sig, c["num_constants"], c["pi"], alphas, constraint_offset=offset)
    t = q.commit(2)
    q.free()
    return sig, wires, zs_b, t, offset


def _identity_holds(c, sig, wires, zs_b, t, offset, selectors, groups, alphas, betas, gammas, zeta, n_ch=2):
    """the verifier's check at zeta: Z_H(zeta) sum_c zeta^(cN) t_c(zeta) == alpha-combination of the permutation terms and eval_filtered,
    all from the committed polynomials opened at zeta"""
    n = c["n"]
    n_chunks = -(-N_ROUTED // DEGREE)
    gz = zeta * pow(W32, 1 << (32 - c["log_n"]), P) % P
    cw, cs, cz, ct = wires.polynomials, sig.polynomials, zs_b.polynomials, t.polynomials
    ew = [_eval_poly(cw[j], zeta) for j in range(N_WIRES)]
    ec = [_eval_poly(cs[j], zeta) for j in range(c["num_constants"])]
    es = [_eval_poly(cs[c["num_constants"] + j], zeta) for j in range(N_ROUTED)]
    ez = [_eval_poly(cz[j], zeta) for j in range(n_ch * n_chunks)]
    ezn = [_eval_poly(cz[j], gz) for j in range(n_ch * n_chunks)]
    perm = go.vanishing_permutation_terms(ew[:N_ROUTED], es, ez, ezn, zeta, c["k_is"], betas, gammas, DEGREE, c["log_n"])
    assert len(perm) == offset
    gate_terms = eval_filtered(CIRCUIT_GATES, selectors, groups, ec, ew, c["pi"])
    z_h = (pow(zeta, n, P) - 1) % P
    ok = True
    for ch in range(n_ch):
        t_zeta = 0
        for k in reversed(range(8)):
            t_zeta = (t_zeta * pow(zeta, n, P) + _eval_poly(ct[ch * 8 + k], zeta)) % P
        ok &= z_h * t_zeta % P == pgo.reduce_with_powers(perm + gate_terms, alphas[ch])
    return ok


@pytest.mark.gpu
@pytest.mark.parametrize("log_n", [5, 6])
def test_verifier_identity_for_a_whole_circuit(ctx, log_n):
    """a circuit of Poseidon2 (gl_poseidon2_gate_witness rows), U32Arithmetic, Arithmetic with per-row constants, Constant, PublicInput,
    BaseSum and Noop rows under three selector groups, the identity copy permutation: the quotient the device commits satisfies
    Z_H(zeta) t(zeta) = vanishing(zeta) at a random zeta — and does not when one wire is tampered, when a gate is given the wrong
    group, or when an ArithmeticGate constant is changed after the witness was made"""
    import plonky25_b200 as g
    c = build_circuit(log_n, 40 + log_n, lambda ins: g.poseidon2_gate_witness(np.array(ins, dtype=np.uint64), ctx=ctx))
    rnd = random.Random(log_n)
    n_ch = 2
    alphas, betas, gammas = ([rnd.randrange(P) for _ in range(n_ch)] for _ in range(3))
    zeta = rnd.randrange(2, P)
    row_gate = c["row_gate"]

    def run(wires_cols, const_cols, selectors=CIRCUIT_SELECTORS, groups=CIRCUIT_GROUPS):
        sig, wires, zs_b, t, offset = _prove_quotient(g, ctx, c, wires_cols, const_cols, selectors, groups, alphas, betas, gammas)
        assert np.array_equal(zs_b.polynomials[:, 1:], np.zeros_like(zs_b.polynomials[:, 1:]))     # identity permutation: Z = 1
        ok = _identity_holds(c, sig, wires, zs_b, t, offset, selectors, groups, alphas, betas, gammas, zeta)
        for b in (sig, wires, zs_b, t):
            b.merkle_tree.free()
        return ok

    assert run(c["wires"], c["consts"]), "Z_H(zeta) t(zeta) != vanishing(zeta) for a valid circuit"
    # one tampered wire (an output of an ArithmeticGate row)
    r_ar = next(r for r in range(c["n"]) if row_gate[r] == 2)
    w = c["wires"].copy()
    w[3, r_ar] = (int(w[3, r_ar]) + 1) % P
    assert not run(w, c["consts"])
    # PublicInputGate moved to the last group: a valid SelectorsInfo that does not match the committed selector columns
    assert not run(c["wires"], c["consts"], [0, 1, 1, 1, 2, 2, 2], [(0, 1), (1, 4), (4, 7)])
    # an ArithmeticGate constant changed after the witness was computed
    k = c["consts"].copy()
    k[len(CIRCUIT_GROUPS), r_ar] = (int(k[len(CIRCUIT_GROUPS), r_ar]) + 5) % P
    assert not run(c["wires"], k)


@pytest.mark.gpu
def test_add_gates_error_paths(ctx):
    import plonky25_b200 as g
    from plonky25_b200 import _lib
    from oracle_c import splitmix_columns
    lib = ctx.lib
    wires = g.PolynomialBatch.from_values(list(splitmix_columns(1, N_WIRES, 16)), 3, False, 0, ctx=ctx)
    cs = g.PolynomialBatch.from_values(list(splitmix_columns(2, 10, 16)), 3, False, 0, ctx=ctx)
    cs_r1 = g.PolynomialBatch.from_values(list(splitmix_columns(3, 10, 16)), 1, False, 0, ctx=ctx)
    cs_32 = g.PolynomialBatch.from_values(list(splitmix_columns(4, 10, 32)), 2, False, 0, ctx=ctx)
    q = g.Quotient(wires, 2, ctx=ctx)
    before = q.values()
    info = g.SelectorsInfo([0, 0, 1], [(0, 2), (2, 3)])
    gates = [(pgo.ARITHMETIC, 20), (pgo.CONSTANT, 2), (pgo.PUBLIC_INPUT, 0)]
    pi, al = [1, 2, 3, 4], [5, 6]

    def refused(match, gates=gates, info=info, batch=cs, num_constants=4, n_lookup=0):
        with pytest.raises(ValueError, match=match):
            q.add_gates(gates, info, batch, num_constants, pi, al, num_lookup_selectors=n_lookup)

    refused("No gates", gates=[], info=g.SelectorsInfo([], [(0, 0)]))
    refused("selector index 2 >= num_selectors 2", info=g.SelectorsInfo([0, 0, 2], [(0, 2), (2, 3)]))
    refused("gate 2 is outside its selector group", info=g.SelectorsInfo([0, 0, 0], [(0, 2), (2, 3)]))
    refused("is not a range of the 3 gates", info=g.SelectorsInfo([0, 0, 1], [(0, 2), (2, 4)]))
    refused("Polynomial degrees inconsistent", batch=cs_r1)
    refused("Polynomial degrees inconsistent", batch=cs_32)
    refused("num_constants 11 exceeds", num_constants=11)
    refused("2 selector columns \\+ 2 gate constants exceed num_constants 3", num_constants=3)
    refused("3 selector columns \\+ 2 gate constants exceed num_constants 4", n_lookup=1)
    refused("unknown gate kind 14", gates=[(14, 0), (pgo.NOOP, 0), (pgo.NOOP, 0)])
    refused("parameter 9 out of range", gates=[(pgo.CONSTANT, 9), (pgo.NOOP, 0), (pgo.NOOP, 0)])
    refused("parameter 1 out of range", gates=[(pgo.NOOP, 1), (pgo.NOOP, 0), (pgo.NOOP, 0)])
    refused("parameter 4353 out of range", gates=[(pgo.BASE_SUM, 1 | 17 << 8), (pgo.NOOP, 0), (pgo.NOOP, 0)])
    # NULL pointers and unknown handles through the raw ABI
    k = np.array([12, 9, 9], dtype=np.int32)
    p = np.array([20, 0, 0], dtype=np.uint32)
    s = np.array([0, 0, 1], dtype=np.uint32)
    gr = np.array([0, 2, 2, 3], dtype=np.uint32)
    h4 = np.array(pi, dtype=np.uint64)
    a2 = np.array(al, dtype=np.uint64)
    args = [ctx.handle, q._h, k.ctypes.data, p.ctypes.data, 3, s.ctypes.data, gr.ctypes.data, 2, 0, cs.merkle_tree._h, 4, h4.ctypes.data,
            a2.ctypes.data, 0]
    assert lib.gl_quotient_add_gates(*args) == _lib.GL_OK
    for pos in (2, 3, 5, 6, 11, 12):
        bad = list(args)
        bad[pos] = None
        assert lib.gl_quotient_add_gates(*bad) == _lib.GL_ERR_INVALID
        assert "NULL pointer" in lib.gl_ctx_last_error(ctx.handle).decode()
    bad = list(args)
    bad[9] = 987654321
    assert lib.gl_quotient_add_gates(*bad) == _lib.GL_ERR_HANDLE
    # the refused calls above launched nothing: only the one valid call changed the accumulator
    q2 = g.Quotient(wires, 2, ctx=ctx)
    q2.add_gates([(pgo.ARITHMETIC, 20), (pgo.NOOP, 0), (pgo.NOOP, 0)], info, cs, 4, pi, al)     # the raw call that succeeded
    assert np.array_equal(q.values(), q2.values()) and not np.array_equal(q.values(), before)
    q2.free()
    # the old entry points refuse the gates that read constants or the public-inputs hash, and take Noop / BaseSum
    for kind, param in [(pgo.CONSTANT, 2), (pgo.ARITHMETIC, 20), (pgo.PUBLIC_INPUT, 0)]:
        with pytest.raises(ValueError, match="gl_quotient_add_gates"):
            q.add_gate(kind, param, al)
        with pytest.raises(ValueError, match="gl_gate_eval_rows_with_constants"):
            g.evaluate_gate_constraints(kind, param, np.zeros((2, pgo.shape(kind, param)[0]), dtype=np.uint64), ctx=ctx)
    assert q.add_gate(pgo.NOOP, 0, al) == 0.0
    acc = q.values()
    q.add_gate(pgo.BASE_SUM, BASE_SUM_2, al, filter=(cs, 3))
    assert not np.array_equal(q.values(), acc)
    assert g.evaluate_gate_constraints(pgo.NOOP, 0, np.zeros((3, 0), dtype=np.uint64), ctx=ctx).shape == (3, 0)
    assert lib.gl_gate_eval_rows_with_constants(ctx.handle, pgo.ARITHMETIC, 20, h4.ctypes.data, None, h4.ctypes.data, 1,
                                                h4.ctypes.data) == _lib.GL_ERR_INVALID
    assert lib.gl_gate_eval_rows_with_constants(ctx.handle, pgo.CONSTANT, 1, h4.ctypes.data, h4.ctypes.data, None, 1,
                                                h4.ctypes.data) == _lib.GL_ERR_INVALID
    assert lib.gl_gate_num_constants(pgo.ARITHMETIC, 20) == 2 and lib.gl_gate_num_constants(pgo.CONSTANT, 9) == -1
    assert lib.gl_gate_num_constants(POSEIDON2, 0) == 0 and lib.gl_gate_num_constants(14, 0) == -1
    q.free()
    for b in (wires, cs, cs_r1, cs_32):
        b.merkle_tree.free()


@pytest.mark.gpu
def test_cpp_quotient_selectors_on_gpu(tmp_path):
    import plonky25_b200 as g
    lib = g.build()
    exe = str(tmp_path / "quotient_selectors_test")
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    env = dict(os.environ)
    env.pop("CC", None); env.pop("CXX", None)
    subprocess.run([cxx, "-std=c++17", "-O2", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "tests", "cpp", "quotient_selectors_test.cpp"), "-o", exe, "-L", os.path.dirname(lib), "-lgl_commit",
                    "-Wl,-rpath," + os.path.dirname(lib), "-pthread"], check=True, env=env)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "ALL OK" in r.stdout, r.stdout[-3000:] + r.stderr[-2000:]
