"""plonky2's PoseidonGate, ExponentiationGate and RandomAccessGate (GATE_POSEIDON / GATE_EXPONENTIATION / GATE_RANDOM_ACCESS) and the
PoseidonGate witness generator on the device.  CPU: the restated oracle's own consistency (PoseidonGate witness outputs are the KAT-pinned
permutation), random_access_params against new_from_config, every refused parameter, and the C++ mirror compiles.  GPU: the gates bit for
bit against the oracle, gl_poseidon_gate_witness against the oracle and the leaf hash's permutation, add_gates row by row, the verifier's
identity for a circuit that hashes its public inputs with PoseidonGate rows (and its failure for each kind of bad witness), every error
path, and the C++ mirror on the real library."""
import os
import random
import subprocess

import numpy as np
import pytest

import gates_oracle as go
import gl_oracle
import plonky2_std_gates_oracle as pgo

P = pgo.P
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W32 = 1753635133440165772   # 2^32nd root of unity
N_ROUTED, N_WIRES, DEGREE = 80, 135, 8
POSEIDON2 = 0
RA_4 = pgo.random_access_params(4)         # 4 copies, 2 extra constants
RA_2 = pgo.random_access_params(2)         # 13 copies, 2 extra constants
NEW_GATES = [(pgo.POSEIDON, 0), (pgo.EXPONENTIATION, 1), (pgo.EXPONENTIATION, 17), (pgo.EXPONENTIATION, 66)] + \
            [(pgo.RANDOM_ACCESS, pgo.random_access_params(b)) for b in range(1, 7)] + \
            [(pgo.RANDOM_ACCESS, 1 | 27 << 8), (pgo.RANDOM_ACCESS, 3 | 2 << 8 | 5 << 16), (pgo.RANDOM_ACCESS, 6 | 1 << 8)]


def _case(kind, param, rnd):
    """(valid wires, gate constants) of one row of a new gate"""
    if kind == pgo.POSEIDON:
        return pgo.poseidon_gate_witness([rnd.randrange(P) for _ in range(12)], rnd.randrange(2)), []
    if kind == pgo.EXPONENTIATION:
        return pgo.exponentiation_witness(rnd.randrange(P), rnd.getrandbits(param), param), []
    bits, copies, extras = pgo.random_access_fields(param)
    k = [rnd.randrange(P) for _ in range(extras)]
    lists = [(rnd.randrange(1 << bits), [rnd.randrange(P) for _ in range(1 << bits)]) for _ in range(copies)]
    return pgo.random_access_witness(lists, k, param), k


def constraints(kind, param, w, k, pi):
    if kind == POSEIDON2:
        return go.poseidon2_gate_eval(w)
    return pgo.gate_eval(kind, param, w, k, pi)


# ------------------------------------------------------------------------------------------------ CPU
def test_poseidon_gate_oracle_witness():
    """witness rows satisfy all 123 constraints for swap 0 and 1; outputs are gl_oracle.poseidon of the (swapped) inputs, hence the
    reference's KAT vectors; tampering any single wire breaks a constraint"""
    import json
    rnd = random.Random(1)
    for swap in (0, 1):
        x = [rnd.randrange(P) for _ in range(12)]
        w = pgo.poseidon_gate_witness(x, swap)
        assert len(w) == 135 and pgo.shape(pgo.POSEIDON) == (135, 123, 0)
        c = pgo.poseidon_gate_eval(w)
        assert len(c) == 123 and not any(c)
        assert w[12:24] == gl_oracle.poseidon(x[4:8] + x[:4] + x[8:] if swap else x)
        for i in range(135):
            t = list(w)
            t[i] = (t[i] + 1 + rnd.randrange(P - 1)) % P
            assert any(pgo.poseidon_gate_eval(t)), (swap, i)
    kat = json.load(open(os.path.join(ROOT, "tests", "golden", "poseidon_kat.json")))["vectors"]
    assert len(kat) == 4
    for v in kat:
        w = pgo.poseidon_gate_witness(v["input"], 0)
        assert w[12:24] == v["output"] and not any(pgo.poseidon_gate_eval(w))


def test_exponentiation_and_random_access_oracle():
    rnd = random.Random(2)
    assert pgo.exponentiation_max_power_bits() == 66
    for n in (1, 17, 66):
        for _ in range(3):
            base, power = rnd.randrange(P), rnd.getrandbits(n)
            w = pgo.exponentiation_witness(base, power, n)
            assert len(w) == pgo.shape(pgo.EXPONENTIATION, n)[0] and w[1 + n] == pow(base, power, P)
            c = pgo.exponentiation_eval(w, n)
            assert len(c) == n + 1 and not any(c)
            t = list(w)
            t[1 + rnd.randrange(n)] ^= 1                       # flipped power bit
            assert any(pgo.exponentiation_eval(t, n))
            t = list(w)
            t[1 + n] = (t[1 + n] + 1) % P                      # wrong output
            assert any(pgo.exponentiation_eval(t, n))
    for bits in range(1, 7):
        param = pgo.random_access_params(bits)
        _, copies, extras = pgo.random_access_fields(param)
        nw, nc, nk = pgo.shape(pgo.RANDOM_ACCESS, param)
        assert nw <= 135 and nk == extras == min(80 - (2 + (1 << bits)) * copies, 2) and nc == (bits + 2) * copies + extras
        for _ in range(3):
            w, k = _case(pgo.RANDOM_ACCESS, param, rnd)
            assert len(w) == nw and not any(pgo.random_access_eval(w, k, param))
            routed = (2 + (1 << bits)) * copies + extras
            c = rnd.randrange(copies)
            t = list(w)
            t[routed + c * bits + rnd.randrange(bits)] ^= 1       # flipped index bit
            assert any(pgo.random_access_eval(t, k, param))
            t = list(w)
            t[(2 + (1 << bits)) * c + 1] = (t[(2 + (1 << bits)) * c + 1] + 1) % P     # wrong claimed element
            assert any(pgo.random_access_eval(t, k, param))
            if extras:
                t = list(k)
                t[rnd.randrange(extras)] ^= 1                      # changed extra constant
                assert any(pgo.random_access_eval(w, t, param))


def test_random_access_params_match_new_from_config():
    import plonky25_b200 as g
    assert pgo.random_access_fields(pgo.random_access_params(4)) == (4, 4, 2)
    assert pgo.random_access_fields(pgo.random_access_params(2)) == (2, 13, 2)
    for bits in range(1, 7):
        for nw, nr, nk in ((135, 80, 2), (135, 80, 4), (100, 60, 0)):
            assert g.random_access_params(bits, nw, nr, nk) == pgo.random_access_params(bits, nw, nr, nk)


def test_shapes_and_refused_params():
    """the library's shape queries equal the oracle's, and every refused parameter is refused (no device needed)"""
    import plonky25_b200 as g
    lib = g._lib.load()
    assert (g.GATE_POSEIDON, g.GATE_EXPONENTIATION, g.GATE_RANDOM_ACCESS) == (pgo.POSEIDON, pgo.EXPONENTIATION, pgo.RANDOM_ACCESS)
    for kind, param in NEW_GATES:
        assert (lib.gl_gate_num_wires(kind, param), lib.gl_gate_num_constraints(kind, param), lib.gl_gate_num_constants(kind, param)) == \
            pgo.shape(kind, param), (kind, param)
        assert g.gate_shape(kind, param) == pgo.shape(kind, param)[:2]
    assert pgo.shape(pgo.RANDOM_ACCESS, 1 | 27 << 8)[1] == 81
    for kind, param in [(14, 0), (18, 0), (pgo.POSEIDON, 1), (pgo.EXPONENTIATION, 0), (pgo.EXPONENTIATION, 67), (pgo.RANDOM_ACCESS, 0 | 1 << 8),
                        (pgo.RANDOM_ACCESS, 7 | 1 << 8), (pgo.RANDOM_ACCESS, 2), (pgo.RANDOM_ACCESS, 1 | 28 << 8),
                        (pgo.RANDOM_ACCESS, 4 | 7 << 8), (pgo.RANDOM_ACCESS, 4 | 4 << 8 | 48 << 16), (pgo.RANDOM_ACCESS, 6 | 2 << 8)]:
        assert lib.gl_gate_num_wires(kind, param) == -1 and lib.gl_gate_num_constants(kind, param) == -1, (kind, param)
        with pytest.raises(ValueError, match="unknown gate kind"):
            g.gate_shape(kind, param)
    assert lib.gl_gate_num_wires(pgo.RANDOM_ACCESS, 4 | 4 << 8 | 47 << 16) == 135 and lib.gl_gate_num_wires(pgo.RANDOM_ACCESS, 4 | 6 << 8) == 132


def test_cpp_mirror_compiles():
    """tests/cpp/std_gates_test.cpp compiles warning-free against include/gl_plonky2.hpp and include/gl_commit.h"""
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    env = dict(os.environ)
    env.pop("CC", None); env.pop("CXX", None)
    subprocess.run([cxx, "-std=c++17", "-Wall", "-Wextra", "-Werror", "-fsyntax-only", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "tests", "cpp", "std_gates_test.cpp")], check=True, env=env)


# ------------------------------------------------------------------------------------------------ GPU
def _eval_rows(ctx, kind, param, rows, consts, pi):
    lib = ctx.lib
    nc = lib.gl_gate_num_constraints(kind, param)
    out = np.zeros((rows.shape[0], nc), dtype=np.uint64)
    pi_a = np.array(pi, dtype=np.uint64)
    assert lib.gl_gate_eval_rows_with_constants(ctx.handle, kind, param, rows.ctypes.data, consts.ctypes.data if consts.size else None,
                                                pi_a.ctypes.data, rows.shape[0], out.ctypes.data) == 0, lib.gl_ctx_last_error(ctx.handle)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("kind,param", NEW_GATES)
def test_new_gates_match_oracle(ctx, kind, param):
    """valid, tampered and arbitrary rows (non-canonical words included) against the oracle, bit for bit"""
    import plonky25_b200 as g
    lib, rnd = ctx.lib, random.Random(kind * 1000003 + param)
    nw, nc, nk = pgo.shape(kind, param)
    assert (lib.gl_gate_num_wires(kind, param), lib.gl_gate_num_constraints(kind, param), lib.gl_gate_num_constants(kind, param)) == (nw, nc, nk)
    pi = [rnd.getrandbits(64) for _ in range(4)]
    rows, consts = [], []
    for r in range(48):
        w, k = _case(kind, param, rnd)
        if r % 3 == 1:
            w[rnd.randrange(nw)] = rnd.randrange(P)
        if r % 3 == 2:
            w, k = [rnd.getrandbits(64) for _ in range(nw)], [rnd.getrandbits(64) for _ in range(nk)]
        if r % 6 == 0:                                      # the same row with non-canonical words (x + p where that fits)
            w = [x + P if x < (1 << 64) - P else x for x in w]
        rows.append(w)
        consts.append(k)
    rows = np.array(rows, dtype=np.uint64).reshape(48, nw)
    consts = np.array(consts, dtype=np.uint64).reshape(48, nk)
    out = _eval_rows(ctx, kind, param, rows, consts, pi)
    for r in range(48):
        want = pgo.gate_eval(kind, param, rows[r].tolist(), consts[r].tolist(), pi)
        assert out[r].tolist() == want, r
        if r % 3 == 0:
            assert not any(want), r
    if nk == 0:
        assert np.array_equal(g.evaluate_gate_constraints(kind, param, rows, ctx=ctx), out)
    assert np.array_equal(g.evaluate_gate_constraints(kind, param, rows, ctx=ctx, constants=consts, public_inputs_hash=pi), out)


@pytest.mark.gpu
def test_poseidon_gate_witness_on_device(ctx):
    """gl_poseidon_gate_witness == the oracle's PoseidonGenerator for 10240 rows (non-canonical inputs and swap words included), and the
    outputs equal Context.poseidon_permute (the leaf hash's permutation) of the swapped inputs"""
    import plonky25_b200 as g
    rnd = random.Random(7)
    n = 10240
    ins = []
    for r in range(n):
        x = [rnd.getrandbits(64) if r % 4 == 3 else rnd.randrange(P) for _ in range(12)]
        swap = rnd.randrange(2)
        ins.append(x + [swap + P if r % 8 == 5 else swap])
    x = np.array(ins, dtype=np.uint64)
    rows = g.poseidon_gate_witness(x, ctx=ctx)
    ms = ctypes_ms(ctx)
    assert rows.shape == (n, 135) and ms > 0
    assert int(rows.max()) < P
    for r in range(n):
        assert rows[r].tolist() == pgo.poseidon_gate_witness(ins[r][:12], ins[r][12] % P), r
    canon = x[:, :12] % np.uint64(P)
    swapped = canon.copy()
    sw = (x[:, 12] % np.uint64(P)) == 1
    swapped[sw, :4], swapped[sw, 4:8] = canon[sw, 4:8], canon[sw, :4]
    assert np.array_equal(ctx.poseidon_permute(swapped), rows[:, 12:24])
    assert g.poseidon_gate_witness(np.zeros((0, 13), dtype=np.uint64), ctx=ctx).shape == (0, 135)
    with pytest.raises(ValueError, match=r"\[n\]\[13\]"):
        g.poseidon_gate_witness(np.zeros((2, 12), dtype=np.uint64), ctx=ctx)


def ctypes_ms(ctx):
    import ctypes
    ms = ctypes.c_float()
    assert ctx.lib.gl_ctx_aux_ms(ctx.handle, ctypes.byref(ms)) == 0
    return ms.value


def _rows_at(batch, rows):
    return batch.merkle_tree.open_batch(rows)[0]


@pytest.mark.gpu
@pytest.mark.parametrize("groups,selectors,n_ch", [
    ([(0, 1), (1, 4), (4, 8)], [0, 1, 1, 1, 2, 2, 2, 2], 2),
    ([(0, 8)], [0] * 8, 1),
    ([(0, 2), (2, 3), (3, 6), (6, 8)], [0, 0, 1, 2, 2, 2, 3, 3], 4)])
def test_add_gates_row_by_row(ctx, groups, selectors, n_ch):
    """the new gates mixed with existing ones into selector groups; random wires and constants/sigmas columns (selector values are
    arbitrary field elements at the LDE points): every sampled accumulator row is the oracle's eval_filtered reduced with alpha_k"""
    import plonky25_b200 as g
    from oracle_c import splitmix_columns
    gates = [(pgo.POSEIDON, 0), (pgo.EXPONENTIATION, 66), (pgo.RANDOM_ACCESS, RA_4), (pgo.ARITHMETIC, 20), (POSEIDON2, 0),
             (pgo.RANDOM_ACCESS, RA_2), (pgo.CONSTANT, 2), (pgo.RANDOM_ACCESS, 3 | 3 << 8)]
    log_n, r = 6, 3
    n, R = 1 << log_n, 1 << (log_n + r)
    nsel = len(groups)
    num_constants = nsel + 2
    wires = g.PolynomialBatch.from_values(list(splitmix_columns(700 + n_ch, N_WIRES, n)), r, False, 1, ctx=ctx)
    cs = g.PolynomialBatch.from_values(list(splitmix_columns(800 + n_ch, num_constants + 5, n)), r, False, 1, ctx=ctx)
    rnd = random.Random(n_ch)
    alphas = [rnd.randrange(P) for _ in range(n_ch)]
    pi = [rnd.getrandbits(64) for _ in range(4)]
    offset = 9
    q = g.Quotient(wires, n_ch, ctx=ctx)
    assert q.add_gates(gates, g.SelectorsInfo(selectors, groups), cs, num_constants, pi, alphas, constraint_offset=offset) > 0
    acc = q.values()
    q.free()
    rows = sorted(set([0, 1, R - 1] + [rnd.randrange(R) for _ in range(16)]))
    lw, lc = _rows_at(wires, rows), _rows_at(cs, rows)
    for j, row in enumerate(rows):
        w, k = lw[j].tolist(), lc[j].tolist()
        want = [0] * n_ch
        for i, (kind, param) in enumerate(gates):
            f = pgo.compute_filter(i, groups[selectors[i]], k[selectors[i]], nsel > 1)
            c = constraints(kind, param, w, k[nsel:num_constants], [x % P for x in pi])
            for ch in range(n_ch):
                want[ch] = (want[ch] + f * pgo.reduce_with_powers(c, alphas[ch], offset)) % P
        assert [int(acc[ch, row]) for ch in range(n_ch)] == want, row
    wires.merkle_tree.free(); cs.merkle_tree.free()


# ------------------------------------------------------------------------------------------------ a circuit that hashes its public inputs
# [Poseidon] [Exponentiation(66), RandomAccess(bits 2), Constant(2), PublicInput] [RandomAccess(bits 4), Arithmetic(20), Noop]
# degree + group size <= 8 in every group: 7 + 1, 4 + 4, 5 + 3
CIRCUIT_GATES = [(pgo.POSEIDON, 0), (pgo.EXPONENTIATION, 66), (pgo.RANDOM_ACCESS, RA_2), (pgo.CONSTANT, 2), (pgo.PUBLIC_INPUT, 0),
                 (pgo.RANDOM_ACCESS, RA_4), (pgo.ARITHMETIC, 20), (pgo.NOOP, 0)]
CIRCUIT_GROUPS = [(0, 1), (1, 5), (5, 8)]
CIRCUIT_SELECTORS = [0, 1, 1, 1, 1, 2, 2, 2]
NUM_GATE_CONSTANTS = 2


def build_hashing_circuit(log_n, seed, public_inputs, poseidon_witness):
    """N rows: a chain of PoseidonGate rows absorbs `public_inputs` as hash_n_to_hash_no_pad does (each chunk overwrites lanes
    [0, len), the other lanes are copied from the previous row's outputs, the first row's from a ConstantGate zero, every swap wire is
    copied from that zero); the last row's outputs 0..3 are copied to the PublicInputGate row.  Exponentiation, RandomAccess (with
    per-row extra constants), Arithmetic and Constant rows fill the rest; Noop rows are random.  The copy permutation is made of those
    cycles (sigma = identity elsewhere)."""
    rnd = random.Random(seed)
    n = 1 << log_n
    chunks = [public_inputs[i:i + 8] for i in range(0, len(public_inputs), 8)]
    row_gate = [0] * len(chunks) + [3, 4] + [1, 1, 2, 2, 5, 5, 6, 6, 3]
    row_gate += [7] * (n - len(row_gate))
    order = list(range(n))
    rnd.shuffle(order)                                   # row r of the circuit holds entry order[r] of row_gate
    row_of = {}                                          # entry index -> row
    for r, e in enumerate(order):
        row_of[e] = r
    gate_at = [row_gate[order[r]] for r in range(n)]
    chain = [row_of[t] for t in range(len(chunks))]
    zero_row, pi_row = row_of[len(chunks)], row_of[len(chunks) + 1]
    wires = [[rnd.randrange(P) for _ in range(N_WIRES)] for _ in range(n)]
    gconsts = [[0] * NUM_GATE_CONSTANTS for _ in range(n)]
    cycles = [[(0, zero_row)]]                           # cells (column, row) holding the value 0
    state = [0] * 12
    for t, chunk in enumerate(chunks):
        state = [c % P for c in chunk] + state[len(chunk):]
        row = poseidon_witness([state + [0]])[0]
        wires[chain[t]][:135] = [int(x) for x in row]
        cycles[0].append((24, chain[t]))
        for i in range(len(chunk), 12):
            if t == 0:
                cycles[0].append((i, chain[0]))
            else:
                cycles.append([(12 + i, chain[t - 1]), (i, chain[t])])
        state = [int(x) for x in row[12:24]]
    cycles += [[(12 + i, chain[-1]), (i, pi_row)] for i in range(4)]
    pi_hash = gl_oracle.hash_no_pad(public_inputs)
    for r in range(n):
        kind, param = CIRCUIT_GATES[gate_at[r]]
        if r in chain or kind == pgo.NOOP:
            continue
        if r == zero_row:
            w, k = [0, 0], [0, 0]
        elif kind == pgo.PUBLIC_INPUT:
            w, k = [int(x) for x in wires[chain[-1]][12:16]], []
        elif kind == pgo.CONSTANT:
            k = [rnd.randrange(P) for _ in range(2)]
            w = pgo.constant_witness(k)
        elif kind == pgo.ARITHMETIC:
            k = [rnd.randrange(P), rnd.randrange(P)]
            w = pgo.arithmetic_witness([(rnd.randrange(P), rnd.randrange(P), rnd.randrange(P)) for _ in range(20)], *k)
        else:
            w, k = _case(kind, param, rnd)
        wires[r][:len(w)] = [int(x) for x in w]
        gconsts[r][:len(k)] = k
    w_n = pow(W32, 1 << (32 - log_n), P)
    xs = [pow(w_n, i, P) for i in range(n)]
    k_is = [pow(7, j, P) for j in range(N_ROUTED)]
    sigma_of = {}
    for cyc in cycles:
        for a, b in zip(cyc, cyc[1:] + cyc[:1]):
            assert a[0] < N_ROUTED and a not in sigma_of
            sigma_of[a] = b
    sigmas = [[k_is[sigma_of.get((j, i), (j, i))[0]] * xs[sigma_of.get((j, i), (j, i))[1]] % P for i in range(n)] for j in range(N_ROUTED)]
    nsel = len(CIRCUIT_GROUPS)
    sel_cols = [[gate_at[r] if CIRCUIT_SELECTORS[gate_at[r]] == j else pgo.UNUSED_SELECTOR for r in range(n)] for j in range(nsel)]
    const_cols = sel_cols + [[gconsts[r][j] for r in range(n)] for j in range(NUM_GATE_CONSTANTS)]
    return {"n": n, "log_n": log_n, "gate_at": gate_at, "chain": chain, "wires": np.array(wires, dtype=np.uint64).T.copy(),
            "consts": np.array(const_cols, dtype=np.uint64), "sigmas": np.array(sigmas, dtype=np.uint64), "pi": pi_hash, "k_is": k_is,
            "num_constants": nsel + NUM_GATE_CONSTANTS}


@pytest.mark.parametrize("log_n", [5, 6])
def test_hashing_circuit_vanishes_on_H(log_n):
    """the circuit built with the oracle's PoseidonGate witness: every row's filtered constraint sum is 0 and every wire of a copy cycle
    holds the same value (so Z closes); the PublicInputGate row holds hash_no_pad of the public inputs"""
    rnd = random.Random(log_n)
    pis = [rnd.randrange(P) for _ in range(20 if log_n == 5 else 37)]
    c = build_hashing_circuit(log_n, 60 + log_n, pis, lambda ins: [pgo.poseidon_gate_witness(x[:12], x[12]) for x in ins])
    n, w, k = c["n"], c["wires"], c["consts"]
    for r in range(n):
        assert not any(pgo.eval_filtered(CIRCUIT_GATES, CIRCUIT_SELECTORS, CIRCUIT_GROUPS, k[:, r].tolist(), w[:, r].tolist(), c["pi"], 0,
                                         constraints)), r
    w_n = pow(W32, 1 << (32 - log_n), P)
    cell = {c["k_is"][j] * pow(w_n, i, P) % P: (j, i) for j in range(N_ROUTED) for i in range(n)}
    moved = 0
    for j in range(N_ROUTED):
        for i in range(n):
            jj, ii = cell[int(c["sigmas"][j, i])]
            assert w[j, i] == w[jj, ii]
            moved += (jj, ii) != (j, i)
    assert moved >= 4 + 12
    pi_row = next(r for r in range(n) if c["gate_at"][r] == 4)
    assert w[:4, pi_row].tolist() == gl_oracle.hash_no_pad(pis)


def _eval_poly(coeffs, x):
    acc = 0
    for c in reversed(coeffs):
        acc = (acc * x + int(c)) % P
    return acc


def _identity_holds(g, ctx, c, wires_cols, const_cols, pi, alphas, betas, gammas, zeta, n_ch=2, r=3):
    """commit constants+sigmas, wires and Z / partial products; add_permutation, add_gates at offset n_ch (1 + n_chunks); commit the
    quotient; then the verifier's check Z_H(zeta) sum_c zeta^(cN) t_c(zeta) == the alpha-combination of the permutation terms and
    eval_filtered, all from the committed polynomials opened at zeta"""
    n = c["n"]
    sig = g.PolynomialBatch.from_values(list(const_cols) + list(c["sigmas"]), r, False, 2, ctx=ctx)
    wires = g.PolynomialBatch.from_values(list(wires_cols), r, False, 2, ctx=ctx)
    zs = g.partial_products_and_zs(list(wires_cols[:N_ROUTED]), list(c["sigmas"]), c["k_is"], betas, gammas, DEGREE, ctx=ctx)
    zs_b = g.PolynomialBatch.from_values(list(zs), r, False, 2, ctx=ctx)
    n_chunks = -(-N_ROUTED // DEGREE)
    offset = n_ch * (1 + n_chunks)
    q = g.Quotient(wires, n_ch, ctx=ctx)
    q.add_permutation(sig, c["num_constants"], zs_b, N_ROUTED, DEGREE, c["k_is"], betas, gammas, alphas)
    q.add_gates(CIRCUIT_GATES, g.SelectorsInfo(CIRCUIT_SELECTORS, CIRCUIT_GROUPS), sig, c["num_constants"], pi, alphas, constraint_offset=offset)
    t = q.commit(2)
    q.free()
    gz = zeta * pow(W32, 1 << (32 - c["log_n"]), P) % P
    cw, cs, cz, ct = wires.polynomials, sig.polynomials, zs_b.polynomials, t.polynomials
    ew = [_eval_poly(cw[j], zeta) for j in range(N_WIRES)]
    ec = [_eval_poly(cs[j], zeta) for j in range(c["num_constants"])]
    es = [_eval_poly(cs[c["num_constants"] + j], zeta) for j in range(N_ROUTED)]
    ez = [_eval_poly(cz[j], zeta) for j in range(n_ch * n_chunks)]
    ezn = [_eval_poly(cz[j], gz) for j in range(n_ch * n_chunks)]
    perm = go.vanishing_permutation_terms(ew[:N_ROUTED], es, ez, ezn, zeta, c["k_is"], betas, gammas, DEGREE, c["log_n"])
    gate_terms = pgo.eval_filtered(CIRCUIT_GATES, CIRCUIT_SELECTORS, CIRCUIT_GROUPS, ec, ew, pi, 0, constraints)
    z_h = (pow(zeta, n, P) - 1) % P
    ok = True
    for ch in range(n_ch):
        t_zeta = 0
        for k in reversed(range(8)):
            t_zeta = (t_zeta * pow(zeta, n, P) + _eval_poly(ct[ch * 8 + k], zeta)) % P
        ok &= z_h * t_zeta % P == pgo.reduce_with_powers(perm + gate_terms, alphas[ch])
    for b in (sig, wires, zs_b, t):
        b.merkle_tree.free()
    return ok


@pytest.mark.gpu
@pytest.mark.parametrize("log_n", [5, 6])
def test_verifier_identity_for_a_circuit_hashing_its_public_inputs(ctx, log_n):
    """the quotient the device commits satisfies Z_H(zeta) t(zeta) = vanishing(zeta) at a random zeta for a valid circuit, and does not
    for a tampered partial S-box wire, for public inputs whose hash is not pi_hash, for a flipped exponent bit, or for a RandomAccessGate
    extra constant changed after the witness was made"""
    import plonky25_b200 as g
    rnd = random.Random(log_n)
    pis = [rnd.randrange(P) for _ in range(20 if log_n == 5 else 37)]

    def witness(ins):
        return g.poseidon_gate_witness(np.array(ins, dtype=np.uint64), ctx=ctx)
    c = build_hashing_circuit(log_n, 60 + log_n, pis, witness)
    assert c["pi"] == gl_oracle.hash_no_pad(pis)
    n_ch = 2
    alphas, betas, gammas = ([rnd.randrange(P) for _ in range(n_ch)] for _ in range(3))
    zeta = rnd.randrange(2, P)

    def holds(wires_cols, const_cols, circuit=c):
        return _identity_holds(g, ctx, circuit, wires_cols, const_cols, c["pi"], alphas, betas, gammas, zeta)

    assert holds(c["wires"], c["consts"]), "Z_H(zeta) t(zeta) != vanishing(zeta) for a valid circuit"
    # a partial-round S-box input of the second PoseidonGate row
    w = c["wires"].copy()
    w[pgo.POSEIDON_START_PARTIAL + 7, c["chain"][1]] = (int(w[pgo.POSEIDON_START_PARTIAL + 7, c["chain"][1]]) + 1) % P
    assert not holds(w, c["consts"])
    # other public inputs (a valid witness of their own hash) against the original pi_hash
    other = list(pis)
    other[-1] = (other[-1] + 1) % P
    c2 = build_hashing_circuit(log_n, 60 + log_n, other, witness)
    assert c2["pi"] != c["pi"]
    assert _identity_holds(g, ctx, c2, c2["wires"], c2["consts"], c2["pi"], alphas, betas, gammas, zeta)
    assert not holds(c2["wires"], c2["consts"], circuit=c2)
    # a flipped exponent bit of an ExponentiationGate row
    r_exp = next(r for r in range(c["n"]) if c["gate_at"][r] == 1)
    w = c["wires"].copy()
    w[1 + 30, r_exp] ^= np.uint64(1)
    assert not holds(w, c["consts"])
    # a RandomAccessGate(bits 4) extra constant changed after the witness was made
    r_ra = next(r for r in range(c["n"]) if c["gate_at"][r] == 5)
    k = c["consts"].copy()
    k[len(CIRCUIT_GROUPS) + 1, r_ra] = (int(k[len(CIRCUIT_GROUPS) + 1, r_ra]) + 3) % P
    assert not holds(c["wires"], k)


@pytest.mark.gpu
def test_error_paths(ctx):
    """every refused parameter, and a RandomAccessGate with extra constants through the entry points without gate constants: each
    returns its message and leaves the accumulator unchanged"""
    import plonky25_b200 as g
    from plonky25_b200 import _lib
    from oracle_c import splitmix_columns
    lib = ctx.lib
    wires = g.PolynomialBatch.from_values(list(splitmix_columns(11, N_WIRES, 16)), 3, False, 0, ctx=ctx)
    cs = g.PolynomialBatch.from_values(list(splitmix_columns(12, 8, 16)), 3, False, 0, ctx=ctx)
    q = g.Quotient(wires, 2, ctx=ctx)
    q.add_gate(pgo.POSEIDON, 0, [3, 4])
    before = q.values()
    info = g.SelectorsInfo([0, 0, 1], [(0, 2), (2, 3)])
    pi, al = [1, 2, 3, 4], [5, 6]
    bad = [(14, 0, "unknown gate kind 14"), (18, 0, "unknown gate kind 18"), (pgo.POSEIDON, 1, "parameter 1 out of range"),
           (pgo.EXPONENTIATION, 0, "parameter 0 out of range"), (pgo.EXPONENTIATION, 67, "parameter 67 out of range"),
           (pgo.RANDOM_ACCESS, 256, "parameter 256 out of range"), (pgo.RANDOM_ACCESS, 7 | 1 << 8, "parameter 263 out of range"),
           (pgo.RANDOM_ACCESS, 2, "parameter 2 out of range"), (pgo.RANDOM_ACCESS, 1 | 28 << 8, "parameter 7169 out of range"),
           (pgo.RANDOM_ACCESS, 4 | 4 << 8 | 64 << 16, "parameter 4195332 out of range")]
    for kind, param, msg in bad:
        with pytest.raises(ValueError, match=msg):
            q.add_gates([(kind, param), (pgo.NOOP, 0), (pgo.NOOP, 0)], info, cs, 4, pi, al)
        with pytest.raises(ValueError, match=msg):
            q.add_gate(kind, param, al)
        with pytest.raises(ValueError, match="unknown gate kind"):
            g.evaluate_gate_constraints(kind, param, np.zeros((1, 4), dtype=np.uint64), ctx=ctx)
        one = np.zeros(4, dtype=np.uint64)
        assert lib.gl_gate_eval_rows_with_constants(ctx.handle, kind, param, one.ctypes.data, one.ctypes.data, one.ctypes.data, 1,
                                                    one.ctypes.data) == _lib.GL_ERR_INVALID
        assert msg in lib.gl_ctx_last_error(ctx.handle).decode()
    # RandomAccessGate with extra constants: only the entry points with gate constants take it
    with pytest.raises(ValueError, match="gl_quotient_add_gates"):
        q.add_gate(pgo.RANDOM_ACCESS, RA_4, al)
    nw = pgo.shape(pgo.RANDOM_ACCESS, RA_4)[0]
    with pytest.raises(ValueError, match="gl_gate_eval_rows_with_constants"):
        g.evaluate_gate_constraints(pgo.RANDOM_ACCESS, RA_4, np.zeros((2, nw), dtype=np.uint64), ctx=ctx)
    with pytest.raises(ValueError, match="2 selector columns \\+ 2 gate constants exceed num_constants 3"):
        q.add_gates([(pgo.RANDOM_ACCESS, RA_4), (pgo.NOOP, 0), (pgo.NOOP, 0)], info, cs, 3, pi, al)
    assert np.array_equal(q.values(), before)
    q.add_gates([(pgo.RANDOM_ACCESS, RA_4), (pgo.EXPONENTIATION, 66), (pgo.POSEIDON, 0)], info, cs, 4, pi, al)
    assert not np.array_equal(q.values(), before)
    assert lib.gl_poseidon_gate_witness(ctx.handle, None, 1, None) == _lib.GL_ERR_INVALID
    assert "NULL pointer" in lib.gl_ctx_last_error(ctx.handle).decode()
    q.free()
    wires.merkle_tree.free(); cs.merkle_tree.free()


@pytest.mark.gpu
def test_cpp_std_gates_on_gpu(tmp_path):
    import plonky25_b200 as g
    lib = g.build()
    exe = str(tmp_path / "std_gates_test")
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    env = dict(os.environ)
    env.pop("CC", None); env.pop("CXX", None)
    subprocess.run([cxx, "-std=c++17", "-O2", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "tests", "cpp", "std_gates_test.cpp"), "-o", exe, "-L", os.path.dirname(lib), "-lgl_commit",
                    "-Wl,-rpath," + os.path.dirname(lib), "-pthread"], check=True, env=env)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "ALL OK" in r.stdout, r.stdout[-3000:] + r.stderr[-2000:]
