"""plonky2's extension-field gates ArithmeticExtensionGate, MulExtensionGate and ReducingExtensionGate (GATE_ARITHMETIC_EXTENSION /
GATE_MUL_EXTENSION / GATE_REDUCING_EXTENSION) on the device.  CPU: the restated oracle's own consistency (witness rows satisfy every
constraint, any changed wire component or constant breaks one), the library's shape queries and refused parameters, and an extension-field
circuit that vanishes on H.  GPU: the gates bit for bit against the oracle, add_gates row by row, every error path, and the verifier's
identity for that circuit (and its failure for each kind of bad witness)."""
import random

import numpy as np
import pytest

import gates_oracle as go
import gl_oracle
import plonky2_ext_gates_oracle as ego
import test_plonky2_std_gates as std

P = ego.P
AE, ME, RE = ego.ARITHMETIC_EXTENSION, ego.MUL_EXTENSION, ego.REDUCING_EXTENSION
N_ROUTED, N_WIRES, DEGREE, W32 = std.N_ROUTED, std.N_WIRES, std.DEGREE, std.W32
# every kind at 1, at its new_from_config value and at the largest param the 135-wire shape takes
EXT_GATES = [(kind, p) for kind, (config, top) in ego.CONFIG.items() for p in sorted({1, config, top})]


def _rnd_ext(rnd):
    return rnd.randrange(P), rnd.randrange(P)


def _case(kind, param, rnd):
    """(valid wires, gate constants) of one row of an extension gate, random operands and constants"""
    if kind == AE:
        k = [rnd.randrange(P), rnd.randrange(P)]
        return ego.arithmetic_extension_witness([(_rnd_ext(rnd), _rnd_ext(rnd), _rnd_ext(rnd)) for _ in range(param)], *k), k
    if kind == ME:
        k = [rnd.randrange(P)]
        return ego.mul_extension_witness([(_rnd_ext(rnd), _rnd_ext(rnd)) for _ in range(param)], k[0]), k
    return ego.reducing_extension_witness(_rnd_ext(rnd), _rnd_ext(rnd), [_rnd_ext(rnd) for _ in range(param)]), []


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("kind,param", EXT_GATES)
def test_oracle_witness_satisfies_and_every_wire_matters(kind, param):
    """witness rows satisfy every constraint; changing any single wire (either component of any extension value) or any gate constant
    breaks one"""
    rnd = random.Random(kind * 100 + param)
    nw, nc, nk = ego.shape(kind, param)
    for _ in range(2):
        w, k = _case(kind, param, rnd)
        assert len(w) == nw and len(k) == nk
        c = ego.gate_eval(kind, param, w, k)
        assert len(c) == nc and not any(c)
        for i in range(nw):
            t = list(w)
            t[i] = (t[i] + 1 + rnd.randrange(P - 1)) % P
            assert any(ego.gate_eval(kind, param, t, k)), i
        for j in range(nk):
            t = list(k)
            t[j] = (t[j] + 1 + rnd.randrange(P - 1)) % P
            assert any(ego.gate_eval(kind, param, w, t)), j


def test_oracle_reducing_is_horner_and_arithmetic_is_multiply_add():
    """ReducingExtensionGate's output is sum_i coeff_i alpha^(n-1-i) + old_acc alpha^n; ArithmeticExtensionGate's outputs are
    c0 m0 m1 + c1 addend in F_p[X]/(X^2 - 7), written out by components"""
    rnd = random.Random(3)
    alpha, old, coeffs = _rnd_ext(rnd), _rnd_ext(rnd), [_rnd_ext(rnd) for _ in range(32)]
    w = ego.reducing_extension_witness(alpha, old, coeffs)
    want = gl_oracle.ext_mul(old, gl_oracle.ext_pow(alpha, 32))
    for i, c in enumerate(coeffs):
        want = gl_oracle.ext_add(want, gl_oracle.ext_mul(c, gl_oracle.ext_pow(alpha, 31 - i)))
    assert tuple(w[0:2]) == want
    (a0, a1), (b0, b1), (d0, d1) = _rnd_ext(rnd), _rnd_ext(rnd), _rnd_ext(rnd)
    c0, c1 = rnd.randrange(P), rnd.randrange(P)
    w = ego.arithmetic_extension_witness([((a0, a1), (b0, b1), (d0, d1))], c0, c1)
    assert w[6:8] == [(c0 * (a0 * b0 + 7 * a1 * b1) + c1 * d0) % P, (c0 * (a0 * b1 + a1 * b0) + c1 * d1) % P]


def test_shapes_and_refused_params():
    """the library's shape queries equal the table, a param of 0 or one past its bound is refused, kinds 14, 18 and 22 are unknown"""
    import plonky25_b200 as g
    lib = g._lib.load()
    assert (g.GATE_ARITHMETIC_EXTENSION, g.GATE_MUL_EXTENSION, g.GATE_REDUCING_EXTENSION) == (AE, ME, RE)
    table = {AE: lambda n: (8 * n, 2 * n, 2), ME: lambda n: (6 * n, 2 * n, 1), RE: lambda n: (4 + 4 * n, 2 * n, 0)}
    for kind, (config, top) in ego.CONFIG.items():
        for p in range(1, top + 1):
            got = (lib.gl_gate_num_wires(kind, p), lib.gl_gate_num_constraints(kind, p), lib.gl_gate_num_constants(kind, p))
            assert got == table[kind](p) == ego.shape(kind, p), (kind, p)
            assert got[0] <= N_WIRES
        assert ego.shape(kind, config)[0] <= N_ROUTED or kind == RE
        assert table[kind](top + 1)[0] > N_WIRES
        for p in (0, top + 1):
            assert (lib.gl_gate_num_wires(kind, p), lib.gl_gate_num_constraints(kind, p), lib.gl_gate_num_constants(kind, p)) == (-1, -1, -1)
            with pytest.raises(ValueError, match="unknown gate kind"):
                g.gate_shape(kind, p)
    assert ego.shape(AE, 10)[0] == N_ROUTED and 6 * 14 > N_ROUTED >= ego.shape(ME, 13)[0]
    assert min((N_WIRES - 4) // 4, (N_ROUTED - 6) // 2) == 32                    # ReducingExtensionGate::max_coeffs_len(135, 80)
    for kind in (14, 18, 22):
        for p in (0, 1, 10):
            assert lib.gl_gate_num_wires(kind, p) == -1 and lib.gl_gate_num_constants(kind, p) == -1


# ------------------------------------------------------------------------------------------------ an extension-field circuit
# [ArithmeticExtension(10), MulExtension(13)] [ReducingExtension(32), Noop]: degree + group size <= 8 in both groups (3 + 2, 2 + 2)
CIRCUIT_GATES = [(AE, 10), (ME, 13), (RE, 32), (ego.NOOP, 0)]
CIRCUIT_GROUPS = [(0, 2), (2, 4)]
CIRCUIT_SELECTORS = [0, 0, 1, 1]
NUM_GATE_CONSTANTS = 2
RED_ROWS = 2                                  # ReducingExtensionGate(32) rows: a polynomial of 64 coefficients + the leading one


def build_extension_circuit(log_n, seed):
    """N rows evaluating one polynomial with extension coefficients at an extension point x in two ways.  x = k u v comes out of op 0 of a
    MulExtensionGate(13) row with a gate constant k != 1.  First way: a chain of ReducingExtensionGate(32) rows, every alpha joined to x and
    every old_acc joined to the previous row's output.  Second way: Horner over ArithmeticExtensionGate(10) ops with k(0) = k(1) = 1, op j
    computing acc_j x + c_j, every m1 joined to x, every m0 to the previous op's output.  The leading coefficient (the first reducing row's
    old_acc) is op 0's m0, the reducing rows' coefficients are the ops' addends, and the two results are joined, so Z closes only if the
    two evaluations agree.  Every join covers both components; the copy permutation is made of those cycles (sigma = identity elsewhere)."""
    rnd = random.Random(seed)
    n = 1 << log_n
    n_coeffs = 32 * RED_ROWS
    n_arith_rows = -(-n_coeffs // 10)
    row_gate = [2] * RED_ROWS + [0] * n_arith_rows + [1, 0, 1]   # one more ArithmeticExtension and MulExtension row of random ops
    row_gate += [3] * (n - len(row_gate))
    order = list(range(n))
    rnd.shuffle(order)
    gate_at = [row_gate[order[r]] for r in range(n)]
    row_of = {e: r for r, e in enumerate(order)}
    red = [row_of[t] for t in range(RED_ROWS)]
    arith = [row_of[RED_ROWS + t] for t in range(n_arith_rows)]
    mul_row = row_of[RED_ROWS + n_arith_rows]
    wires = [[rnd.randrange(P) for _ in range(N_WIRES)] for _ in range(n)]
    gconsts = [[rnd.randrange(P) for _ in range(NUM_GATE_CONSTANTS)] for _ in range(n)]
    for r in range(n):                                            # every row not written below is a valid row of its gate
        kind, param = CIRCUIT_GATES[gate_at[r]]
        if kind != ego.NOOP:
            w, k = _case(kind, param, rnd)
            wires[r][:len(w)], gconsts[r][:len(k)] = w, k
    k_mul = rnd.randrange(2, P)
    mul_ops = [(_rnd_ext(rnd), _rnd_ext(rnd)) for _ in range(13)]
    wires[mul_row][:78] = ego.mul_extension_witness(mul_ops, k_mul)
    gconsts[mul_row][0] = k_mul
    x = tuple(wires[mul_row][4:6])
    lead, coeffs = _rnd_ext(rnd), [_rnd_ext(rnd) for _ in range(n_coeffs)]
    acc = lead
    for t in range(RED_ROWS):
        w = ego.reducing_extension_witness(x, acc, coeffs[32 * t:32 * t + 32])
        wires[red[t]][:len(w)] = w
        acc = tuple(w[0:2])
    ops, acc = [], lead
    for c in coeffs:
        ops.append((acc, x, c))
        acc = gl_oracle.ext_add(gl_oracle.ext_mul(acc, x), c)
    ops += [(_rnd_ext(rnd), _rnd_ext(rnd), _rnd_ext(rnd)) for _ in range(10 * n_arith_rows - n_coeffs)]
    for t in range(n_arith_rows):
        wires[arith[t]][:80] = ego.arithmetic_extension_witness(ops[10 * t:10 * t + 10], 1, 1)
        gconsts[arith[t]][:2] = [1, 1]

    def op(j, part):                                              # first wire (column, row) of m0 / m1 / addend / output of Horner op j
        return 8 * (j % 10) + 2 * part, arith[j // 10]
    joins = [((4, mul_row), (2, r)) for r in red] + [((4, mul_row), op(j, 1)) for j in range(n_coeffs)]
    joins += [((4, red[0]), op(0, 0))] + [((4, red[t]), (0, red[t - 1])) for t in range(1, RED_ROWS)]
    joins += [((6 + 2 * (j % 32), red[j // 32]), op(j, 2)) for j in range(n_coeffs)]
    joins += [(op(j, 3), op(j + 1, 0)) for j in range(n_coeffs - 1)] + [((0, red[-1]), op(n_coeffs - 1, 3))]
    parent = {}

    def find(a):
        while parent.setdefault(a, a) != a:
            a = parent[a]
        return a
    for (ca, ra), (cb, rb) in joins:
        for d in range(2):
            parent[find((ca + d, ra))] = find((cb + d, rb))
    cycles = {}
    for cell in parent:
        cycles.setdefault(find(cell), []).append(cell)
    w_n = pow(W32, 1 << (32 - log_n), P)
    xs = [pow(w_n, i, P) for i in range(n)]
    k_is = [pow(7, j, P) for j in range(N_ROUTED)]
    sigma_of = {}
    for cyc in cycles.values():
        for a, b in zip(cyc, cyc[1:] + cyc[:1]):
            assert a[0] < N_ROUTED
            sigma_of[a] = b
    sigmas = [[k_is[sigma_of.get((j, i), (j, i))[0]] * xs[sigma_of.get((j, i), (j, i))[1]] % P for i in range(n)] for j in range(N_ROUTED)]
    nsel = len(CIRCUIT_GROUPS)
    sel_cols = [[gate_at[r] if CIRCUIT_SELECTORS[gate_at[r]] == j else ego.UNUSED_SELECTOR for r in range(n)] for j in range(nsel)]
    const_cols = sel_cols + [[gconsts[r][j] for r in range(n)] for j in range(NUM_GATE_CONSTANTS)]
    value = lead
    for c in coeffs:
        value = gl_oracle.ext_add(gl_oracle.ext_mul(value, x), c)
    return {"n": n, "log_n": log_n, "gate_at": gate_at, "red": red, "arith": arith, "mul_row": mul_row, "x": x, "value": value,
            "n_cycles": len(cycles), "wires": np.array(wires, dtype=np.uint64).T.copy(), "consts": np.array(const_cols, dtype=np.uint64),
            "sigmas": np.array(sigmas, dtype=np.uint64), "k_is": k_is, "num_constants": nsel + NUM_GATE_CONSTANTS}


@pytest.mark.parametrize("log_n", [5, 6])
def test_extension_circuit_vanishes_on_H(log_n):
    """every row's filtered constraint sum is 0, every wire of a copy cycle holds the same value, and both evaluations equal the
    polynomial's value at x"""
    c = build_extension_circuit(log_n, 90 + log_n)
    n, w, k = c["n"], c["wires"], c["consts"]
    for r in range(n):
        assert not any(ego.eval_filtered(CIRCUIT_GATES, CIRCUIT_SELECTORS, CIRCUIT_GROUPS, k[:, r].tolist(), w[:, r].tolist(), [0] * 4)), r
    w_n = pow(W32, 1 << (32 - log_n), P)
    cell = {c["k_is"][j] * pow(w_n, i, P) % P: (j, i) for j in range(N_ROUTED) for i in range(n)}
    moved = 0
    for j in range(N_ROUTED):
        for i in range(n):
            jj, ii = cell[int(c["sigmas"][j, i])]
            assert w[j, i] == w[jj, ii]
            moved += (jj, ii) != (j, i)
    # per component: x (1 + RED_ROWS alphas + 64 m1), the leading coefficient, the reducing chain, 64 coefficients, 63 Horner links,
    # the two results
    sizes = [1 + RED_ROWS + 64, 2] + [2] * (RED_ROWS - 1) + [2] * 64 + [2] * 63 + [2]
    assert c["n_cycles"] == 2 * len(sizes) and moved == 2 * sum(sizes)
    assert tuple(w[0:2, c["red"][-1]].tolist()) == c["value"] == tuple(w[6 + 8 * 3:8 + 8 * 3, c["arith"][-1]].tolist())
    assert tuple(w[4:6, c["mul_row"]].tolist()) == c["x"]


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("kind,param", EXT_GATES)
def test_ext_gates_match_oracle(ctx, kind, param):
    """valid, tampered and arbitrary rows (non-canonical words included) against the oracle, bit for bit"""
    import plonky25_b200 as g
    lib, rnd = ctx.lib, random.Random(kind * 1000003 + param)
    nw, nc, nk = ego.shape(kind, param)
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
            k = [x + P if x < (1 << 64) - P else x for x in k]
        rows.append(w)
        consts.append(k)
    rows = np.array(rows, dtype=np.uint64).reshape(48, nw)
    consts = np.array(consts, dtype=np.uint64).reshape(48, nk)
    out = std._eval_rows(ctx, kind, param, rows, consts, pi)
    for r in range(48):
        want = ego.gate_eval(kind, param, rows[r].tolist(), consts[r].tolist(), pi)
        assert out[r].tolist() == want, r
        if r % 3 == 0:
            assert not any(want), r
    if nk == 0:
        assert np.array_equal(g.evaluate_gate_constraints(kind, param, rows, ctx=ctx), out)
    assert np.array_equal(g.evaluate_gate_constraints(kind, param, rows, ctx=ctx, constants=consts, public_inputs_hash=pi), out)


def _constraints(kind, param, w, k, pi):
    return go.poseidon2_gate_eval(w) if kind == std.POSEIDON2 else ego.gate_eval(kind, param, w, k, pi)


@pytest.mark.gpu
@pytest.mark.parametrize("groups,selectors,n_ch", [
    ([(0, 1), (1, 4), (4, 8)], [0, 1, 1, 1, 2, 2, 2, 2], 2),
    ([(0, 8)], [0] * 8, 1),
    ([(0, 2), (2, 3), (3, 6), (6, 8)], [0, 0, 1, 2, 2, 2, 3, 3], 4)])
def test_add_gates_row_by_row(ctx, groups, selectors, n_ch):
    """the extension gates mixed with existing ones into selector groups; random wires and constants/sigmas columns (selector values are
    arbitrary field elements at the LDE points): every sampled accumulator row is the oracle's eval_filtered reduced with alpha_k"""
    import plonky25_b200 as g
    from oracle_c import splitmix_columns
    gates = [(AE, 10), (RE, 32), (ME, 13), (ego.ARITHMETIC, 20), (std.POSEIDON2, 0), (AE, 16), (ego.RANDOM_ACCESS, std.RA_4), (ME, 22)]
    log_n, r = 6, 3
    n, R = 1 << log_n, 1 << (log_n + r)
    nsel = len(groups)
    num_constants = nsel + 2
    wires = g.PolynomialBatch.from_values(list(splitmix_columns(900 + n_ch, N_WIRES, n)), r, False, 1, ctx=ctx)
    cs = g.PolynomialBatch.from_values(list(splitmix_columns(950 + n_ch, num_constants + 5, n)), r, False, 1, ctx=ctx)
    rnd = random.Random(40 + n_ch)
    alphas = [rnd.randrange(P) for _ in range(n_ch)]
    pi = [rnd.getrandbits(64) for _ in range(4)]
    offset = 11
    q = g.Quotient(wires, n_ch, ctx=ctx)
    assert q.add_gates(gates, g.SelectorsInfo(selectors, groups), cs, num_constants, pi, alphas, constraint_offset=offset) > 0
    acc = q.values()
    q.free()
    rows = sorted(set([0, 1, R - 1] + [rnd.randrange(R) for _ in range(16)]))
    lw, lc = std._rows_at(wires, rows), std._rows_at(cs, rows)
    for j, row in enumerate(rows):
        w, k = lw[j].tolist(), lc[j].tolist()
        want = [0] * n_ch
        for i, (kind, param) in enumerate(gates):
            f = ego.compute_filter(i, groups[selectors[i]], k[selectors[i]], nsel > 1)
            c = _constraints(kind, param, w, k[nsel:num_constants], [x % P for x in pi])
            for ch in range(n_ch):
                want[ch] = (want[ch] + f * ego.reduce_with_powers(c, alphas[ch], offset)) % P
        assert [int(acc[ch, row]) for ch in range(n_ch)] == want, row
    wires.merkle_tree.free(); cs.merkle_tree.free()


@pytest.mark.gpu
def test_error_paths(ctx):
    """every refused parameter and kind, and the two extension gates that read gate constants through the entry points without them:
    each returns its message and leaves the accumulator unchanged; ReducingExtensionGate goes through every entry point"""
    import plonky25_b200 as g
    from plonky25_b200 import _lib
    from oracle_c import splitmix_columns
    lib = ctx.lib
    wires = g.PolynomialBatch.from_values(list(splitmix_columns(13, N_WIRES, 16)), 3, False, 0, ctx=ctx)
    cs = g.PolynomialBatch.from_values(list(splitmix_columns(14, 8, 16)), 3, False, 0, ctx=ctx)
    q = g.Quotient(wires, 2, ctx=ctx)
    al = [5, 6]
    q.add_gate(RE, 32, al)
    before = q.values()
    info = g.SelectorsInfo([0, 0, 1], [(0, 2), (2, 3)])
    pi = [1, 2, 3, 4]
    bad = [(14, 1, "unknown gate kind 14"), (18, 1, "unknown gate kind 18"), (22, 1, "unknown gate kind 22"),
           (AE, 0, "parameter 0 out of range"), (AE, 17, "parameter 17 out of range"), (ME, 0, "parameter 0 out of range"),
           (ME, 23, "parameter 23 out of range"), (RE, 0, "parameter 0 out of range"), (RE, 33, "parameter 33 out of range")]
    for kind, param, msg in bad:
        with pytest.raises(ValueError, match=msg):
            q.add_gates([(kind, param), (ego.NOOP, 0), (ego.NOOP, 0)], info, cs, 4, pi, al)
        with pytest.raises(ValueError, match=msg):
            q.add_gate(kind, param, al)
        with pytest.raises(ValueError, match="unknown gate kind"):
            g.evaluate_gate_constraints(kind, param, np.zeros((1, 4), dtype=np.uint64), ctx=ctx)
        one = np.zeros(4, dtype=np.uint64)
        assert lib.gl_gate_eval_rows_with_constants(ctx.handle, kind, param, one.ctypes.data, one.ctypes.data, one.ctypes.data, 1,
                                                    one.ctypes.data) == _lib.GL_ERR_INVALID
        assert msg in lib.gl_ctx_last_error(ctx.handle).decode()
    # the gates with gate constants: only the entry points with gate constants take them
    for kind, param in ((AE, 10), (ME, 13)):
        with pytest.raises(ValueError, match="reads gate constants or the public-inputs hash: use gl_quotient_add_gates"):
            q.add_gate(kind, param, al)
        nw = ego.shape(kind, param)[0]
        with pytest.raises(ValueError, match="use gl_gate_eval_rows_with_constants"):
            g.evaluate_gate_constraints(kind, param, np.zeros((2, nw), dtype=np.uint64), ctx=ctx)
    with pytest.raises(ValueError, match="2 selector columns \\+ 2 gate constants exceed num_constants 3"):
        q.add_gates([(AE, 10), (ego.NOOP, 0), (ego.NOOP, 0)], info, cs, 3, pi, al)
    with pytest.raises(ValueError, match="parameter 33 out of range"):   # a refused gate after valid ones: nothing has launched
        q.add_gates([(AE, 10), (ME, 13), (RE, 33)], info, cs, 4, pi, al)
    assert np.array_equal(q.values(), before)
    nw = ego.shape(RE, 32)[0]
    rows = np.array(splitmix_columns(15, nw, 3).T, dtype=np.uint64)
    assert np.array_equal(g.evaluate_gate_constraints(RE, 32, rows, ctx=ctx),
                          np.array([ego.gate_eval(RE, 32, r.tolist()) for r in rows], dtype=np.uint64))
    q.add_gates([(AE, 10), (ME, 13), (RE, 32)], info, cs, 4, pi, al)
    assert not np.array_equal(q.values(), before)
    q.free()
    wires.merkle_tree.free(); cs.merkle_tree.free()


def _identity_holds(g, ctx, c, wires_cols, const_cols, alphas, betas, gammas, zeta, n_ch=2, r=3):
    """tests/test_plonky2_std_gates.py · _identity_holds for this file's circuit: commit constants+sigmas, wires and Z / partial products;
    add_permutation, add_gates at offset n_ch (1 + n_chunks); commit the quotient; then the verifier's check
    Z_H(zeta) sum_c zeta^(cN) t_c(zeta) == the alpha-combination of the permutation terms and eval_filtered, from the polynomials at zeta"""
    n = c["n"]
    pi = [0] * 4
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
    ew = [std._eval_poly(cw[j], zeta) for j in range(N_WIRES)]
    ec = [std._eval_poly(cs[j], zeta) for j in range(c["num_constants"])]
    es = [std._eval_poly(cs[c["num_constants"] + j], zeta) for j in range(N_ROUTED)]
    ez = [std._eval_poly(cz[j], zeta) for j in range(n_ch * n_chunks)]
    ezn = [std._eval_poly(cz[j], gz) for j in range(n_ch * n_chunks)]
    perm = go.vanishing_permutation_terms(ew[:N_ROUTED], es, ez, ezn, zeta, c["k_is"], betas, gammas, DEGREE, c["log_n"])
    gate_terms = ego.eval_filtered(CIRCUIT_GATES, CIRCUIT_SELECTORS, CIRCUIT_GROUPS, ec, ew, pi)
    z_h = (pow(zeta, n, P) - 1) % P
    ok = True
    for ch in range(n_ch):
        t_zeta = 0
        for k in reversed(range(1 << r)):
            t_zeta = (t_zeta * pow(zeta, n, P) + std._eval_poly(ct[ch * (1 << r) + k], zeta)) % P
        ok &= z_h * t_zeta % P == ego.reduce_with_powers(perm + gate_terms, alphas[ch])
    for b in (sig, wires, zs_b, t):
        b.merkle_tree.free()
    return ok


@pytest.mark.gpu
@pytest.mark.parametrize("log_n", [5, 6])
def test_verifier_identity_for_an_extension_circuit(ctx, log_n):
    """the quotient the device commits satisfies Z_H(zeta) t(zeta) = vanishing(zeta) at a random zeta for the valid extension circuit,
    and does not for the second component of one ReducingExtensionGate accumulator, for an ArithmeticExtensionGate k(1) changed after the
    witness was made, or for the first component of one MulExtensionGate output"""
    import plonky25_b200 as g
    rnd = random.Random(20 + log_n)
    c = build_extension_circuit(log_n, 90 + log_n)
    n_ch = 2
    alphas, betas, gammas = ([rnd.randrange(P) for _ in range(n_ch)] for _ in range(3))
    zeta = rnd.randrange(2, P)

    def holds(wires_cols, const_cols):
        return _identity_holds(g, ctx, c, wires_cols, const_cols, alphas, betas, gammas, zeta)

    assert holds(c["wires"], c["consts"]), "Z_H(zeta) t(zeta) != vanishing(zeta) for a valid circuit"
    # the second component of accumulator 5 of the first ReducingExtensionGate row (not a routed wire)
    w = c["wires"].copy()
    col = 6 + 2 * 32 + 2 * 5 + 1
    w[col, c["red"][0]] = (int(w[col, c["red"][0]]) + 1) % P
    assert not holds(w, c["consts"])
    # k(1) of an ArithmeticExtensionGate row changed after the witness was made
    k = c["consts"].copy()
    k[len(CIRCUIT_GROUPS) + 1, c["arith"][2]] = (int(k[len(CIRCUIT_GROUPS) + 1, c["arith"][2]]) + 3) % P
    assert not holds(c["wires"], k)
    # the first component of op 5's output of the MulExtensionGate row (a wire no copy cycle holds)
    w = c["wires"].copy()
    w[6 * 5 + 4, c["mul_row"]] = (int(w[6 * 5 + 4, c["mul_row"]]) + 1) % P
    assert not holds(w, c["consts"])
