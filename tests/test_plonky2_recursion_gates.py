"""plonky2's CosetInterpolationGate, ReducingGate and PoseidonMdsGate (GATE_COSET_INTERPOLATION / GATE_REDUCING / GATE_POSEIDON_MDS) on the
device: the three gates plonky2's recursive verifier circuit registers besides the ones already built.  CPU: the restated oracle's own
consistency (witness rows satisfy every constraint, any changed wire component breaks one), CosetInterpolation against
fri_verifier.compute_evaluation and the FRI fold steps of an oracle proof, PoseidonMds against gl_oracle._mds_layer, the library's shapes
and refusals, and a recursion-shaped circuit that vanishes on H.  GPU: the gates bit for bit against the oracle through every entry
point, add_gate / add_gates row by row (the whole gate list of a standard_recursion_config verifier circuit in one call), the fold rows
of a device FRI proof, every error path, and the verifier's identity for the circuit (and its failure for each kind of bad witness)."""
import copy
import random

import numpy as np
import pytest

import fri_verifier as fv
import gl_oracle
import plonky2_ext_gates_oracle as ego
import plonky2_recursion_gates_oracle as ro
import test_plonky2_ext_gates as ext
import test_plonky2_std_gates as std

P = ro.P
CI, RED, MDS = ro.COSET_INTERPOLATION, ro.REDUCING, ro.POSEIDON_MDS
N_ROUTED, N_WIRES, DEGREE, W32 = std.N_ROUTED, std.N_WIRES, std.DEGREE, std.W32
CI_4 = ro.coset_interpolation_params(4)                                        # with_max_degree(4, 8) = (4, 6): the wrapper's FRI arity
# with_max_degree(1..5, 8), the smallest degree at 2 and 5 subgroup bits, the largest shape (5, 3) and a degree-n gate
CI_PARAMS = sorted({ro.coset_interpolation_params(b) for b in range(1, 6)} | {2 | 2 << 8, 5 | 3 << 8, 5 | 32 << 8, 3 | 2 << 8})
NEW_GATES = [(CI, p) for p in CI_PARAMS] + [(RED, 1), (RED, 16), (RED, ro.REDUCING_MAX), (MDS, 0)]


def _rnd_ext(rnd):
    return rnd.randrange(P), rnd.randrange(P)


def _case(kind, param, rnd):
    """valid wires of one row, random operands"""
    if kind == CI:
        n = 1 << (param & 0xFF)
        return ro.coset_interpolation_witness(param, rnd.randrange(1, P), [_rnd_ext(rnd) for _ in range(n)], _rnd_ext(rnd))
    if kind == RED:
        return ro.reducing_witness(_rnd_ext(rnd), _rnd_ext(rnd), [rnd.randrange(P) for _ in range(param)])
    return ro.poseidon_mds_witness([_rnd_ext(rnd) for _ in range(12)])


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("kind,param", NEW_GATES)
def test_oracle_witness_satisfies_and_every_wire_matters(kind, param):
    """witness rows satisfy every constraint; changing any single wire (either component of any extension value) breaks one"""
    rnd = random.Random(kind * 100000 + param)
    nw, nc, nk = ro.shape(kind, param)
    assert nk == 0
    for _ in range(2):
        w = _case(kind, param, rnd)
        assert len(w) == nw
        c = ro.gate_eval(kind, param, w)
        assert len(c) == nc and not any(c)
        for i in range(nw):
            t = list(w)
            t[i] = (t[i] + 1 + rnd.randrange(P - 1)) % P
            assert any(ro.gate_eval(kind, param, t)), i


def test_coset_chunks_cover_the_domain_and_weights_are_closed_form():
    """for every (subgroup_bits, degree) the chunks cover all n points once, in order; barycentric_weights' product form equals the
    closed form x_i / n the kernel uses"""
    for bits in range(1, 6):
        n = 1 << bits
        for degree in range(2, n + 1):
            assert [j for a, b in ro.coset_chunks(bits | degree << 8) for j in range(a, b)] == list(range(n)), (bits, degree)
        xs = ro.coset_domain(bits)
        assert ro.barycentric_weights(xs) == [x * gl_oracle.inv(n) % P for x in xs]


@pytest.mark.parametrize("arity_bits", [1, 2, 3, 4, 5])
def test_coset_interpolation_is_compute_evaluation(arity_bits):
    """the gate's evaluation value is fri_verifier.compute_evaluation's interpolant on shift H at the point, for random cosets"""
    rnd = random.Random(arity_bits)
    n = 1 << arity_bits
    g = gl_oracle.primitive_root_of_unity(arity_bits)
    for _ in range(4):
        x, within = rnd.randrange(1, P), rnd.randrange(n)
        evals, beta = [_rnd_ext(rnd) for _ in range(n)], _rnd_ext(rnd)
        coset_start = x * pow(g, n - gl_oracle.reverse_bits(within, arity_bits), P) % P
        for param in {ro.coset_interpolation_params(arity_bits), arity_bits | n << 8, arity_bits | 2 << 8}:
            if ro.shape(CI, param)[0] > N_WIRES:
                continue
            w = ro.coset_interpolation_witness(param, coset_start, [evals[gl_oracle.reverse_bits(k, arity_bits)] for k in range(n)], beta)
            lay = ro.coset_interpolation_layout(param)
            assert tuple(w[lay["value_out"]:lay["value_out"] + 2]) == fv.compute_evaluation(x, within, arity_bits, evals, beta)


def test_poseidon_mds_on_base_inputs_is_the_mds_layer():
    """PoseidonMdsGate applied to (x, 0) vectors reproduces gl_oracle._mds_layer(x) in component 0 and 0 in component 1"""
    rnd = random.Random(5)
    for _ in range(8):
        x = [rnd.randrange(P) for _ in range(12)]
        w = ro.poseidon_mds_witness([(v, 0) for v in x])
        assert w[24::2] == gl_oracle._mds_layer(x) and not any(w[25::2])


def fold_rows(ch, commit_caps, x_indices, steps, arities, lde_bits, final_poly):
    """the CosetInterpolationGate rows plonky2's recursive verifier builds for every FRI query step: shift = coset_start, values = the
    bit-reversed evals, point = beta (betas from the transcript, as verify_fri_proof draws them; `ch` is in the state prove_openings
    started from).  Yields (param, row, value the next step needs: its evals[within], or final_poly(x) after the last step)"""
    ch.get_extension_challenge()                                   # alpha
    betas = []
    for cap in commit_caps:
        ch.observe_cap(cap)
        betas.append(ch.get_extension_challenge())
    for x_index, rnd_steps in zip(x_indices, steps):
        subgroup_x = gl_oracle.MULTIPLICATIVE_GROUP_GENERATOR * pow(gl_oracle.primitive_root_of_unity(lde_bits),
                                                                   gl_oracle.reverse_bits(x_index, lde_bits), P) % P
        x = x_index
        for i, arity_bits in enumerate(arities):
            n = 1 << arity_bits
            evals = rnd_steps[i]
            within = x & (n - 1)
            g = gl_oracle.primitive_root_of_unity(arity_bits)
            coset_start = subgroup_x * pow(g, n - gl_oracle.reverse_bits(within, arity_bits), P) % P
            param = ro.coset_interpolation_params(arity_bits)
            row = ro.coset_interpolation_witness(param, coset_start, [evals[gl_oracle.reverse_bits(k, arity_bits)] for k in range(n)],
                                                 betas[i])
            subgroup_x, x = pow(subgroup_x, n, P), x >> arity_bits
            if i + 1 < len(arities):
                nxt = rnd_steps[i + 1][x & ((1 << arities[i + 1]) - 1)]
            else:
                nxt = gl_oracle.ext_eval_poly(list(final_poly), subgroup_x)
            yield param, row, tuple(nxt)


@pytest.mark.parametrize("cfg", [(5, 2, 1, [2, 1], 4, 5), (6, 1, 2, [3], 3, 4), (6, 3, 0, [1, 2, 1], 2, 4), (6, 2, 1, [4], 2, 4)])
def test_fri_fold_rows_of_an_oracle_proof(cfg):
    """for every query step of an oracle FRI proof the recursive verifier's CosetInterpolationGate row is satisfied and its evaluation
    value is the next step's evals[within] (or final_poly(x) after the last step)"""
    import test_oracle
    proof, ch = test_oracle._prove_for_verifier(*cfg, seed=93)
    fv.verify_fri_proof(challenger=copy.deepcopy(ch), **proof)
    log_n, r, _, arities = cfg[:4]
    steps = [[[tuple(e) for e in st["evals"]] for st in rnd["steps"]] for rnd in proof["query_rounds"]]
    n_rows = 0
    for param, row, nxt in fold_rows(ch, proof["commit_caps"], [rnd["x_index"] for rnd in proof["query_rounds"]], steps, arities,
                                     log_n + r, proof["final_poly"]):
        lay = ro.coset_interpolation_layout(param)
        assert not any(ro.gate_eval(CI, param, row))
        assert tuple(row[lay["value_out"]:lay["value_out"] + 2]) == nxt
        n_rows += 1
    assert n_rows == len(proof["query_rounds"]) * len(arities)


def test_shapes_and_refused_params():
    """the library's shape queries equal the table; out-of-range params and kinds 14, 18, 22 and 26 are refused"""
    import plonky25_b200 as g
    lib = g._lib.load()
    assert (g.GATE_COSET_INTERPOLATION, g.GATE_REDUCING, g.GATE_POSEIDON_MDS) == (CI, RED, MDS)

    def got(kind, p):
        return lib.gl_gate_num_wires(kind, p), lib.gl_gate_num_constraints(kind, p), lib.gl_gate_num_constants(kind, p)
    refused = (-1, -1, -1)
    assert lib.gl_gate_num_wires(CI, g.coset_interpolation_params(4)) == 47
    for bits, md, want in ((4, 8, (4, 6, 47, 12)), (5, 8, (5, 8, 87, 20)), (3, 8, (3, 8, 23, 4)), (1, 8, (1, 2, 11, 4))):
        p = g.coset_interpolation_params(bits, md)
        assert p == ro.coset_interpolation_params(bits, md) and (p & 0xFF, p >> 8, *got(CI, p)[:2]) == want
    assert got(CI, 5 | 3 << 8) == (131, 64, 0) and got(CI, 5 | 2 << 8) == refused      # (5, 2) would need 191 wires
    for bits in range(1, 6):
        n = 1 << bits
        for degree in range(2, n + 1):
            p = bits | degree << 8
            want = ro.shape(CI, p)
            assert got(CI, p) == (want if want[0] <= N_WIRES else refused), (bits, degree)
        for p in (bits | 1 << 8, bits | 0 << 8, bits | (n + 1) << 8, bits | 2 << 8 | 1 << 16, bits | 2 << 8 | 1 << 31):
            assert got(CI, p) == refused, hex(p)
    for p in (0 | 2 << 8, 6 | 8 << 8, 6 | 64 << 8):
        assert got(CI, p) == refused
    for m in range(1, ro.REDUCING_MAX + 1):
        assert got(RED, m) == ro.shape(RED, m) == (4 + 3 * m, 2 * m, 0)
    assert min((N_WIRES - 4) // 3, N_ROUTED - 6) == ro.REDUCING_MAX                 # ReducingGate::max_coeffs_len(135, 80)
    assert got(RED, 0) == got(RED, ro.REDUCING_MAX + 1) == refused
    assert got(MDS, 0) == ro.shape(MDS, 0) == (48, 24, 0) and got(MDS, 1) == refused
    for kind in (14, 18, 22, 26):
        for p in (0, 1, 10, CI_4):
            assert got(kind, p) == refused
            with pytest.raises(ValueError, match="unknown gate kind"):
                g.gate_shape(kind, p)


# ------------------------------------------------------------------------------------------------ a recursion-shaped circuit
# [CosetInterpolation(4, 6)] [Reducing(16), PoseidonMds, ArithmeticExtension(10), Noop]: degree + group size <= 8 (6 + 1, 3 + 4)
CIRCUIT_GATES = [(CI, CI_4), (RED, 16), (MDS, 0), (ego.ARITHMETIC_EXTENSION, 10), (ego.NOOP, 0)]
CIRCUIT_GROUPS = [(0, 1), (1, 5)]
CIRCUIT_SELECTORS = [0, 1, 1, 1, 1]
NUM_GATE_CONSTANTS = 2


def _copy_sigmas(joins, log_n):
    """sigma columns of the copy permutation made of the cycles that `joins` (pairs of (column, row) extension cells, both components
    joined) generate; identity elsewhere.  Returns (sigmas [N_ROUTED][n], number of cycles)"""
    n = 1 << log_n
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
    return np.array(sigmas, dtype=np.uint64), len(cycles), k_is


def build_recursion_circuit(log_n, seed):
    """N rows evaluating a base-coefficient polynomial p (deg < 16) at an extension point beta in two ways: one CosetInterpolationGate(4, 6)
    row over p's values on s H_16, and a ReducingGate(16) Horner chain (coefficients from the leading one down, old_acc 0) whose alpha is
    joined to beta.  beta is output 0 of a PoseidonMdsGate row and is joined to the coset row's evaluation point; the two results are
    joined, so Z closes only if the two evaluations agree.  Every other row is a valid random row of its gate."""
    rnd = random.Random(seed)
    n = 1 << log_n
    row_gate = [0, 1, 2, 0, 1, 2, 2, 3, 3] + [4] * (n - 9)
    order = list(range(n))
    rnd.shuffle(order)
    gate_at = [row_gate[order[r]] for r in range(n)]
    row_of = {e: r for r, e in enumerate(order)}
    ci_row, red_row, mds_row = row_of[0], row_of[1], row_of[2]
    wires = [[rnd.randrange(P) for _ in range(N_WIRES)] for _ in range(n)]
    gconsts = [[rnd.randrange(P) for _ in range(NUM_GATE_CONSTANTS)] for _ in range(n)]
    for r in range(n):
        kind, param = CIRCUIT_GATES[gate_at[r]]
        if kind == ego.ARITHMETIC_EXTENSION:
            w, k = ext._case(kind, param, rnd)
            wires[r][:len(w)], gconsts[r][:len(k)] = w, k
        elif kind != ego.NOOP:
            w = _case(kind, param, rnd)
            wires[r][:len(w)] = w
    mds = ro.poseidon_mds_witness([_rnd_ext(rnd) for _ in range(12)])
    wires[mds_row][:48] = mds
    beta = tuple(mds[24:26])
    coeffs = [rnd.randrange(P) for _ in range(16)]
    shift = gl_oracle.MULTIPLICATIVE_GROUP_GENERATOR * rnd.randrange(1, P) % P
    om = gl_oracle.primitive_root_of_unity(4)
    vals = [(gl_oracle.eval_poly(coeffs, shift * pow(om, i, P) % P), 0) for i in range(16)]
    wires[ci_row][:47] = ro.coset_interpolation_witness(CI_4, shift, vals, beta)
    wires[red_row][:52] = ro.reducing_witness(beta, (0, 0), coeffs[::-1])
    lay = ro.coset_interpolation_layout(CI_4)
    joins = [((24, mds_row), (lay["point"], ci_row)), ((24, mds_row), (2, red_row)), ((lay["value_out"], ci_row), (0, red_row))]
    sigmas, n_cycles, k_is = _copy_sigmas(joins, log_n)
    nsel = len(CIRCUIT_GROUPS)
    sel_cols = [[gate_at[r] if CIRCUIT_SELECTORS[gate_at[r]] == j else ro.UNUSED_SELECTOR for r in range(n)] for j in range(nsel)]
    const_cols = sel_cols + [[gconsts[r][j] for r in range(n)] for j in range(NUM_GATE_CONSTANTS)]
    value = gl_oracle.ext_eval_poly_ext([(c, 0) for c in coeffs], beta)
    return {"n": n, "log_n": log_n, "gate_at": gate_at, "ci_row": ci_row, "red_row": red_row, "mds_row": mds_row, "beta": beta,
            "value": value, "n_cycles": n_cycles, "wires": np.array(wires, dtype=np.uint64).T.copy(),
            "consts": np.array(const_cols, dtype=np.uint64), "sigmas": sigmas, "k_is": k_is, "num_constants": nsel + NUM_GATE_CONSTANTS}


@pytest.mark.parametrize("log_n", [5, 6])
def test_recursion_circuit_vanishes_on_H(log_n):
    """every row's filtered constraint sum is 0, every wire of a copy cycle holds the same value, and both evaluations equal p(beta)"""
    c = build_recursion_circuit(log_n, 70 + log_n)
    n, w, k = c["n"], c["wires"], c["consts"]
    for r in range(n):
        assert not any(ro.eval_filtered(CIRCUIT_GATES, CIRCUIT_SELECTORS, CIRCUIT_GROUPS, k[:, r].tolist(), w[:, r].tolist(), [0] * 4)), r
    w_n = pow(W32, 1 << (32 - log_n), P)
    cell = {c["k_is"][j] * pow(w_n, i, P) % P: (j, i) for j in range(N_ROUTED) for i in range(n)}
    moved = sum((cell[int(c["sigmas"][j, i])] != (j, i)) for j in range(N_ROUTED) for i in range(n))
    for j in range(N_ROUTED):
        for i in range(n):
            jj, ii = cell[int(c["sigmas"][j, i])]
            assert w[j, i] == w[jj, ii]
    assert c["n_cycles"] == 4 and moved == 2 * (3 + 2)                  # per component: beta (3 cells), the two results (2 cells)
    lay = ro.coset_interpolation_layout(CI_4)
    assert tuple(w[0:2, c["red_row"]].tolist()) == c["value"] == tuple(w[lay["value_out"]:lay["value_out"] + 2, c["ci_row"]].tolist())


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("kind,param", NEW_GATES)
def test_recursion_gates_match_oracle(ctx, kind, param):
    """valid, tampered and arbitrary rows (non-canonical words included) against the oracle, bit for bit, through
    gl_gate_eval_rows_with_constants and gl_gate_eval_rows"""
    import plonky25_b200 as g
    lib, rnd = ctx.lib, random.Random(kind * 1000003 + param)
    nw, nc, nk = ro.shape(kind, param)
    assert (lib.gl_gate_num_wires(kind, param), lib.gl_gate_num_constraints(kind, param), lib.gl_gate_num_constants(kind, param)) == (nw, nc, nk)
    pi = [rnd.getrandbits(64) for _ in range(4)]
    rows = []
    for r in range(48):
        w = _case(kind, param, rnd)
        if r % 3 == 1:
            w[rnd.randrange(nw)] = rnd.randrange(P)
        if r % 3 == 2:
            w = [rnd.getrandbits(64) for _ in range(nw)]
        if r % 6 == 0:                                      # the same row with non-canonical words (x + p where that fits)
            w = [x + P if x < (1 << 64) - P else x for x in w]
        rows.append(w)
    rows = np.array(rows, dtype=np.uint64).reshape(48, nw)
    out = std._eval_rows(ctx, kind, param, rows, np.zeros((48, 0), dtype=np.uint64), pi)
    for r in range(48):
        want = ro.gate_eval(kind, param, rows[r].tolist())
        assert out[r].tolist() == want, r
        if r % 3 == 0:
            assert not any(want), r
    assert np.array_equal(g.evaluate_gate_constraints(kind, param, rows, ctx=ctx), out)
    assert np.array_equal(g.evaluate_gate_constraints(kind, param, rows, ctx=ctx, constants=np.zeros((48, 0), dtype=np.uint64),
                                                      public_inputs_hash=pi), out)


def _constraints(kind, param, w, k, pi):
    return ro.gate_eval(kind, param, w, k, pi)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,param", [(CI, CI_4), (CI, 5 | 3 << 8), (RED, 43), (MDS, 0)])
def test_add_gate_row_by_row(ctx, kind, param):
    """gl_quotient_add_gate without a filter and with a filter column: every sampled accumulator row is filter(row) times the oracle's
    constraints reduced with alpha_k, added to what the accumulator held"""
    import plonky25_b200 as g
    from oracle_c import splitmix_columns
    log_n, r, n_ch = 6, 3, 3
    n, R = 1 << log_n, 1 << (log_n + r)
    wires = g.PolynomialBatch.from_values(list(splitmix_columns(300 + kind, N_WIRES, n)), r, False, 1, ctx=ctx)
    fb = g.PolynomialBatch.from_values(list(splitmix_columns(310 + kind, 3, n)), r, False, 1, ctx=ctx)
    rnd = random.Random(param)
    alphas = [rnd.randrange(P) for _ in range(n_ch)]
    offset = 7
    q = g.Quotient(wires, n_ch, ctx=ctx)
    q.add_gate(kind, param, alphas, constraint_offset=offset)
    once = q.values()
    q.add_gate(kind, param, alphas, constraint_offset=offset, filter=(fb, 2))
    twice = q.values()
    q.free()
    rows = sorted(set([0, 1, R - 1] + [rnd.randrange(R) for _ in range(16)]))
    lw, lf = std._rows_at(wires, rows), std._rows_at(fb, rows)
    for j, row in enumerate(rows):
        c = ro.gate_eval(kind, param, lw[j].tolist())
        f = int(lf[j][2]) % P
        for ch in range(n_ch):
            v = ro.reduce_with_powers(c, alphas[ch], offset)
            assert int(once[ch, row]) == v, row
            assert int(twice[ch, row]) == (v + f * v) % P, row
    wires.merkle_tree.free(); fb.merkle_tree.free()


# the gates of plonky2's verify_proof_circuit under standard_recursion_config, in selector groups of degree + size <= 8
RECURSION_GATES = [(ro.NOOP, 0), (ro.CONSTANT, 2), (MDS, 0), (ro.PUBLIC_INPUT, 0), (ro.BASE_SUM, 63 | 2 << 8),
                   (ro.REDUCING_EXTENSION, 32), (RED, 43), (ro.ARITHMETIC_EXTENSION, 10), (ro.ARITHMETIC, 20), (ro.MUL_EXTENSION, 13),
                   (ro.RANDOM_ACCESS, std.RA_4), (ro.EXPONENTIATION, 66), (CI, CI_4), (ro.POSEIDON, 0)]
RECURSION_GROUPS = [(0, 5), (5, 10), (10, 12), (12, 13), (13, 14)]
RECURSION_SELECTORS = [0] * 5 + [1] * 5 + [2] * 2 + [3, 4]


@pytest.mark.gpu
@pytest.mark.parametrize("gates,groups,selectors,n_ch", [
    (RECURSION_GATES, RECURSION_GROUPS, RECURSION_SELECTORS, 2),
    ([(CI, CI_4), (RED, 16), (MDS, 0), (ego.ARITHMETIC, 20), (CI, 5 | 8 << 8), (RED, 43)], [(0, 6)], [0] * 6, 1),
    ([(MDS, 0), (CI, 3 | 8 << 8), (RED, 1), (ego.REDUCING_EXTENSION, 32)], [(0, 1), (1, 3), (3, 4)], [0, 1, 1, 2], 4)])
def test_add_gates_row_by_row(ctx, gates, groups, selectors, n_ch):
    """one add_gates call (the first case: a standard_recursion_config verifier circuit's whole gate list); random wires and
    constants/sigmas columns (selector values are arbitrary field elements at the LDE points): every sampled accumulator row is the
    oracle's eval_filtered reduced with alpha_k"""
    import plonky25_b200 as g
    from oracle_c import splitmix_columns
    log_n, r = 6, 3
    n, R = 1 << log_n, 1 << (log_n + r)
    nsel = len(groups)
    num_constants = nsel + 2
    wires = g.PolynomialBatch.from_values(list(splitmix_columns(700 + n_ch, N_WIRES, n)), r, False, 1, ctx=ctx)
    cs = g.PolynomialBatch.from_values(list(splitmix_columns(750 + n_ch, num_constants + 5, n)), r, False, 1, ctx=ctx)
    rnd = random.Random(60 + n_ch)
    alphas = [rnd.randrange(P) for _ in range(n_ch)]
    pi = [rnd.getrandbits(64) for _ in range(4)]
    offset = 5
    q = g.Quotient(wires, n_ch, ctx=ctx)
    assert q.add_gates(gates, g.SelectorsInfo(selectors, groups), cs, num_constants, pi, alphas, constraint_offset=offset) > 0
    acc = q.values()
    q.free()
    rows = sorted(set([0, R - 1] + [rnd.randrange(R) for _ in range(10)]))
    lw, lc = std._rows_at(wires, rows), std._rows_at(cs, rows)
    for j, row in enumerate(rows):
        w, k = lw[j].tolist(), lc[j].tolist()
        want = [0] * n_ch
        for i, (kind, param) in enumerate(gates):
            f = ro.compute_filter(i, groups[selectors[i]], k[selectors[i]], nsel > 1)
            c = _constraints(kind, param, w, k[nsel:num_constants], [x % P for x in pi])
            for ch in range(n_ch):
                want[ch] = (want[ch] + f * ro.reduce_with_powers(c, alphas[ch], offset)) % P
        assert [int(acc[ch, row]) for ch in range(n_ch)] == want, row
    wires.merkle_tree.free(); cs.merkle_tree.free()


@pytest.mark.gpu
@pytest.mark.parametrize("arities", [(4,), (2, 1)])
def test_fold_rows_of_a_device_fri_proof(ctx, arities):
    """the CosetInterpolationGate rows of every query step of a proof the device made (opening_set_pipeline.run_product) give all-zero
    constraints on the device, each evaluation value is the next step's evals[within] (or final_poly(x)), and a tampered eval does not
    give zero"""
    import plonky25_b200 as g
    import opening_set_pipeline as osp
    import wrapper_pipeline as wp
    log_n, r, h, pow_bits = 6, 3, 4, 4
    proof = osp.run_product(g, ctx, wp.make_columns(log_n), log_n, r=r, h=h, arities=arities, pow_bits=pow_bits, n_queries=6)
    ch = gl_oracle.Challenger()
    ch.observe_elements([int(v) for v in wp.PREFIX])
    for cap in proof["commit_caps"]:
        ch.observe_cap(cap.tolist())
    ch.get_extension_challenge()                                   # zeta
    for batch in proof["openings"]:
        for e in batch:
            ch.observe_extension_element((int(e[0]), int(e[1])))
    steps = [[[(int(e[0]), int(e[1])) for e in ev] for ev, _ in rnd["steps"]] for rnd in proof["query_rounds"]]
    final = [(int(c[0]), int(c[1])) for c in proof["final_poly"]]
    by_param = {}
    for param, row, nxt in fold_rows(ch, [c.tolist() for c in proof["commit_phase_caps"]], proof["query_indices"], steps, arities,
                                     log_n + r, final):
        lay = ro.coset_interpolation_layout(param)
        assert tuple(row[lay["value_out"]:lay["value_out"] + 2]) == nxt
        by_param.setdefault(param, []).append(row)
    assert sum(len(v) for v in by_param.values()) == 6 * len(arities)
    for param, rows in by_param.items():
        rows = np.array(rows, dtype=np.uint64)
        assert not g.evaluate_gate_constraints(CI, param, rows, ctx=ctx).any()
        bad = rows.copy()
        bad[:, 1] = (bad[:, 1] + np.uint64(1)) % np.uint64(P)     # component 0 of value 0: one eval of the coset
        out = g.evaluate_gate_constraints(CI, param, bad, ctx=ctx)
        assert out.any(axis=1).all()
        assert out.tolist() == [ro.gate_eval(CI, param, b.tolist()) for b in bad]


@pytest.mark.gpu
def test_error_paths(ctx):
    """every refused parameter and kind through every entry point returns its message and leaves the accumulator unchanged; the three
    gates go through gl_quotient_add_gate and gl_gate_eval_rows"""
    import plonky25_b200 as g
    from plonky25_b200 import _lib
    from oracle_c import splitmix_columns
    lib = ctx.lib
    wires = g.PolynomialBatch.from_values(list(splitmix_columns(23, N_WIRES, 16)), 3, False, 0, ctx=ctx)
    cs = g.PolynomialBatch.from_values(list(splitmix_columns(24, 8, 16)), 3, False, 0, ctx=ctx)
    q = g.Quotient(wires, 2, ctx=ctx)
    al = [5, 6]
    q.add_gate(CI, CI_4, al)
    q.add_gate(RED, 43, al, filter=(cs, 1))
    before = q.values()
    info = g.SelectorsInfo([0, 0, 1], [(0, 2), (2, 3)])
    pi = [1, 2, 3, 4]
    bad = [(14, 1, "unknown gate kind 14"), (18, 1, "unknown gate kind 18"), (22, 1, "unknown gate kind 22"),
           (26, 0, "unknown gate kind 26"), (CI, 5 | 2 << 8, f"parameter {5 | 2 << 8} out of range"),
           (CI, 4 | 1 << 8, f"parameter {4 | 1 << 8} out of range"), (CI, 3 | 9 << 8, f"parameter {3 | 9 << 8} out of range"),
           (CI, 6 | 8 << 8, f"parameter {6 | 8 << 8} out of range"), (CI, 0 | 2 << 8, f"parameter {2 << 8} out of range"),
           (CI, CI_4 | 1 << 16, f"parameter {CI_4 | 1 << 16} out of range"), (RED, 0, "parameter 0 out of range"),
           (RED, 44, "parameter 44 out of range"), (MDS, 1, "parameter 1 out of range")]
    for kind, param, msg in bad:
        with pytest.raises(ValueError, match=msg):
            q.add_gates([(kind, param), (ego.NOOP, 0), (ego.NOOP, 0)], info, cs, 4, pi, al)
        with pytest.raises(ValueError, match=msg):
            q.add_gate(kind, param, al)
        with pytest.raises(ValueError, match=msg):
            q.add_gate(kind, param, al, filter=(cs, 0))
        with pytest.raises(ValueError, match="unknown gate kind"):
            g.evaluate_gate_constraints(kind, param, np.zeros((1, 4), dtype=np.uint64), ctx=ctx)
        one = np.zeros(4, dtype=np.uint64)
        assert lib.gl_gate_eval_rows(ctx.handle, kind, param, one.ctypes.data, 1, one.ctypes.data) == _lib.GL_ERR_INVALID
        assert msg in lib.gl_ctx_last_error(ctx.handle).decode()
        assert lib.gl_gate_eval_rows_with_constants(ctx.handle, kind, param, one.ctypes.data, one.ctypes.data, one.ctypes.data, 1,
                                                    one.ctypes.data) == _lib.GL_ERR_INVALID
        assert msg in lib.gl_ctx_last_error(ctx.handle).decode()
    with pytest.raises(ValueError, match="parameter 44 out of range"):   # a refused gate after valid ones: nothing has launched
        q.add_gates([(CI, CI_4), (MDS, 0), (RED, 44)], info, cs, 4, pi, al)
    assert np.array_equal(q.values(), before)
    q.add_gates([(CI, CI_4), (MDS, 0), (RED, 43)], info, cs, 4, pi, al)
    assert not np.array_equal(q.values(), before)
    q.free()
    wires.merkle_tree.free(); cs.merkle_tree.free()


def _identity_holds(g, ctx, c, wires_cols, const_cols, alphas, betas, gammas, zeta, n_ch=2, r=3):
    """tests/test_plonky2_ext_gates.py · _identity_holds for this file's circuit: commit constants+sigmas, wires and Z / partial products;
    add_permutation, add_gates at offset n_ch (1 + n_chunks); commit the quotient; then the verifier's check
    Z_H(zeta) sum_c zeta^(cN) t_c(zeta) == the alpha-combination of the permutation terms and eval_filtered, from the polynomials at zeta"""
    import gates_oracle as go
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
    gate_terms = ro.eval_filtered(CIRCUIT_GATES, CIRCUIT_SELECTORS, CIRCUIT_GROUPS, ec, ew, pi)
    z_h = (pow(zeta, n, P) - 1) % P
    ok = True
    for ch in range(n_ch):
        t_zeta = 0
        for k in reversed(range(1 << r)):
            t_zeta = (t_zeta * pow(zeta, n, P) + std._eval_poly(ct[ch * (1 << r) + k], zeta)) % P
        ok &= z_h * t_zeta % P == ro.reduce_with_powers(perm + gate_terms, alphas[ch])
    for b in (sig, wires, zs_b, t):
        b.merkle_tree.free()
    return ok


@pytest.mark.gpu
@pytest.mark.parametrize("log_n", [5, 6])
def test_verifier_identity_for_a_recursion_circuit(ctx, log_n):
    """the quotient the device commits satisfies Z_H(zeta) t(zeta) = vanishing(zeta) at a random zeta for the valid circuit, and does not
    for a tampered coset value, a changed shift, a tampered Reducing coefficient or a tampered PoseidonMds output component"""
    import plonky25_b200 as g
    rnd = random.Random(30 + log_n)
    c = build_recursion_circuit(log_n, 70 + log_n)
    n_ch = 2
    alphas, betas, gammas = ([rnd.randrange(P) for _ in range(n_ch)] for _ in range(3))
    zeta = rnd.randrange(2, P)

    def holds(wires_cols):
        return _identity_holds(g, ctx, c, wires_cols, c["consts"], alphas, betas, gammas, zeta)

    def bumped(col, row):
        w = c["wires"].copy()
        w[col, row] = (int(w[col, row]) + 1) % P
        return w

    assert holds(c["wires"]), "Z_H(zeta) t(zeta) != vanishing(zeta) for a valid circuit"
    lay = ro.coset_interpolation_layout(CI_4)
    assert not holds(bumped(lay["value"][5], c["ci_row"]))            # component 0 of the coset value at x_5
    assert not holds(bumped(0, c["ci_row"]))                          # the shift
    assert not holds(bumped(6 + 7, c["red_row"]))                     # coefficient 7 of the Horner chain
    assert not holds(bumped(24 + 2 * 4 + 1, c["mds_row"]))            # component 1 of MDS output 4 (no copy cycle holds it)
