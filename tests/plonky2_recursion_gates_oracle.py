"""CPU oracle for plonky2's CosetInterpolationGate, ReducingGate and PoseidonMdsGate — TEST INFRASTRUCTURE ONLY.

Restated, parity unpinned: the upstream source (plonky2 @ 3de92d9, un-vendored) is not in this tree, so these functions are restated
from the published items, like plonky2_ext_gates_oracle.py, whose names this module re-exports and whose shape() / gate_eval() /
eval_filtered() it extends with the three kinds.  They are the gates plonky2's recursive verifier circuit registers besides the ones
already on the device.  D = 2: an extension value is two consecutive wires [a0, a1] of F_p[X]/(X^2 - 7), and every extension constraint is
emitted as to_basefield_array(), component 0 first.

  coset_interpolation_*   gates/coset_interpolation.rs   CosetInterpolationGate { subgroup_bits, degree }: n = 2^subgroup_bits values,
                          k = (n - 2) / (degree - 1) intermediate (eval, prod) pairs.  Wires: shift 0, value i at 1 + 2i, evaluation point
                          1 + 2n, evaluation value 3 + 2n, s = 5 + 2n: intermediate eval i at s + 2i, intermediate prod i at s + 2(k + i),
                          shifted evaluation point s + 4k.  The weights are barycentric_weights' literal product-and-inverse form over
                          the domain of primitive_root_of_unity(subgroup_bits)
  reducing_*              gates/reducing.rs              ReducingGate { num_coeffs }: output 0, alpha 2, old_acc 4, base coefficient i at
                          6 + i, accumulator i at 6 + m + 2i (i < m - 1; accumulator m - 1 is the output); acc alpha + coeff_i - acc_i
  poseidon_mds_*          gates/poseidon_mds.rs          PoseidonMdsGate: ext input i at 2i, ext output i at 24 + 2i; the Poseidon MDS
                          layer (gl_oracle.MDS_CIRC / MDS_DIAG) applied to each component

What the tests check independently of upstream: witness rows satisfy every constraint, any changed wire component breaks one, the
CosetInterpolation evaluation value is the interpolant of fri_verifier.compute_evaluation, and PoseidonMds on base inputs is
gl_oracle._mds_layer.
"""
import gl_oracle
import plonky2_ext_gates_oracle as _ext
from plonky2_ext_gates_oracle import (ARITHMETIC, ARITHMETIC_EXTENSION, BASE_SUM, CONSTANT, EXPONENTIATION, MUL_EXTENSION, NOOP, P,  # noqa: F401
                                      POSEIDON, PUBLIC_INPUT, RANDOM_ACCESS, REDUCING_EXTENSION, UNUSED_SELECTOR, compute_filter,
                                      reduce_with_powers)

# include/gl_commit.h gate kinds (14, 18 and 22 are not assigned)
COSET_INTERPOLATION, REDUCING, POSEIDON_MDS = 23, 24, 25
REDUCING_MAX = 43                 # ReducingGate::max_coeffs_len(135, 80) = min((135 - 4) / 3, 80 - 6)


def coset_interpolation_params(subgroup_bits, max_degree=8):
    """CosetInterpolationGate::with_max_degree as (subgroup_bits | degree << 8)"""
    n = 1 << subgroup_bits
    k = (n - 2) // (max_degree - 1)
    return subgroup_bits | ((n - 2) // (k + 1) + 2) << 8


def coset_interpolation_fields(param):
    """(subgroup_bits, degree, n, num_intermediates)"""
    bits, degree = param & 0xFF, param >> 8
    n = 1 << bits
    return bits, degree, n, (n - 2) // (degree - 1)


def shape(kind: int, param: int = 0):
    """(num_wires, num_constraints, num_constants) of any gate of plonky2_ext_gates_oracle.shape and of the three kinds here"""
    if kind == COSET_INTERPOLATION:
        _, _, n, k = coset_interpolation_fields(param)
        return 7 + 2 * n + 4 * k, 4 + 4 * k, 0
    if kind == REDUCING:
        return 4 + 3 * param, 2 * param, 0
    if kind == POSEIDON_MDS:
        return 48, 24, 0
    return _ext.shape(kind, param)


def gate_eval(kind, param, w, k=(), pi_hash=(0, 0, 0, 0)):
    """eval_unfiltered of one row, for the kinds of plonky2_ext_gates_oracle.gate_eval and the three kinds here"""
    if kind == COSET_INTERPOLATION:
        return coset_interpolation_eval(w, param)
    if kind == REDUCING:
        return reducing_eval(w, param)
    if kind == POSEIDON_MDS:
        return poseidon_mds_eval(w)
    return _ext.gate_eval(kind, param, w, k, pi_hash)


def eval_filtered(gates, selector_indices, groups, constants_row, wires_row, pi_hash, num_lookup_selectors=0, constraint_evals=gate_eval):
    """plonky2_ext_gates_oracle.eval_filtered with this module's gate_eval as the default constraint evaluator"""
    return _ext.eval_filtered(gates, selector_indices, groups, constants_row, wires_row, pi_hash, num_lookup_selectors, constraint_evals)


def _ext_at(w, i):
    return int(w[i]) % P, int(w[i + 1]) % P


# ---- CosetInterpolationGate -----------------------------------------------------------------------------------------------------------
def coset_interpolation_layout(param):
    """first wire of each item: dict(value=[...], point, value_out, int_eval=[...], int_prod=[...], shifted)"""
    _, _, n, k = coset_interpolation_fields(param)
    s = 5 + 2 * n
    return {"value": [1 + 2 * i for i in range(n)], "point": 1 + 2 * n, "value_out": 3 + 2 * n,
            "int_eval": [s + 2 * i for i in range(k)], "int_prod": [s + 2 * (k + i) for i in range(k)], "shifted": s + 4 * k}


def coset_domain(subgroup_bits):
    g = gl_oracle.primitive_root_of_unity(subgroup_bits)
    return [pow(g, i, P) for i in range(1 << subgroup_bits)]


def barycentric_weights(xs):
    """interpolation.rs · barycentric_weights: 1 / prod_{j != i} (x_i - x_j), the product formed and inverted"""
    out = []
    for i, xi in enumerate(xs):
        d = 1
        for j, xj in enumerate(xs):
            if j != i:
                d = d * (xi - xj) % P
        out.append(gl_oracle.inv(d))
    return out


def coset_chunks(param):
    """the domain ranges partial_interpolate runs over: [0, degree), then [1 + (degree - 1)(i + 1), min(+ degree - 1, n)) for i < k"""
    _, degree, n, k = coset_interpolation_fields(param)
    out = [(0, degree)]
    for i in range(k):
        start = 1 + (degree - 1) * (i + 1)
        out.append((start, min(start + degree - 1, n)))
    return out


def partial_interpolate(xs, values, weights, z, eval_, prod):
    """interpolation.rs · partial_interpolate(_ext_algebra): t = z - x_i; eval <- eval t + (v_i w_i) prod; prod <- prod t"""
    for x, v, wt in zip(xs, values, weights):
        t = gl_oracle.ext_sub(z, (x, 0))
        eval_ = gl_oracle.ext_add(gl_oracle.ext_mul(eval_, t), gl_oracle.ext_mul(gl_oracle.ext_scale(v, wt), prod))
        prod = gl_oracle.ext_mul(prod, t)
    return eval_, prod


def coset_interpolation_eval(w, param):
    bits, _, _, k = coset_interpolation_fields(param)
    lay = coset_interpolation_layout(param)
    xs = coset_domain(bits)
    wts = barycentric_weights(xs)
    shift, z = int(w[0]) % P, _ext_at(w, lay["shifted"])
    vals = [_ext_at(w, a) for a in lay["value"]]
    out = list(gl_oracle.ext_sub(_ext_at(w, lay["point"]), gl_oracle.ext_scale(z, shift)))
    chunks = coset_chunks(param)
    a, b = chunks[0]
    ev, pr = partial_interpolate(xs[a:b], vals[a:b], wts[a:b], z, (0, 0), (1, 0))
    for i in range(k):
        ie, ip = _ext_at(w, lay["int_eval"][i]), _ext_at(w, lay["int_prod"][i])
        out += list(gl_oracle.ext_sub(ie, ev)) + list(gl_oracle.ext_sub(ip, pr))
        a, b = chunks[i + 1]
        ev, pr = partial_interpolate(xs[a:b], vals[a:b], wts[a:b], z, ie, ip)
    return out + list(gl_oracle.ext_sub(_ext_at(w, lay["value_out"]), ev))


def coset_interpolation_witness(param, shift, values, point):
    """InterpolationGenerator: shifted point = point / shift, every intermediate (eval, prod) written, the evaluation value last"""
    bits, _, n, k = coset_interpolation_fields(param)
    assert len(values) == n and shift % P
    lay = coset_interpolation_layout(param)
    w = [0] * shape(COSET_INTERPOLATION, param)[0]
    w[0] = shift % P
    for a, v in zip(lay["value"], values):
        w[a:a + 2] = v
    w[lay["point"]:lay["point"] + 2] = point
    z = gl_oracle.ext_scale(point, gl_oracle.inv(shift % P))
    w[lay["shifted"]:lay["shifted"] + 2] = z
    xs = coset_domain(bits)
    wts = barycentric_weights(xs)
    ev, pr = (0, 0), (1, 0)
    for i, (a, b) in enumerate(coset_chunks(param)):
        if i:
            w[lay["int_eval"][i - 1]:lay["int_eval"][i - 1] + 2] = ev
            w[lay["int_prod"][i - 1]:lay["int_prod"][i - 1] + 2] = pr
        ev, pr = partial_interpolate(xs[a:b], values[a:b], wts[a:b], z, ev, pr)
    w[lay["value_out"]:lay["value_out"] + 2] = ev
    return [int(x) % P for x in w]


# ---- ReducingGate ---------------------------------------------------------------------------------------------------------------------
def reducing_acc_wire(i, m):
    """the first wire of accumulator i: the output for i = m - 1"""
    return 0 if i == m - 1 else 6 + m + 2 * i


def reducing_eval(w, m):
    alpha, acc = _ext_at(w, 2), _ext_at(w, 4)
    out = []
    for i in range(m):
        acc_i = _ext_at(w, reducing_acc_wire(i, m))
        out += list(gl_oracle.ext_sub(gl_oracle.ext_add(gl_oracle.ext_mul(acc, alpha), (int(w[6 + i]) % P, 0)), acc_i))
        acc = acc_i
    return out


def reducing_witness(alpha, old_acc, coeffs):
    """ReducingGenerator with base coefficients: acc <- acc alpha + coeff_i from old_acc, every accumulator written; the last is the output"""
    m = len(coeffs)
    w = [0] * (4 + 3 * m)
    w[2:4], w[4:6] = alpha, old_acc
    acc = tuple(old_acc)
    for i, c in enumerate(coeffs):
        w[6 + i] = c
        acc = gl_oracle.ext_add(gl_oracle.ext_mul(acc, alpha), (c % P, 0))
        a = reducing_acc_wire(i, m)
        w[a:a + 2] = acc
    return [int(x) % P for x in w]


# ---- PoseidonMdsGate ------------------------------------------------------------------------------------------------------------------
def poseidon_mds_ext(inputs):
    """mds_layer_algebra: output i = sum_j CIRC[j] in_{(i + j) % 12} + DIAG[i] in_i, the constants as base scalars"""
    out = []
    for i in range(12):
        acc = gl_oracle.ext_scale(inputs[i], gl_oracle.MDS_DIAG[i])
        for j in range(12):
            acc = gl_oracle.ext_add(acc, gl_oracle.ext_scale(inputs[(i + j) % 12], gl_oracle.MDS_CIRC[j]))
        out.append(acc)
    return out


def poseidon_mds_eval(w):
    want = poseidon_mds_ext([_ext_at(w, 2 * i) for i in range(12)])
    out = []
    for i in range(12):
        out += list(gl_oracle.ext_sub(_ext_at(w, 24 + 2 * i), want[i]))
    return out


def poseidon_mds_witness(inputs):
    """PoseidonMdsGenerator: the 12 extension inputs, then their MDS layer"""
    return [int(c) % P for e in list(inputs) + poseidon_mds_ext(inputs) for c in e]
