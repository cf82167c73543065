"""CPU oracle for plonky2's ArithmeticExtensionGate, MulExtensionGate and ReducingExtensionGate — TEST INFRASTRUCTURE ONLY.

Restated, parity unpinned: the upstream source (plonky2 @ 3de92d9, un-vendored) is not in this tree, so these functions are restated
from the published items, like plonky2_std_gates_oracle.py, whose names this module re-exports and whose shape() / gate_eval() /
eval_filtered() it extends with the three kinds.  D = 2: an extension value is two consecutive wires [a0, a1] of F_p[X]/(X^2 - 7)
(gl_oracle.ext_*), and every extension constraint is emitted as to_basefield_array(), component 0 first.

  arithmetic_extension_*    gates/arithmetic_extension.rs      ArithmeticExtensionGate { num_ops }: op i at wires 8i + [m0, m1, addend,
                            output]; output - ((m0 m1) k(0) + addend k(1))
  mul_extension_*           gates/multiplication_extension.rs  MulExtensionGate { num_ops }: op i at wires 6i + [m0, m1, output];
                            output - (m0 m1) k(0)
  reducing_extension_*      gates/reducing_extension.rs        ReducingExtensionGate { num_coeffs }: output 0, alpha 2, old_acc 4,
                            coefficient i at 6 + 2i, accumulator i at 6 + 2n + 2i (i < n - 1; accumulator n - 1 is the output);
                            acc alpha + coeff_i - acc_i from acc = old_acc

The witness side is the three generators: one extension multiply-add per op or coefficient.  What the tests check independently of
upstream: witness rows satisfy every constraint and any changed wire component or constant breaks one.
"""
import gl_oracle
import plonky2_std_gates_oracle as _std
from plonky2_std_gates_oracle import (ARITHMETIC, BASE_SUM, CONSTANT, EXPONENTIATION, NOOP, P, POSEIDON, PUBLIC_INPUT,  # noqa: F401
                                      RANDOM_ACCESS, UNUSED_SELECTOR, compute_filter, reduce_with_powers)

# include/gl_commit.h gate kinds (14 and 18 are not assigned)
ARITHMETIC_EXTENSION, MUL_EXTENSION, REDUCING_EXTENSION = 19, 20, 21
# (kind, new_from_config value at 135 wires / 80 routed, largest param the 135-wire shape takes)
CONFIG = {ARITHMETIC_EXTENSION: (10, 16), MUL_EXTENSION: (13, 22), REDUCING_EXTENSION: (32, 32)}


def shape(kind: int, param: int = 0):
    """(num_wires, num_constraints, num_constants) of any gate of plonky2_std_gates_oracle.shape and of the three kinds here"""
    if kind == ARITHMETIC_EXTENSION:
        return 8 * param, 2 * param, 2
    if kind == MUL_EXTENSION:
        return 6 * param, 2 * param, 1
    if kind == REDUCING_EXTENSION:
        return 4 + 4 * param, 2 * param, 0
    return _std.shape(kind, param)


def gate_eval(kind, param, w, k=(), pi_hash=(0, 0, 0, 0)):
    """eval_unfiltered of one row, for the kinds of plonky2_std_gates_oracle.gate_eval and the three kinds here"""
    if kind == ARITHMETIC_EXTENSION:
        return arithmetic_extension_eval(w, k, param)
    if kind == MUL_EXTENSION:
        return mul_extension_eval(w, k, param)
    if kind == REDUCING_EXTENSION:
        return reducing_extension_eval(w, param)
    return _std.gate_eval(kind, param, w, k, pi_hash)


def eval_filtered(gates, selector_indices, groups, constants_row, wires_row, pi_hash, num_lookup_selectors=0, constraint_evals=gate_eval):
    """plonky2_std_gates_oracle.eval_filtered with this module's gate_eval as the default constraint evaluator"""
    return _std.eval_filtered(gates, selector_indices, groups, constants_row, wires_row, pi_hash, num_lookup_selectors, constraint_evals)


def _ext(w, i):
    return int(w[i]) % P, int(w[i + 1]) % P


def _flat(exts):
    return [c for e in exts for c in e]


# ---- ArithmeticExtensionGate ----------------------------------------------------------------------------------------------------------
def arithmetic_extension_eval(w, k, num_ops):
    c0, c1 = int(k[0]) % P, int(k[1]) % P
    out = []
    for i in range(num_ops):
        m0, m1, add, o = (_ext(w, 8 * i + 2 * j) for j in range(4))
        computed = gl_oracle.ext_add(gl_oracle.ext_scale(gl_oracle.ext_mul(m0, m1), c0), gl_oracle.ext_scale(add, c1))
        out += list(gl_oracle.ext_sub(o, computed))
    return out


def arithmetic_extension_witness(ops, c0, c1):
    """ArithmeticExtensionGenerator: ops = (m0, m1, addend) extension triples -> [m0, m1, addend, (m0 m1) c0 + addend c1] per op"""
    rows = []
    for m0, m1, add in ops:
        out = gl_oracle.ext_add(gl_oracle.ext_scale(gl_oracle.ext_mul(m0, m1), c0 % P), gl_oracle.ext_scale(add, c1 % P))
        rows += [m0, m1, add, out]
    return [int(x) % P for x in _flat(rows)]


# ---- MulExtensionGate -----------------------------------------------------------------------------------------------------------------
def mul_extension_eval(w, k, num_ops):
    c0 = int(k[0]) % P
    out = []
    for i in range(num_ops):
        m0, m1, o = (_ext(w, 6 * i + 2 * j) for j in range(3))
        out += list(gl_oracle.ext_sub(o, gl_oracle.ext_scale(gl_oracle.ext_mul(m0, m1), c0)))
    return out


def mul_extension_witness(ops, c0):
    """MulExtensionGenerator: ops = (m0, m1) extension pairs -> [m0, m1, (m0 m1) c0] per op"""
    rows = []
    for m0, m1 in ops:
        rows += [m0, m1, gl_oracle.ext_scale(gl_oracle.ext_mul(m0, m1), c0 % P)]
    return [int(x) % P for x in _flat(rows)]


# ---- ReducingExtensionGate ------------------------------------------------------------------------------------------------------------
def reducing_extension_acc_wire(i, n):
    """the first wire of accumulator i: the output for i = n - 1"""
    return 0 if i == n - 1 else 6 + 2 * n + 2 * i


def reducing_extension_eval(w, n):
    alpha, acc = _ext(w, 2), _ext(w, 4)
    out = []
    for i in range(n):
        acc_i = _ext(w, reducing_extension_acc_wire(i, n))
        out += list(gl_oracle.ext_sub(gl_oracle.ext_add(gl_oracle.ext_mul(acc, alpha), _ext(w, 6 + 2 * i)), acc_i))
        acc = acc_i
    return out


def reducing_extension_witness(alpha, old_acc, coeffs):
    """ReducingGenerator: acc <- acc alpha + coeff_i from old_acc, every accumulator written; the last is the output"""
    n = len(coeffs)
    w = [0] * (4 + 4 * n)
    w[2:4], w[4:6] = alpha, old_acc
    acc = tuple(old_acc)
    for i, c in enumerate(coeffs):
        w[6 + 2 * i:8 + 2 * i] = c
        acc = gl_oracle.ext_add(gl_oracle.ext_mul(acc, alpha), c)
        a = reducing_extension_acc_wire(i, n)
        w[a:a + 2] = acc
    return [int(x) % P for x in w]
