"""CPU oracle for plonky2's core gates and the selector filters of evaluate_gate_constraints — TEST INFRASTRUCTURE ONLY.

Restated, parity unpinned: the upstream source (plonky2 @ 3de92d9, un-vendored) is not in this tree, so these functions are restated
from the published items, not transcribed next to their source as gates_oracle.py is:

  compute_filter()          plonky2 gates/gate.rs · compute_filter (UNUSED_SELECTOR = u32::MAX from gates/selectors.rs)
  eval_filtered()           gates/gate.rs · eval_filtered_base_batch + plonk/vanishing_poly.rs · evaluate_gate_constraints_base_batch
                            at one point: sum over gates of filter_i * constraints_i, by constraint index
  noop                      gates/noop.rs                 0 wires, 0 constraints
  constant_*                gates/constant.rs             ConstantGate { num_consts }: local_constants[i] - local_wires[i]
  public_input_*            gates/public_input.rs         local_wires[i] - public_inputs_hash[i], i < 4
  arithmetic_*              gates/arithmetic_base.rs      ArithmeticGate { num_ops }: per op, output - (c0 m0 m1 + c1 addend)
  base_sum_*                gates/base_sum.rs             BaseSumGate<B> { num_limbs }: sum(limb_j B^j) - sum, prod_{v<B}(limb - v)

What the tests check independently of upstream: witness rows satisfy every constraint and a tampered wire, constant or hash word breaks
one; the filter of gate i vanishes at every other selector value of its group (and at UNUSED_SELECTOR); a circuit of mixed gates has a
filtered constraint sum that vanishes on H, and the device's quotient satisfies the verifier's identity at a random point.
"""
from typing import List, Sequence, Tuple

P = 0xFFFF_FFFF_0000_0001
UNUSED_SELECTOR = (1 << 32) - 1

# include/gl_commit.h gate kinds
NOOP, CONSTANT, PUBLIC_INPUT, ARITHMETIC, BASE_SUM = 9, 10, 11, 12, 13


def compute_filter(i: int, group: Tuple[int, int], s: int, many_selectors: bool) -> int:
    """prod_{j in group, j != i} (j - s), times (UNUSED_SELECTOR - s) when there is more than one selector"""
    f = 1
    js = [j for j in range(group[0], group[1]) if j != i] + ([UNUSED_SELECTOR] if many_selectors else [])
    for j in js:
        f = f * ((j - s) % P) % P
    return f


# ---- gates: (num_wires, num_constraints, num_constants), eval(wires, consts, pi_hash) -> constraints, witness fill ---------------------
def shape(kind: int, param: int = 0) -> Tuple[int, int, int]:
    if kind == NOOP:
        return 0, 0, 0
    if kind == CONSTANT:
        return param, param, param
    if kind == PUBLIC_INPUT:
        return 4, 4, 0
    if kind == ARITHMETIC:
        return 4 * param, param, 2
    if kind == BASE_SUM:
        n = param & 0xFF
        return 1 + n, 1 + n, 0
    raise ValueError(kind)


def constant_eval(w, k, num_consts):
    return [(int(k[i]) - int(w[i])) % P for i in range(num_consts)]


def public_input_eval(w, pi_hash):
    return [(int(w[i]) - int(pi_hash[i])) % P for i in range(4)]


def arithmetic_eval(w, k, num_ops):
    c0, c1 = int(k[0]) % P, int(k[1]) % P
    out = []
    for i in range(num_ops):
        m0, m1, add, o = (int(x) % P for x in w[4 * i:4 * i + 4])
        out.append((o - (m0 * m1 % P * c0 + add * c1)) % P)
    return out


def base_sum_eval(w, num_limbs, base):
    w = [int(x) % P for x in w]
    limbs = w[1:1 + num_limbs]
    acc = 0
    for limb in reversed(limbs):                       # reduce_with_powers(limbs, B)
        acc = (acc * base + limb) % P
    out = [(acc - w[0]) % P]
    for limb in limbs:
        prod = 1
        for v in range(base):
            prod = prod * ((limb - v) % P) % P
        out.append(prod)
    return out


def gate_eval(kind: int, param: int, w: Sequence[int], k: Sequence[int] = (), pi_hash: Sequence[int] = (0, 0, 0, 0)) -> List[int]:
    """eval_unfiltered of one row: w = the gate's wires, k = its constants (after the selector columns), pi_hash = 4 words"""
    if kind == NOOP:
        return []
    if kind == CONSTANT:
        return constant_eval(w, k, param)
    if kind == PUBLIC_INPUT:
        return public_input_eval(w, pi_hash)
    if kind == ARITHMETIC:
        return arithmetic_eval(w, k, param)
    if kind == BASE_SUM:
        return base_sum_eval(w, param & 0xFF, param >> 8)
    raise ValueError(kind)


def constant_witness(consts):
    """ConstantGate's generator: wire i <- constant i"""
    return [int(c) % P for c in consts]


def public_input_witness(pi_hash):
    return [int(x) % P for x in pi_hash]


def arithmetic_witness(ops, c0, c1):
    """ops: (m0, m1, addend) per op -> [m0, m1, addend, c0 m0 m1 + c1 addend] per op"""
    w = []
    for m0, m1, add in ops:
        w += [m0 % P, m1 % P, add % P, (c0 * m0 % P * m1 + c1 * add) % P]
    return w


def base_sum_witness(value, num_limbs, base):
    """value < base^num_limbs -> [value, limb_0, .., limb_{n-1}] (little-endian digits)"""
    limbs = []
    v = value
    for _ in range(num_limbs):
        limbs.append(v % base)
        v //= base
    assert v == 0, "value does not fit in num_limbs digits"
    return [value % P] + limbs


def reduce_with_powers(terms: Sequence[int], alpha: int, start_power: int = 0) -> int:
    acc, pw = 0, pow(alpha, start_power, P)
    for t in terms:
        acc = (acc + t * pw) % P
        pw = pw * alpha % P
    return acc


def eval_filtered(gates, selector_indices, groups, constants_row, wires_row, pi_hash, num_lookup_selectors, constraint_evals):
    """evaluate_gate_constraints at one point: res[c] = sum_i compute_filter(i, group_i, s_i, many) * constraints_i[c].
    gates: [(kind, param)]; groups: [(start, end)] per selector; constants_row: the opened constants (selectors first);
    constraint_evals(kind, param, wires, consts, pi_hash) -> constraints of one gate (lets callers add the reference's own gates)."""
    num_selectors = len(groups)
    k0 = num_selectors + num_lookup_selectors
    res: List[int] = []
    for i, (kind, param) in enumerate(gates):
        s_idx = selector_indices[i]
        f = compute_filter(i, groups[s_idx], int(constants_row[s_idx]) % P, num_selectors > 1)
        cs = constraint_evals(kind, param, wires_row, list(constants_row[k0:]), pi_hash)
        if len(cs) > len(res):
            res += [0] * (len(cs) - len(res))
        for c, v in enumerate(cs):
            res[c] = (res[c] + f * v) % P
    return res
