"""CPU oracle for plonky2's PoseidonGate, ExponentiationGate and RandomAccessGate — TEST INFRASTRUCTURE ONLY.

Restated, parity unpinned: the upstream source (plonky2 @ 3de92d9, un-vendored) is not in this tree, so these functions are restated
from the published items, like oracle/plonky2_gates_oracle.py, whose names this module re-exports and whose shape() / gate_eval() it
extends with the three kinds:

  poseidon_gate_*           gates/poseidon.rs             PoseidonGate: 135 wires, 123 constraints, the naive-form rounds of
                            gl_oracle.poseidon with an S-box input wire substituted at every stored S-box input
  exponentiation_*          gates/exponentiation.rs       ExponentiationGate { num_power_bits }: square-and-multiply, bits big-endian
  random_access_*           gates/random_access.rs        RandomAccessGate { bits, num_copies, num_extra_constants }: the list
                            folded pairwise by the index bits, plus extra constants

What the tests check independently of upstream: PoseidonGate witness outputs are gl_oracle.poseidon (pinned by the four KATs), witness
rows satisfy every constraint, and a tampered wire, bit or constant breaks one.
"""
import gl_oracle
import plonky2_gates_oracle as _core
from plonky2_gates_oracle import (ARITHMETIC, BASE_SUM, CONSTANT, NOOP, P, PUBLIC_INPUT, UNUSED_SELECTOR, arithmetic_witness,  # noqa: F401
                                  base_sum_witness, compute_filter, constant_witness, eval_filtered, public_input_witness,
                                  reduce_with_powers)

# include/gl_commit.h gate kinds
POSEIDON, EXPONENTIATION, RANDOM_ACCESS = 15, 16, 17


def shape(kind: int, param: int = 0):
    """(num_wires, num_constraints, num_constants) of any gate of plonky2_gates_oracle.shape and of the three kinds here"""
    if kind == POSEIDON:
        return POSEIDON_NUM_WIRES, POSEIDON_NUM_CONSTRAINTS, 0
    if kind == EXPONENTIATION:
        return 2 + 2 * param, param + 1, 0
    if kind == RANDOM_ACCESS:
        bits, copies, extras = random_access_fields(param)
        return (2 + (1 << bits) + bits) * copies + extras, (bits + 2) * copies + extras, extras
    return _core.shape(kind, param)


def gate_eval(kind, param, w, k=(), pi_hash=(0, 0, 0, 0)):
    """eval_unfiltered of one row, for the kinds of plonky2_gates_oracle.gate_eval and the three kinds here"""
    if kind == POSEIDON:
        return poseidon_gate_eval(w)
    if kind == EXPONENTIATION:
        return exponentiation_eval(w, param)
    if kind == RANDOM_ACCESS:
        return random_access_eval(w, k, param)
    return _core.gate_eval(kind, param, w, k, pi_hash)


# ---- PoseidonGate (gates/poseidon.rs): wire layout ----------------------------------------------------------------------------------
POSEIDON_WIRE_SWAP, POSEIDON_START_DELTA, POSEIDON_START_FULL_0 = 24, 25, 29
POSEIDON_START_PARTIAL = POSEIDON_START_FULL_0 + 12 * 3          # 65
POSEIDON_START_FULL_1 = POSEIDON_START_PARTIAL + 22              # 87
POSEIDON_NUM_WIRES = POSEIDON_START_FULL_1 + 12 * 4              # 135
POSEIDON_NUM_CONSTRAINTS = 1 + 4 + 12 * 3 + 22 + 12 * 4 + 12     # 123


def _poseidon_rounds(state, at):
    """gl_oracle.poseidon (naive form) from the swapped input state; at(wire, v) -> the value the S-box takes for every stored S-box
    input (upstream writes the partial rounds in the "fast" form, whose lane-0 S-box inputs are the same values)"""
    rc, s = gl_oracle.ALL_ROUND_CONSTANTS, list(state)
    for r in range(30):
        s = [(x + rc[12 * r + i]) % P for i, x in enumerate(s)]
        if r < 4 or r >= 26:
            for i in range(12):
                if r != 0:
                    s[i] = at((POSEIDON_START_FULL_0 + 12 * (r - 1) if r < 4 else POSEIDON_START_FULL_1 + 12 * (r - 26)) + i, s[i])
                s[i] = pow(s[i], 7, P)
        else:
            s[0] = pow(at(POSEIDON_START_PARTIAL + r - 4, s[0]), 7, P)
        s = gl_oracle._mds_layer(s)
    return s


def poseidon_gate_eval(w):
    """eval_unfiltered: swap(swap - 1), swap (rhs - lhs) - delta_i, then (computed - wire) at every stored S-box input, then outputs"""
    w = [int(x) % P for x in w]
    swap = w[POSEIDON_WIRE_SWAP]
    out = [swap * (swap - 1) % P]
    s = list(w[:12])
    for i in range(4):
        d = w[POSEIDON_START_DELTA + i]
        out.append((swap * (w[i + 4] - w[i]) - d) % P)
        s[i], s[i + 4] = (w[i] + d) % P, (w[i + 4] - d) % P

    def at(wire, v):
        out.append((v - w[wire]) % P)
        return w[wire]
    s = _poseidon_rounds(s, at)
    out += [(s[i] - w[12 + i]) % P for i in range(12)]
    return out


def poseidon_gate_witness(inputs, swap):
    """PoseidonGenerator::run_once, every wire of the row: inputs, outputs, swap, deltas, S-box inputs"""
    st = [int(x) % P for x in inputs]
    swap = int(swap) % P
    w = [0] * POSEIDON_NUM_WIRES
    w[:12], w[POSEIDON_WIRE_SWAP] = st, swap
    for i in range(4):
        w[POSEIDON_START_DELTA + i] = swap * (st[i + 4] - st[i]) % P
    if swap == 1:
        st = st[4:8] + st[:4] + st[8:]

    def at(wire, v):
        w[wire] = v
        return v
    w[12:24] = _poseidon_rounds(st, at)
    return w


# ---- ExponentiationGate (gates/exponentiation.rs) -------------------------------------------------------------------------------------
def exponentiation_max_power_bits(num_wires=135, num_routed=80):
    """ExponentiationGate::max_power_bits: base and output are routed"""
    return min(num_routed - 2, (num_wires - 2) // 2)


def exponentiation_eval(w, n):
    w = [int(x) % P for x in w]
    base, bits, output, inter = w[0], w[1:1 + n], w[1 + n], w[2 + n:2 + 2 * n]
    out = []
    for i in range(n):
        prev = 1 if i == 0 else inter[i - 1] * inter[i - 1] % P
        b = bits[n - 1 - i]                    # power bits are little-endian, accumulated big-endian
        out.append((prev * (b * base + 1 - b) - inter[i]) % P)
    out.append((output - inter[n - 1]) % P)
    return out


def exponentiation_witness(base, power, n):
    """ExponentiationGenerator: [base, bits (LE), output, intermediates]; power < 2^n"""
    assert 0 <= power < 1 << n
    bits = [(power >> i) & 1 for i in range(n)]
    inter, cur = [], 1
    for i in range(n):
        if bits[n - 1 - i]:
            cur = cur * base % P
        inter.append(cur)
        cur = cur * cur % P
    return [base % P] + bits + [inter[-1]] + inter


# ---- RandomAccessGate (gates/random_access.rs) ----------------------------------------------------------------------------------------
def random_access_fields(param):
    """(bits, num_copies, num_extra_constants) of a GATE_RANDOM_ACCESS param"""
    return param & 0xFF, (param >> 8) & 0xFF, param >> 16


def random_access_params(bits, num_wires=135, num_routed=80, num_constants=2):
    """RandomAccessGate::new_from_config(config, bits) as a param"""
    v = 1 << bits
    copies = min(num_routed // (2 + v), num_wires // (2 + v + bits))
    extras = min(num_routed - (2 + v) * copies, num_constants)
    return bits | copies << 8 | extras << 16


def random_access_eval(w, k, param):
    bits, copies, extras = random_access_fields(param)
    v = 1 << bits
    w = [int(x) % P for x in w]
    routed = (2 + v) * copies + extras
    out = []
    for c in range(copies):
        index, claimed = w[(2 + v) * c], w[(2 + v) * c + 1]
        items = w[(2 + v) * c + 2:(2 + v) * c + 2 + v]
        bs = w[routed + c * bits:routed + (c + 1) * bits]
        out += [b * (b - 1) % P for b in bs]
        acc = 0
        for b in reversed(bs):
            acc = (2 * acc + b) % P
        out.append((acc - index) % P)
        for b in bs:                           # fold pairs (x, y) -> x + b (y - x)
            items = [(items[j] + b * (items[j + 1] - items[j])) % P for j in range(0, len(items), 2)]
        out.append((items[0] - claimed) % P)
    out += [(int(k[i]) - w[(2 + v) * copies + i]) % P for i in range(extras)]
    return out


def random_access_witness(copies, extra_constants, param):
    """copies: [(index, list of 2^bits items)] per copy; extra_constants: the row's gate constants -> the row's wires"""
    bits, n_copies, extras = random_access_fields(param)
    v = 1 << bits
    assert len(copies) == n_copies and len(extra_constants) == extras
    w = []
    for index, items in copies:
        assert 0 <= index < v and len(items) == v
        w += [index, int(items[index]) % P] + [int(x) % P for x in items]
    w += [int(x) % P for x in extra_constants]
    for index, _ in copies:
        w += [(index >> i) & 1 for i in range(bits)]
    return w
