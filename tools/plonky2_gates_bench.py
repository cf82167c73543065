"""Device time of plonky2's PoseidonGate, ExponentiationGate(66), RandomAccessGate(bits 4, 4 copies, 2 extra constants) and of the
extension-field gates ArithmeticExtensionGate(10), MulExtensionGate(13) and ReducingExtensionGate(32), and of the recursive verifier's
CosetInterpolationGate(4, 6), ReducingGate(43) and PoseidonMdsGate in gl_quotient_add_gates at the wrapper shape, and of the PoseidonGate
witness generator; prints one JSON line (and writes it to --out).

    python tools/plonky2_gates_bench.py [--repeats 20] [--warmup 3] [--out FILE]

Shape (as tools/quotient_gates_bench.py): N = 2^16, rate_bits 3 (R = 2^19 LDE rows), a 135-column wires commit, a constants/sigmas commit
with 5 selectors, 2 gate constants and 80 sigmas, 2 challenges.  Gate list [Poseidon] [Poseidon2] [Exponentiation(66), RandomAccess]
[ArithmeticExtension(10), Arithmetic(20), MulExtension(13), ReducingExtension(32)] [CosetInterpolation(4, 6), Reducing(43), PoseidonMds]
in 5 selector groups.
  per_gate_ms         one add_gates call with every other gate replaced by NoopGate: one launch, median over the repeats.  PoseidonGate
                      and Poseidon2Gate (same wires, same constraint count) are run alternately in the same process, and so are
                      ArithmeticExtensionGate(10) and ArithmeticGate(20) (both 80 routed wires and 20 constraints: the pair shows
                      what the extension product costs).
  witness_ms          gl_poseidon_gate_witness and gl_poseidon2_gate_witness for 2^16 rows, alternately (kernel time, CUDA events).
  parity              the accumulator of each gate's first timed launch equals the oracle's eval_filtered (reduced with the two alphas)
                      at 64 sampled LDE rows, and the timed PoseidonGate witness rows' outputs equal Context.poseidon_permute of the
                      swapped inputs.
The GPU's name and power limit are read in the same run.  Needs a CUDA device: there is no CPU fallback.
"""
import argparse
import json
import os
import random
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import plonky25_b200 as g  # noqa: E402
import gates_oracle as go  # noqa: E402
import plonky2_recursion_gates_oracle as pgo  # noqa: E402
from oracle_c import splitmix_columns  # noqa: E402
from quotient_gates_bench import gpu_info  # noqa: E402

P = g.api.P
LOG_N, RATE_BITS, N_CH, WITNESS_ROWS = 16, 3, 2, 1 << 16
GATES = [("poseidon", g.GATE_POSEIDON, 0), ("poseidon2", g.GATE_POSEIDON2, 0), ("exponentiation_66", g.GATE_EXPONENTIATION, 66),
         ("random_access_4x4_2", g.GATE_RANDOM_ACCESS, g.random_access_params(4)),
         ("arithmetic_extension_10", g.GATE_ARITHMETIC_EXTENSION, 10), ("arithmetic_20", g.GATE_ARITHMETIC, 20),
         ("mul_extension_13", g.GATE_MUL_EXTENSION, 13), ("reducing_extension_32", g.GATE_REDUCING_EXTENSION, 32),
         ("coset_interpolation_4_6", g.GATE_COSET_INTERPOLATION, g.coset_interpolation_params(4)), ("reducing_43", g.GATE_REDUCING, 43),
         ("poseidon_mds", g.GATE_POSEIDON_MDS, 0)]
GROUPS = [(0, 1), (1, 2), (2, 4), (4, 8), (8, 11)]
SELECTORS = [0, 1, 2, 2, 3, 3, 3, 3, 4, 4, 4]
NUM_CONSTANTS = len(GROUPS) + 2


def constraints(kind, param, w, k, pi):
    return go.poseidon2_gate_eval(w) if kind == g.GATE_POSEIDON2 else pgo.gate_eval(kind, param, w, k, pi)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out")
    args = ap.parse_args()
    ctx = g.Context(0)
    n = 1 << LOG_N
    R = n << RATE_BITS
    wires = g.PolynomialBatch.from_values(list(splitmix_columns(1, 135, n)), RATE_BITS, False, 4, ctx=ctx)
    cs = g.PolynomialBatch.from_values(list(splitmix_columns(2, NUM_CONSTANTS + 80, n)), RATE_BITS, False, 4, ctx=ctx)
    info = g.SelectorsInfo(SELECTORS, GROUPS)
    alphas = [0x1234_5678_9ABC_DEF0 % P, 0x0FED_CBA9_8765_4321 % P]
    pi = [11, 22, 33, 44]
    noop = (g.GATE_NOOP, 0)
    only = [[(k, p) if j == i else noop for j, (_, k, p) in enumerate(GATES)] for i in range(len(GATES))]
    q = g.Quotient(wires, N_CH, ctx=ctx)

    # parity of the first timed launch of every gate (fresh accumulator) against the oracle at 64 sampled rows
    rnd = random.Random(5)
    rows = sorted(rnd.sample(range(R), 64))
    lw, lc = wires.merkle_tree.open_batch(rows)[0], cs.merkle_tree.open_batch(rows)[0]
    t_gate = {name: [] for name, _, _ in GATES}
    parity = True
    for i, (name, kind, param) in enumerate(GATES):
        qi = g.Quotient(wires, N_CH, ctx=ctx)
        t_gate[name].append(qi.add_gates(only[i], info, cs, NUM_CONSTANTS, pi, alphas))
        acc = qi.values()
        qi.free()
        for j, row in enumerate(rows):
            terms = pgo.eval_filtered(only[i], SELECTORS, GROUPS, lc[j].tolist(), lw[j].tolist(), pi, 0, constraints)
            parity &= [int(acc[ch, row]) for ch in range(N_CH)] == [pgo.reduce_with_powers(terms, a) for a in alphas]

    # witness inputs: random states, half of them swapped
    wr = random.Random(6)
    ins = np.array([[wr.randrange(P) for _ in range(12)] + [wr.randrange(2)] for _ in range(WITNESS_ROWS)], dtype=np.uint64)
    swapped = ins[:, :12].copy()
    sw = ins[:, 12] == 1
    swapped[sw, :4], swapped[sw, 4:8] = ins[sw, 4:8], ins[sw, :4]
    want_out = ctx.poseidon_permute(swapped)

    def witness(fn):
        rows_out = fn(ins, ctx=ctx)
        import ctypes
        ms = ctypes.c_float()
        ctx.lib.gl_ctx_aux_ms(ctx.handle, ctypes.byref(ms))
        return rows_out, ms.value

    for _ in range(args.warmup):
        for i in range(len(GATES)):
            q.add_gates(only[i], info, cs, NUM_CONSTANTS, pi, alphas)
        witness(g.poseidon_gate_witness); witness(g.poseidon2_gate_witness)
    t_wit = {"poseidon": [], "poseidon2": []}
    for _ in range(args.repeats):
        for i, (name, _, _) in enumerate(GATES):      # Poseidon / Poseidon2 and ArithmeticExtension / Arithmetic alternate in every repeat
            t_gate[name].append(q.add_gates(only[i], info, cs, NUM_CONSTANTS, pi, alphas))
        rows_p, ms = witness(g.poseidon_gate_witness)
        t_wit["poseidon"].append(ms)
        parity &= bool(np.array_equal(rows_p[:, 12:24], want_out))
        t_wit["poseidon2"].append(witness(g.poseidon2_gate_witness)[1])
    q.free()
    med = lambda ts: round(float(np.median(ts)), 4)   # noqa: E731
    per_gate = {}
    for name, kind, param in GATES:
        nw, nc = g.gate_shape(kind, param)
        per_gate[name] = {"ms": med(t_gate[name]), "min_ms": round(min(t_gate[name]), 4), "max_ms": round(max(t_gate[name]), 4),
                          "wires": nw, "constraints": nc, "constants": ctx.lib.gl_gate_num_constants(kind, param)}
    out = {"tool": "plonky2_gates_bench", **gpu_info(), "log_n": LOG_N, "rate_bits": RATE_BITS, "lde_rows": R, "wires_cols": 135,
           "constants_sigmas_cols": NUM_CONSTANTS + 80, "n_challenges": N_CH, "groups": GROUPS, "repeats": args.repeats,
           "per_gate": per_gate, "poseidon_over_poseidon2": round(per_gate["poseidon"]["ms"] / per_gate["poseidon2"]["ms"], 3),
           "arithmetic_extension_over_arithmetic": round(per_gate["arithmetic_extension_10"]["ms"] / per_gate["arithmetic_20"]["ms"], 3),
           "witness_rows": WITNESS_ROWS, "witness_ms": {k: med(v) for k, v in t_wit.items()}, "parity_rows": len(rows), "parity": bool(parity)}
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    wires.merkle_tree.free(); cs.merkle_tree.free()
    ctx.close()
    return 0 if parity else 1


if __name__ == "__main__":
    sys.exit(main())
