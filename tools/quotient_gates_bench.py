"""Device time of the gate part of compute_quotient_polys with selector filters (gl_quotient_add_gates) at the wrapper shape; prints one
JSON line (and writes it to --out when given).

    python tools/quotient_gates_bench.py [--repeats 20] [--warmup 3] [--out FILE]

Shape: N = 2^16, rate_bits 3 (R = 2^19 LDE rows), a 135-column wires commit and an 86-column constants/sigmas commit (4 selectors,
2 gate constants, 80 sigmas), 2 challenges.  Gate list: Poseidon2, U32Arithmetic(3) and the other u32 / b32 gates, Arithmetic(20),
Constant(2), PublicInput, BaseSum<2>(63 limbs), Noop, in 4 selector groups.  The wires matrix (553 MB) is larger than the 126 MB L2, so
every launch reads its rows from HBM.
  add_gates_ms        CUDA events from the first launch of an add_gates call to its last, median over the repeats.
  per_gate_ms         the same call with every other gate replaced by NoopGate (which launches nothing): one launch, the gate exactly as
                      the full call runs it (same selector column, group and constraint powers).
  bytes_read          algorithmic bytes per launch: R rows x (the gate's wires + its selector word + its constants + the accumulator
                      read-modify-write of n_challenges words) x 8 B.
  unfiltered_ms       Poseidon2 and U32Arithmetic through the existing gl_quotient_add_gate with no filter, run alternately with the
                      selector-filtered launch of the same gate in the same process (and with the filter-column path).
  parity              the per-gate accumulators sum to the full call's accumulator.
The GPU's name and power limit are read in the same run.  Needs a CUDA device: there is no CPU fallback.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import plonky25_b200 as g  # noqa: E402
from oracle_c import splitmix_columns  # noqa: E402

P = g.api.P
LOG_N, RATE_BITS, N_CH = 16, 3, 2
GATES = [("poseidon2", g.GATE_POSEIDON2, 0), ("u32_arithmetic_3", g.GATE_U32_ARITHMETIC, 3), ("u32_add_many_5x5", g.GATE_U32_ADD_MANY, 5 | 5 << 8),
         ("u32_subtraction_6", g.GATE_U32_SUBTRACTION, 6), ("u32_range_check_7", g.GATE_U32_RANGE_CHECK, 7),
         ("u32_interleave_3", g.GATE_U32_INTERLEAVE, 3), ("uninterleave_to_u32_2", g.GATE_UNINTERLEAVE_TO_U32, 2),
         ("uninterleave_to_b32_2", g.GATE_UNINTERLEAVE_TO_B32, 2), ("comparison_32_16", g.GATE_COMPARISON, 32 | 16 << 8),
         ("arithmetic_20", g.GATE_ARITHMETIC, 20), ("constant_2", g.GATE_CONSTANT, 2), ("public_input", g.GATE_PUBLIC_INPUT, 0),
         ("base_sum_2_63", g.GATE_BASE_SUM, 63 | 2 << 8), ("noop", g.GATE_NOOP, 0)]
GROUPS = [(0, 1), (1, 5), (5, 9), (9, 14)]
SELECTORS = [next(s for s, (a, b) in enumerate(GROUPS) if a <= i < b) for i in range(len(GATES))]
NUM_CONSTANTS = len(GROUPS) + 2


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as e:   # the measurement stands without the query; say why the fields are missing
        import torch
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"unavailable ({type(e).__name__})"}


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
    q = g.Quotient(wires, N_CH, ctx=ctx)
    noop = (g.GATE_NOOP, 0)

    def full():
        return q.add_gates([(k, p) for _, k, p in GATES], info, cs, NUM_CONSTANTS, pi, alphas)

    def one(i):
        return q.add_gates([(k, p) if j == i else noop for j, (_, k, p) in enumerate(GATES)], info, cs, NUM_CONSTANTS, pi, alphas)

    # parity: the per-gate launches sum to the full call (fresh accumulators)
    q_full, q_parts = g.Quotient(wires, N_CH, ctx=ctx), g.Quotient(wires, N_CH, ctx=ctx)
    q_full.add_gates([(k, p) for _, k, p in GATES], info, cs, NUM_CONSTANTS, pi, alphas)
    for i in range(len(GATES)):
        q_parts.add_gates([(k, p) if j == i else noop for j, (_, k, p) in enumerate(GATES)], info, cs, NUM_CONSTANTS, pi, alphas)
    parity = bool(np.array_equal(q_full.values(), q_parts.values()))
    q_full.free(); q_parts.free()

    lib = ctx.lib
    baseline = {"poseidon2": (g.GATE_POSEIDON2, 0), "u32_arithmetic_3": (g.GATE_U32_ARITHMETIC, 3)}
    idx = {name: i for i, (name, _, _) in enumerate(GATES)}
    for _ in range(args.warmup):
        full()
        for i in range(len(GATES)):
            one(i)
        for kind, param in baseline.values():
            q.add_gate(kind, param, alphas)
            q.add_gate(kind, param, alphas, filter=(cs, 0))
    t_full, t_gate = [], {name: [] for name, _, _ in GATES}
    t_unf, t_col, t_sel = ({name: [] for name in baseline} for _ in range(3))
    for _ in range(args.repeats):
        t_full.append(full())
        for i, (name, _, _) in enumerate(GATES):
            t_gate[name].append(one(i))
        for name, (kind, param) in baseline.items():     # alternately: no filter, filter column, selector filter
            t_unf[name].append(q.add_gate(kind, param, alphas))
            t_col[name].append(q.add_gate(kind, param, alphas, filter=(cs, 0)))
            t_sel[name].append(one(idx[name]))
    q.free()
    med = lambda ts: round(float(np.median(ts)), 4)   # noqa: E731
    per_gate = {}
    for name, kind, param in GATES:
        nw, nc = g.gate_shape(kind, param)
        nk = lib.gl_gate_num_constants(kind, param)
        nbytes = R * 8 * (nw + 1 + nk + 2 * N_CH) if nc else 0
        ms = med(t_gate[name])
        per_gate[name] = {"ms": ms, "constraints": nc, "bytes_read": nbytes, "gb_per_s": round(nbytes / (ms * 1e-3) / 1e9, 1) if ms else None}
    out = {"tool": "quotient_gates_bench", **gpu_info(), "log_n": LOG_N, "rate_bits": RATE_BITS, "lde_rows": R, "wires_cols": 135,
           "constants_sigmas_cols": NUM_CONSTANTS + 80, "n_challenges": N_CH, "groups": GROUPS, "repeats": args.repeats,
           "add_gates_ms": med(t_full), "sum_of_per_gate_ms": round(sum(v["ms"] for v in per_gate.values()), 4),
           "bytes_read": sum(v["bytes_read"] for v in per_gate.values()), "per_gate": per_gate,
           "filter_cost": {name: {"unfiltered_ms": med(t_unf[name]), "filter_column_ms": med(t_col[name]), "selector_filter_ms": med(t_sel[name])}
                           for name in baseline},
           "parity": parity}
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
