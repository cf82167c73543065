#!/usr/bin/env python3
"""Headline benchmark: PolynomialBatch commit throughput (iNTT + coset LDE + bit-reversed row-major leaves + Poseidon
Merkle tree to the cap) on N B200s, in Melem/s (= N_rows * n_cols input elements per second), BASELINE.json's metric.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

One "step" = one whole commit of the workload (default 2^20 x 135, rate_bits 3, cap_height 4 = BASELINE.json configs[2],
the shape the metric is quoted on; it fits one GPU).  `value` is measured with the columns already resident in HBM
(gl_dev_commit / the sharded device path), `e2e` through the reference-facing C ABI call gl_commit with host buffers
(pinned), i.e. including the host->device copy of the inputs and the device->host read of the Merkle cap, every step.

N > 1 (one process per GPU, torchrun): columns are sharded for the iNTT; the ranks exchange coefficient blocks over NVLink (one
contiguous peer copy per block, overlapped with the NTTs) and every rank evaluates only the LDE cosets whose leaf rows it owns, for
all columns (--exchange coset, the default when N <= 2^rate_bits; p2p / nccl = the column->row shipment of the LDE output by the
copy engines / by an NCCL all-to-all); every rank hashes whole cap subtrees of its contiguous leaf range and the subtree roots are
all-gathered into the cap (SURVEY.md §8e).  Per-rank work shrinks with N ("strong" scaling of one commit).  --single-process drives
the N GPUs from one process through gl_commit_multi.

--impl reference times the CPU restatement of the reference algorithm (oracle/, C + OpenMP, all host threads) on a
bounded sample of the same workload; the reference itself is Rust + an un-vendored crate and cannot be built here
(DESIGN.md).  The oracle is used here only as the timed CPU baseline / checker, never on the product path.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)
sys.dont_write_bytecode = True       # the benchmark leaves the tree it runs from as it found it (no __pycache__ of the modules above)

P = 0xFFFF_FFFF_0000_0001
METRIC = "commit Melem/s (2^20x135 LDE+Poseidon Merkle)"
UNIT = "Melem/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--log-n", type=int, default=20)
    ap.add_argument("--cols", type=int, default=135)
    ap.add_argument("--rate-bits", type=int, default=3)
    ap.add_argument("--cap-height", type=int, default=4)
    ap.add_argument("--cpu-sample-log-n", type=int, default=17, help="rows (log2) of the bounded CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--exchange", default="auto", choices=["auto", "coset", "p2p", "nccl"],
                    help="multi-GPU plan (DESIGN.md §6): coset = exchange coefficients, every rank evaluates its own cosets (default when "
                         "N <= 2^rate_bits); p2p = column->row shipment of the LDE output by the copy engines; nccl = all-to-all baseline")
    ap.add_argument("--workload", default="commit", choices=["commit", "wrapper"],
                    help="commit: the headline PolynomialBatch commit; wrapper: the wrapper-circuit-shaped prove pipeline (commits 86/135/20/16 "
                         "x 2^16 -> prove_openings -> FRI [4,4,4] -> PoW 16 -> 28 query rounds), second line of BASELINE.json's metric")
    ap.add_argument("--single-process", action="store_true",
                    help="--gpus N from ONE process through gl_commit_multi (the form CircuitData::prove can call), instead of torchrun")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (a fixed, seeded sample of "
                         "the large arrays, at most 64 MB in all), so that two builds can be compared output for output")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference" and a.workload == "commit":
        ap.error("--dump-outputs: the reference commit arm times the CPU restatement and keeps no outputs")
    return a


def workload_name(a):
    return f"PolynomialBatch::from_values commit 2^{a.log_n} x {a.cols}, rate_bits={a.rate_bits}, cap_height={a.cap_height}"


def perms_per_commit(log_n, cols, r, h):
    R = 1 << (log_n + r)
    per_leaf = (cols + 7) // 8 if cols > 4 else 0
    return R * per_leaf + (R - (1 << h))


# ------------------------------------------------------------------------------------------------ --dump-outputs
DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Writes every array of field words as out_dir/<name>.npy: float64 with a trailing axis of two, the low and the high 32 bits of each
    uint64 word (a whole word does not fit a float64 mantissa; each half does, so the dump is exact)."""
    import numpy as np
    out = {}
    for name, a in arrays.items():
        w = np.asarray(a, dtype=np.uint64)
        out[name] = np.stack([w & np.uint64(0xFFFFFFFF), w >> np.uint64(32)], axis=-1).astype(np.float64)
    total = sum(x.nbytes for x in out.values())
    if total > DUMP_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, x in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), x)


def dump_sample(n, k, seed):
    """k sorted indices out of range(n), the same for every run and build (all of them when k >= n)"""
    import numpy as np
    if k >= n:
        return np.arange(n, dtype=np.uint64)
    return np.sort(np.random.default_rng(seed).choice(n, size=k, replace=False)).astype(np.uint64)


def tree_outputs(cap, trees, batch=None):
    """What a caller of a commit receives, sized for DUMP_BYTES: the whole cap, seeded samples of the leaf rows with their Merkle paths
    (which carry digests from every layer of the tree) and, when the batch keeps them, of the coefficients.  `trees` cover equal
    consecutive leaf ranges (one tree, or the shard trees of gl_commit_multi)."""
    import numpy as np
    cap = np.asarray(cap, dtype=np.uint64).reshape(-1, 4)
    per, cols = trees[0].n_leaves, trees[0].leaf_len
    depth = per.bit_length() - 1 - trees[0].cap_height
    row_bytes = 16 * (1 + cols + 4 * depth + (1 + cols if batch is not None else 0))
    k = min(4096, max(1, (DUMP_BYTES - 16 * cap.size) // row_bytes))
    idx = dump_sample(per * len(trees), k, seed=1)
    rows = np.zeros((idx.size, cols), dtype=np.uint64)
    paths = np.zeros((idx.size, depth, 4), dtype=np.uint64)
    for q, t in enumerate(trees):
        sel = (idx // per) == q
        if sel.any():
            rows[sel], paths[sel] = t.open_batch(idx[sel] % per)
    out = {"cap": cap, "leaf_index": idx, "leaves": rows, "merkle_paths": paths}
    if batch is not None:
        cidx = dump_sample(1 << batch.degree_log, k, seed=2)
        out.update({"coeff_index": cidx, "coeffs": batch.polynomials[:, cidx]})
    return out


def proof_outputs(proof):
    """every field of a wrapper-pipeline proof (tests/wrapper_pipeline.py), one array per field, tree and FRI layer"""
    out = {"commit_caps": proof["commit_caps"], "commit_phase_caps": proof["commit_phase_caps"], "final_poly": proof["final_poly"],
           "pow_witness": [proof["pow_witness"]], "query_indices": proof["query_indices"]}
    rounds = proof["query_rounds"]
    for k in range(len(rounds[0]["initial"])):
        out[f"query_rows_tree{k}"] = [rn["initial"][k][0] for rn in rounds]
        out[f"query_paths_tree{k}"] = [rn["initial"][k][1] for rn in rounds]
    for j in range(len(rounds[0]["steps"])):
        out[f"query_evals_layer{j}"] = [rn["steps"][j][0] for rn in rounds]
        out[f"query_paths_layer{j}"] = [rn["steps"][j][1] for rn in rounds]
    return out


# ------------------------------------------------------------------------------------------------ CPU baseline
def cpu_commit_time(oc, log_n, cols, r, h, seed=1):
    from oracle_c import splitmix_columns
    x = splitmix_columns(seed, cols, 1 << log_n)
    t = time.perf_counter()
    res = oc.commit(x, r, min(h, log_n + r), want=())
    return time.perf_counter() - t, res["stage_s"]


def cpu_baseline(a, repeats=1):
    from oracle_c import OracleC
    oc = OracleC()
    oc.set_threads(host_threads())
    threads = oc.num_threads()
    log_n = min(a.cpu_sample_log_n, a.log_n)
    best, stages = None, None
    for _ in range(repeats):
        dt, st = cpu_commit_time(oc, log_n, a.cols, a.rate_bits, a.cap_height)
        if best is None or dt < best:
            best, stages = dt, st
    # SURVEY §8(d): the reference as shipped runs the commitment serially (plonky2's `parallel` feature is off in its build), so the
    # same restatement is also timed on ONE thread, on a smaller sample of the same workload
    single = None
    try:
        log_n1 = min(log_n, 14)
        oc.set_threads(1)
        dt1, _ = cpu_commit_time(oc, log_n1, a.cols, a.rate_bits, a.cap_height)
        single = {"value": round((a.cols << log_n1) / dt1 / 1e6, 4), "unit": UNIT, "cores": 1,
                  "sample": f"one commit of 2^{log_n1} x {a.cols}, {dt1:.2f} s on one thread"}
    except Exception as e:   # the baseline is a reported number: never let it break the bench line
        single = {"error": str(e)}
    finally:
        oc.set_threads(threads)
    return {"value": round((a.cols << log_n) / best / 1e6, 4), "unit": UNIT, "cores": threads, "kind": "port", "single_thread": single,
            "sample": f"one commit of 2^{log_n} x {a.cols} (rate_bits {a.rate_bits}, cap_height {a.cap_height}) = 1/{1 << (a.log_n - log_n)} of "
                      f"the workload's rows, {best:.2f} s with {threads} OpenMP threads; oracle/gl_oracle.c (C restatement of the "
                      "reference algorithm; the Rust reference cannot be built in this image)",
            "stage_s": {k: round(v, 3) for k, v in zip(("ifft", "lde_fft", "transpose", "merkle"), stages)}}


def host_threads():
    """threads the CPU arm may use: every core this process is allowed on.  torchrun exports OMP_NUM_THREADS=1 to its children;
    that setting is for GPU ranks and must not throttle the CPU baseline, so the oracle's thread count is set explicitly."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def run_reference(a):
    """--impl reference: the CPU restatement on all host threads, bounded sample per step (rank 0 only; the whole run is sized to
    end within ~2 minutes whatever the core count)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle_c import OracleC
    oc = OracleC()
    threads = host_threads()
    oc.set_threads(threads)
    threads = oc.num_threads()
    # size the sample from a probe: one 2^13 commit is timed, cost is ~linear in rows, and the largest sample <= --cpu-sample-log-n
    # whose (warmup + steps) fits the time budget is used
    probe_log_n = min(13, a.log_n)
    cpu_commit_time(oc, min(10, a.log_n), a.cols, a.rate_bits, a.cap_height)          # page-in, OpenMP pool
    t_probe, _ = cpu_commit_time(oc, probe_log_n, a.cols, a.rate_bits, a.cap_height)
    budget_s = float(os.environ.get("GL_REF_BUDGET_S", "100"))
    log_n = probe_log_n
    while log_n < min(a.cpu_sample_log_n, a.log_n) and t_probe * (1 << (log_n + 1 - probe_log_n)) * (a.steps + min(a.warmup, 1)) <= budget_s:
        log_n += 1
    for _ in range(min(a.warmup, 1)):                                                   # one full-size warm-up, the rest on a small case
        cpu_commit_time(oc, log_n, a.cols, a.rate_bits, a.cap_height)
    for _ in range(max(a.warmup - 1, 0)):
        cpu_commit_time(oc, min(log_n, 12), a.cols, a.rate_bits, a.cap_height)
    t0 = time.perf_counter()
    for s in range(a.steps):
        cpu_commit_time(oc, log_n, a.cols, a.rate_bits, a.cap_height, seed=s + 1)
    dt = time.perf_counter() - t0
    val = a.steps * (a.cols << log_n) / dt / 1e6
    sample = (f"each step = one commit of 2^{log_n} x {a.cols} (1/{1 << (a.log_n - log_n)} of the workload's rows; throughput in "
              f"elements/s is what is compared), oracle/gl_oracle.c with {threads} OpenMP threads")
    line = {"impl": "reference", "metric": METRIC, "value": round(val, 4), "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": round(dt / a.steps * 1e3, 3), "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u64 (Goldilocks field)", "data": "synthetic",
            "config": {"workload": workload_name(a), "sample": sample},
            "cpu_baseline": {"value": round(val, 4), "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": round(val, 4), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.t = threading.Thread(target=self._read, daemon=True)
        self.t.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for t, r in self.rows if t0 <= t <= t1] or [r for _, r in self.rows]
        sm = sorted(int(r[1]) for r in rows if r[1].isdigit())
        reasons = set()
        for r in rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": int(rows[0][2]) if rows and rows[0][2].isdigit() else None,
                "reasons": sorted(reasons), "samples": len(rows),
                "power_w_max": max((float(r[3]) for r in rows if r[3].replace(".", "", 1).isdigit()), default=None)}


# ------------------------------------------------------------------------------------------------ GPU arm
def synth_columns(torch, dev, cols, n, seed):
    """[cols][n] canonical Goldilocks words (SplitMix64 of the element index), generated on the device, int64 storage."""
    idx = torch.arange(1, cols * n + 1, dtype=torch.int64, device=dev)
    z = idx * -7046029254386353131 + (0x706C6F6E6B7932 ^ seed)                      # 0x9E3779B97F4A7C15 as int64
    z = (z ^ ((z >> 30) & ((1 << 34) - 1))) * -4658895280553007687                  # 0xBF58476D1CE4E5B9
    z = (z ^ ((z >> 27) & ((1 << 37) - 1))) * -7723592293110705685                  # 0x94D049BB133111EB
    z = z ^ ((z >> 31) & ((1 << 33) - 1))
    # unsigned z >= p  <=>  signed z in [-(2^32 - 1), -1]
    z = torch.where((z < 0) & (z >= -(2**32 - 1)), z + (2**32 - 1), z)               # z - p (mod 2^64) = z + 2^32 - 1
    return z.view(cols, n)


def run_wrapper(a):
    """--workload wrapper: the hot-path part of `data.prove(pw)` (/root/reference/src/p3/mod.rs:258-262) at the wrapper circuit's
    shape, end to end through the reference-facing interface with HOST (pinned) columns, and the CPU oracle on the same transcript
    beside it; every proof field is hashed and compared.  One JSON line, metric `wrap_hot_path_ms` (lower is better)."""
    import numpy as np
    import wrapper_pipeline as wp
    log_n = 16 if a.log_n == 20 else a.log_n
    cols = wp.make_columns(log_n)
    line = {"metric": "wrap_hot_path_ms (wrapper-shaped commits 86/135/20/16 x 2^%d, r=3, h=4 -> prove_openings -> FRI [4,4,4] -> PoW 16 -> "
                      "28 query rounds)" % log_n, "unit": "ms", "n_gpus": 1, "steps": a.steps, "warmup": a.warmup, "higher_is_better": False,
            "scaling": "strong", "vs_baseline": None, "dtype": "u64 (Goldilocks field, integer + exact fp64 limb arithmetic)", "data": "synthetic",
            "config": {"workload": "wrapper-circuit-shaped prove pipeline (tests/wrapper_pipeline.py): the commitment hot path of data.prove at "
                                   "src/p3/mod.rs:258-262; column contents synthetic, shapes/call order/proof bytes the reference's",
                       "log_n": log_n, "widths": list(wp.WIDTHS), "rate_bits": 3, "cap_height": 4, "arities": list(wp.ARITIES),
                       "pow_bits": wp.POW_BITS, "query_rounds": wp.N_QUERIES,
                       "note": "fib(64) wrap-prove ms itself is not runnable here (no Rust toolchain); this is BASELINE.md §4.6's surrogate"}}
    if a.impl == "reference":
        from oracle_c import OracleC
        oc = OracleC()
        oc.set_threads(host_threads())
        tm = {}
        for _ in range(min(a.warmup, 1)):
            wp.run_oracle(oc, cols, log_n)
        t0 = time.perf_counter()
        for _ in range(a.steps):
            proof = wp.run_oracle(oc, cols, log_n, timings=tm)
        ms = (time.perf_counter() - t0) / a.steps * 1e3
        if a.dump_outputs:
            dump_outputs(a.dump_outputs, proof_outputs(proof))
        line.update({"impl": "reference", "value": round(ms, 2), "ms_per_step": round(ms, 2), "stage_ms": {k: round(v, 2) for k, v in tm.items()},
                     "cpu_baseline": {"value": round(ms, 2), "unit": "ms", "cores": oc.num_threads(), "kind": "port",
                                      "sample": "the whole pipeline, oracle/gl_oracle.c + Python glue"},
                     "e2e": {"value": round(ms, 2), "unit": "ms", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0,
                     "parity": {"proof_sha256": wp.digest(proof)}})
        print(json.dumps(line), flush=True)
        return
    import plonky25_b200 as g
    ctx = g.Context(0)
    lib = ctx.lib
    # pinned host columns (what a binding that cares about PCIe hands over; gl_host_alloc)
    pinned = []
    for c in cols:
        ptr = lib.gl_host_alloc(c.nbytes)
        arr = np.ctypeslib.as_array(ctypes.cast(ptr, ctypes.POINTER(ctypes.c_uint64)), shape=c.shape)
        arr[:] = c
        pinned.append(arr)
    sampler = ClockSampler(0)
    for _ in range(max(a.warmup, 0)):
        wp.run_product(g, ctx, pinned, log_n)
    sampler.start()
    time.sleep(0.2)
    acc = {}
    t0 = time.perf_counter()
    for _ in range(a.steps):
        tm = {}
        proof = wp.run_product(g, ctx, pinned, log_n, timings=tm)
        for k, v in tm.items():
            acc[k] = acc.get(k, 0.0) + v
    t1 = time.perf_counter()
    ms = (t1 - t0) / a.steps * 1e3
    clocks = sampler.stop(t0, t1)
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, proof_outputs(proof))
    h2d = sum(c.nbytes for c in cols)
    d2h = sum(np.asarray(x).nbytes for rnd in proof["query_rounds"] for pair in rnd["initial"] + rnd["steps"] for x in pair) + \
        sum(np.asarray(c).nbytes for c in proof["commit_caps"] + proof["commit_phase_caps"]) + np.asarray(proof["final_poly"]).nbytes
    parity = {"proof_sha256": wp.digest(proof), "oracle": None, "match": None}
    cpu = None
    if not a.no_cpu_baseline:
        from oracle_c import OracleC
        oc = OracleC()
        oc.set_threads(host_threads())
        tmc = {}
        ref = wp.run_oracle(oc, cols, log_n, timings=tmc)
        parity.update({"oracle": "oracle/gl_oracle.c on the same columns and transcript", "match": wp.digest(ref) == parity["proof_sha256"]})
        cpu = {"value": round(tmc["total"], 2), "unit": "ms", "cores": oc.num_threads(), "kind": "port",
               "sample": "the whole pipeline once", "stage_ms": {k: round(v, 2) for k, v in tmc.items()}}
    # ---- SURVEY §8(f) rank 3: gate-constraint evaluation over the resident LDE rows of a wires commit at the wrapper's R = 2^19
    gate_eval = None
    try:
        import random
        import gates_oracle as go
        wires = g.PolynomialBatch.from_values(list(pinned[1]), 3, False, 4, ctx=ctx)
        R = 1 << (log_n + 3)
        alphas = np.array([0x1234567890ABCDEF % P, 0xFEDCBA9876543210 % P], dtype=np.uint64)
        q, ms_ = ctypes.c_uint64(), ctypes.c_float()
        assert lib.gl_quotient_begin(ctx.handle, wires.merkle_tree._h, 2, ctypes.byref(q)) == 0
        t_g = {}
        for name, kind, param, off in (("Poseidon2Gate", 0, 0, 0), ("U32ArithmeticGate", 1, 3, 123)):
            best = 1e9
            for _ in range(3):
                assert lib.gl_quotient_add_gate(ctx.handle, q.value, kind, param, alphas.ctypes.data, off, 0, 0) == 0
                lib.gl_ctx_aux_ms(ctx.handle, ctypes.byref(ms_))
                best = min(best, ms_.value)
            t_g[name] = best
        # parity on sampled rows: (3 accumulations of each gate) == 3 * reduce_with_powers of the oracle's constraints of that leaf row
        out = np.zeros((2, R), dtype=np.uint64)
        assert lib.gl_quotient_read(ctx.handle, q.value, out.ctypes.data) == 0
        lib.gl_quotient_end(ctx.handle, q.value)
        rnd = random.Random(1)
        rows = [0, R - 1] + [rnd.randrange(R) for _ in range(14)]
        lw = wires.merkle_tree.open_batch(rows)[0]
        ok = True
        for j, row in enumerate(rows):
            c0, c1 = go.poseidon2_gate_eval(lw[j].tolist()), go.u32_arithmetic_eval(lw[j].tolist()[:114], num_ops=3)
            for k in range(2):
                want = 3 * (go.reduce_with_powers(c0, int(alphas[k])) + go.reduce_with_powers(c1, int(alphas[k]), start_power=123)) % P
                ok = ok and int(out[k, row]) == want
        wires.merkle_tree.free()
        gate_eval = {"rows": R, "n_challenges": 2, "ms": {k: round(v, 4) for k, v in t_g.items()},
                     "melem_per_s": {k: round(R * 135 / (v * 1e-3) / 1e6, 1) for k, v in t_g.items()},
                     "mconstraints_per_s": {"Poseidon2Gate": round(R * 123 / (t_g["Poseidon2Gate"] * 1e-3) / 1e6, 1),
                                            "U32ArithmeticGate": round(R * 108 / (t_g["U32ArithmeticGate"] * 1e-3) / 1e6, 1)},
                     "unit": "wire elements of the LDE rows consumed per second (R x 135 / kernel time, CUDA events)",
                     "parity": {"sampled_rows": len(rows), "match": bool(ok),
                                "oracle": "oracle/gates_oracle.py (restates poseidon2_gate.rs:233-310, arithmetic_u32.rs:103-166)"}}
        # ---- SURVEY §8(f) rank 4 + the permutation part of rank 3, at the same shape: Z / partial products of 80 routed wires (2 challenges,
        # chunks of 8), their commit, and the permutation-argument terms over the R = 2^19 resident LDE rows.  Sigma VALUES are synthetic
        # (the 86-column batch's first 80 columns), so the argument does not close; parity is per row against the restated formulas.
        n_routed, degree, n = 80, 8, 1 << log_n
        k_is = [pow(7, j, P) for j in range(n_routed)]
        betas, gammas = [0x1111111122222222 % P, 0x3333333344444444 % P], [0x5555555566666666 % P, 0x7777777788888888 % P]
        sig_cols = [pinned[0][j] for j in range(n_routed)]
        t_pp = []
        for _ in range(3):
            ta = time.perf_counter()
            zs = g.partial_products_and_zs([pinned[1][j] for j in range(n_routed)], sig_cols, k_is, betas, gammas, degree, ctx=ctx)
            t_pp.append((time.perf_counter() - ta) * 1e3)
        lib.gl_ctx_aux_ms(ctx.handle, ctypes.byref(ms_))
        pp_kernel_ms = ms_.value
        # rows i: the chunk quotients recomputed from the definition must be the ratios of consecutive outputs
        w_n = pow(1753635133440165772, 1 << (32 - log_n), P)
        ok_pp = True
        for i in [0, 1, n - 2] + [rnd.randrange(n - 1) for _ in range(5)]:
            x = pow(w_n, i, P)
            for k in range(2):
                accs = [int(zs[k, i])] + [int(zs[2 + k * 9 + c, i]) for c in range(9)] + [int(zs[k, i + 1])]
                for c in range(10):
                    num = den = 1
                    for j in range(8 * c, 8 * c + 8):
                        wv = int(pinned[1][j][i])
                        num = num * ((wv + betas[k] * k_is[j] % P * x + gammas[k]) % P) % P
                        den = den * ((wv + betas[k] * int(sig_cols[j][i]) + gammas[k]) % P) % P
                    ok_pp = ok_pp and accs[c] * num % P == accs[c + 1] * den % P
        wires = g.PolynomialBatch.from_values(list(pinned[1]), 3, False, 4, ctx=ctx)
        sig_b = g.PolynomialBatch.from_values(list(pinned[0]), 3, False, 4, ctx=ctx)
        zs_b = g.PolynomialBatch.from_values(list(zs), 3, False, 4, ctx=ctx)
        quot = g.Quotient(wires, 2, ctx=ctx)
        t_v = min(quot.add_permutation(sig_b, 0, zs_b, n_routed, degree, k_is, betas, gammas, [int(a_) for a_ in alphas]) for _ in range(3))
        accq = quot.values()
        quot.free()
        bits = log_n + 3
        w_R = pow(1753635133440165772, 1 << (32 - bits), P)
        rev = lambda i: int(format(i, "0%db" % bits)[::-1], 2)
        ok_v = True
        for row in [0, R - 1] + [rnd.randrange(R) for _ in range(6)]:
            idx = rev(row)
            x = 7 * pow(w_R, idx, P) % P
            lw, ls = wires.merkle_tree.get(row).tolist(), sig_b.merkle_tree.get(row).tolist()
            lz, lzn = zs_b.merkle_tree.get(row).tolist(), zs_b.merkle_tree.get(rev((idx + 8) % R)).tolist()
            terms = go.vanishing_permutation_terms(lw[:n_routed], ls[:n_routed], lz, lzn, x, k_is, betas, gammas, degree, log_n)
            for k in range(2):
                ok_v = ok_v and int(accq[k, row]) == 3 * go.reduce_with_powers(terms, int(alphas[k])) % P
        for b_ in (wires, sig_b, zs_b):
            b_.merkle_tree.free()
        gate_eval["permutation"] = {"partial_products_call_ms": round(min(t_pp), 3), "partial_products_kernels_ms": round(pp_kernel_ms, 3),
                                    "vanishing_terms_kernel_ms": round(t_v, 4), "n_routed": n_routed, "degree": degree,
                                    "note": "partial_products_call_ms includes 84 MB of host->device columns and 10 MB back",
                                    "parity": {"partial_products_rows": bool(ok_pp), "vanishing_terms_rows": bool(ok_v)}}
    except Exception as e:   # a reported extra: never lose the main line over it
        gate_eval = {"error": repr(e)}
    line.update({"value": round(ms, 3), "ms_per_step": round(ms, 3), "stage_ms": {k: round(v / a.steps, 3) for k, v in acc.items()},
                 "clocks": clocks, "gpu_launches": None, "gate_eval": gate_eval,
                 "e2e": {"value": round(ms, 3), "unit": "ms", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                         "api": "PolynomialBatch.from_values/from_coeffs -> prove_openings -> fri_prover_query_rounds (plonky2.5_b200/api.py over "
                                "include/gl_commit.h), pinned host columns in, proof fields out"},
                 "cpu_baseline": cpu, "parity": parity})
    print(json.dumps(line), flush=True)
    ctx.close()
    if parity["match"] is False:
        raise SystemExit("PARITY MISMATCH: the wrapper-pipeline proof differs from the oracle's")


def run_single_process(a):
    """--gpus N --single-process: ONE process drives N GPUs through gl_commit_multi (one context per device, worker threads inside the
    library) — the form CircuitData::prove (/root/reference/src/p3/mod.rs:260), a single process, can actually call.  Host (pinned)
    columns in, cap out: the number is end-to-end by construction, so `value` and `e2e.value` are the same measurement."""
    import numpy as np
    import plonky25_b200 as g
    import headline
    from oracle_c import splitmix_columns
    log_n, cols, r, h = a.log_n, a.cols, a.rate_bits, a.cap_height
    n = 1 << log_n
    ctxs = [g.Context(d) for d in range(a.gpus)]
    lib = ctxs[0].lib
    ptr = lib.gl_host_alloc(cols * n * 8)
    harr = np.ctypeslib.as_array(ctypes.cast(ptr, ctypes.POINTER(ctypes.c_uint64)), shape=(cols, n))
    harr[:] = splitmix_columns(1, cols, n)
    sampler = ClockSampler(0)
    kept = []                        # --dump-outputs: the shard trees of the last timed step, released after the dump

    def step(last=False):
        cap, trees = g.commit_multi(ctxs, list(harr), r, h)
        if last and a.dump_outputs:
            kept.extend(trees)
        else:
            for t in trees:
                t.free()
        return cap.hashes

    for _ in range(max(a.warmup, 0)):
        step()
    sampler.start()
    time.sleep(0.2)
    t0 = time.perf_counter()
    for i in range(a.steps):
        cap = step(last=i == a.steps - 1)
    t1 = time.perf_counter()
    clocks = sampler.stop(t0, t1)
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, tree_outputs(cap, kept))
        for t in kept:
            t.free()
    ms = (t1 - t0) / a.steps * 1e3
    val = cols * n / (ms * 1e-3) / 1e6
    stage = {}
    for d, c in enumerate(ctxs):
        st, _ = c.stage_times()
        stage[f"gpu{d}"] = {k: round(v, 3) for k, v in st.items() if v}
    parity = headline.parity_block(cap, log_n, cols, r, h, seed=1)
    line = {"metric": METRIC, "value": round(val, 3), "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": round(ms, 4), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "u64 (Goldilocks field, integer + exact fp64 limb arithmetic)", "data": "synthetic",
            "config": {"workload": workload_name(a), "mode": "single process, gl_commit_multi: one context per device, column shards -> "
                                                             "copy-engine peer shipments -> per-device subtrees -> cap concatenated on the host",
                       "timing": "host wall clock around the synchronous call (the call returns after every device's cap slice is on the host)"},
            "stage_ms_last_call": stage, "clocks": clocks, "gpu_launches": None,
            "e2e": {"value": round(val, 3), "unit": UNIT, "h2d_bytes_per_step": cols * n * 8, "d2h_bytes_per_step": 32 << h,
                    "ms_per_step": round(ms, 4), "api": "gl_commit_multi (include/gl_commit.h) with pinned host columns"},
            "roofline": None, "cpu_baseline": None, "parity": parity}
    print(json.dumps(line), flush=True)
    for c in ctxs:
        c.close()
    if parity["match"] is False:
        raise SystemExit("PARITY MISMATCH: the Merkle cap differs from the oracle's golden (see the `parity` object)")


def main():
    a = parse()
    if a.workload == "wrapper":
        return run_wrapper(a)
    if a.impl == "reference":
        return run_reference(a)
    if a.single_process and a.gpus > 1:
        return run_single_process(a)

    import numpy as np
    import torch
    import torch.distributed as dist
    import plonky25_b200 as g
    from plonky25_b200 import sharded

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != a.gpus:
        if world == 1 and a.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    ctx = g.Context(local)                      # raises without the CUDA library / a GPU: there is no fallback
    lib = ctx.lib
    stream = torch.cuda.ExternalStream(ctx.stream, device=dev)
    log_n, cols, r, h = a.log_n, a.cols, a.rate_bits, a.cap_height
    n = 1 << log_n
    cap = np.zeros(4 << h, dtype=np.uint64)
    kept = []                        # --dump-outputs: the batch handle of the last timed step, released after the dump

    if world == 1:
        d_cols = synth_columns(torch, dev, cols, n, 1)
        torch.cuda.synchronize()

        def step(last=False):
            hd = ctypes.c_uint64()
            rc = lib.gl_dev_commit(ctx.handle, d_cols.data_ptr(), n, cols, log_n, r, h, 0, cap.ctypes.data, ctypes.byref(hd))
            if rc != 0:
                raise RuntimeError(lib.gl_ctx_last_error(ctx.handle).decode())
            if last and a.dump_outputs:
                kept.append(hd.value)
            else:
                lib.gl_tree_free(ctx.handle, hd.value)
    else:
        plan = sharded.ShardPlan(cols, log_n, r, h, world)
        c0, c1 = plan.col_range(rank)
        d_cols = synth_columns(torch, dev, cols, n, 1)[c0:c1].contiguous()
        state = sharded.ShardedCommit(ctx, plan, rank, dist, torch, exchange=a.exchange)
        torch.cuda.synchronize()

        def step(last=False):
            cap[:] = state.commit(d_cols)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(a.warmup, 0)):
        step()
    stage_acc = {}
    launches = 0
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record(stream)
    for i in range(a.steps):
        step(last=i == a.steps - 1)
        ms, ln = ctx.stage_times()
        for k, v in ms.items():
            stage_acc[k] = stage_acc.get(k, 0.0) + v
        launches += sum(ln.values())
    e1.record(stream)
    barrier()
    t1 = time.perf_counter()
    dev_ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms = float(t.item())
        tl = torch.tensor([launches], dtype=torch.int64, device=dev)
        dist.all_reduce(tl)
        launches = int(tl.item())
    clocks = sampler.stop(t0, t1) if rank == 0 else None
    ms_per_step = dev_ms / a.steps
    value = cols * n / (ms_per_step * 1e-3) / 1e6
    cap_dev = cap.copy()
    # parity: the cap this run produced against the oracle's golden cap for the same synthetic input (tests/golden/headline_*.json,
    # plain JSON — the oracle itself is not executed here).  A mismatch fails the run: a fast wrong commit is not a result.
    import headline
    parity = headline.parity_block(cap_dev, log_n, cols, r, h, seed=1)
    if a.dump_outputs and rank == 0:
        if world == 1:                   # one device: the whole batch stays behind the handle (coefficients, leaves, digests)
            batch = g.PolynomialBatch(ctx, g.MerkleTree(ctx, kept[0], cap_dev), cols)
            dump_outputs(a.dump_outputs, tree_outputs(cap_dev, [batch.merkle_tree], batch))
            batch.merkle_tree.free()
        else:                            # sharded: a caller of ShardedCommit.commit receives the cap
            dump_outputs(a.dump_outputs, {"cap": cap_dev.reshape(-1, 4)})

    # ---- e2e: the C-ABI call a Rust shim would make, host buffers in, cap out, every step --------------------------
    e2e = None
    if not a.no_e2e:
        if world == 1:
            host = ctypes.cast(lib.gl_host_alloc(cols * n * 8), ctypes.POINTER(ctypes.c_uint64))
            if not host:
                raise MemoryError("gl_host_alloc failed")
            harr = np.ctypeslib.as_array(host, shape=(cols, n))
            harr[:] = d_cols.cpu().numpy().view(np.uint64)
            ptrs = (ctypes.c_void_p * cols)(*[harr[j].ctypes.data for j in range(cols)])

            def e2e_step():
                hd = ctypes.c_uint64()
                rc = lib.gl_commit(ctx.handle, ptrs, cols, log_n, r, h, 0, None, None, None, cap.ctypes.data, ctypes.byref(hd))
                if rc != 0:
                    raise RuntimeError(lib.gl_ctx_last_error(ctx.handle).decode())
                lib.gl_tree_free(ctx.handle, hd.value)
            h2d = cols * n * 8
        else:
            idx = state.host_columns()       # the streamed coset plan deals the host columns cyclically (ShardPlan.stream_columns)
            harr = torch.empty((len(idx), n), dtype=torch.int64).pin_memory()
            full = synth_columns(torch, dev, cols, n, 1)
            harr.copy_(full[torch.tensor(idx, device=dev)] if idx else full[:0])
            del full

            def e2e_step():
                cap[:] = state.commit_host(harr)     # chunked / streamed H2D behind the NTTs and the hashing
            h2d = len(idx) * n * 8
        for _ in range(2):
            e2e_step()
        barrier()
        ta = time.perf_counter()
        for _ in range(a.steps):
            e2e_step()
        barrier()
        dt = time.perf_counter() - ta
        if world > 1:
            t = torch.tensor([dt], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
            hb = torch.tensor([h2d], dtype=torch.int64, device=dev)
            dist.all_reduce(hb)
            h2d = int(hb.item())
        parity["e2e_cap_equals_device_cap"] = bool(np.array_equal(cap, cap_dev))
        e2e_stage_ms, _ = ctx.stage_times()
        host_plan = "gl_commit" if world == 1 else (state._host_impl.exchange if state._host_impl is not None else state.exchange)
        e2e = {"value": round(cols * n * a.steps / dt / 1e6, 3), "unit": UNIT, "h2d_bytes_per_step": int(h2d), "plan": host_plan,
               "stage_ms_last_call_rank0": {k: round(v, 3) for k, v in e2e_stage_ms.items() if v},
               "d2h_bytes_per_step": int(cap.nbytes), "ms_per_step": round(dt / a.steps * 1e3, 3),
               "api": "gl_commit (include/gl_commit.h) with pinned host columns; leaves/digests stay device-resident behind the handle"
                      if world == 1 else "ShardedCommit.commit_host: pinned host columns -> gl_commit_coset_stream (waves: H2D, iNTT, NVLink pulls and own-coset NTTs of "
                      "wave w+1 behind the hashing of wave w) or gl_lde_scatter (chunked H2D behind the NTTs) -> cap to host; plan: "
                      + (state._host_impl.exchange if state._host_impl is not None else state.exchange)}

    if world > 1:
        if os.environ.get("GL_BENCH_PHASES"):
            print(f"rank {rank} host-side phase ms of the last commit: " + json.dumps({k: round(v, 3) for k, v in state.phase_ms.items()}),
                  file=sys.stderr, flush=True)
        state.close()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (leaf hashing), live CUDA-event time from the context's stage events -------
    # The BINDING line leads: this kernel is limited by the SM issue port (integer + fp64 work on a 64-bit prime field, no
    # contraction), so `roofline` = executed warp-instructions/s against one warp-instruction per sub-partition per clock.  Its
    # numerator is EXECUTED instructions (ncu smsp__inst_executed per permutation x the live permutation rate): it measures how full
    # the issue port is, not how lean the code is — `imad_wide_floor` is the algorithmic floor (the 1652 IMAD.WIDE.U32 of the 118
    # S-boxes at the measured multiplier rate) and `hbm` the contractual memory line (which does not bind).
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    peak_gbs, peak_src = (peaks["hbm_gbs"], "measured (MEASURED_PEAKS.json)") if "hbm_gbs" in peaks else (6650.0, "fallback (B200_PROFILING.md)")
    R = n << r
    rows_local = R // world
    leaf_ms = stage_acc.get("leaf_hash", 0.0) / a.steps
    alg_bytes = rows_local * (cols * 8 + 32)               # read every leaf word once, write one 32-byte digest per leaf
    perms_leaf = rows_local * ((cols + 7) // 8)
    roof = None
    if leaf_ms > 0:
        ach = alg_bytes / (leaf_ms * 1e-3) / 1e9
        hbm = {"bound": "hbm", "achieved": round(ach, 2), "peak": peak_gbs, "unit": "GB/s", "frac": round(ach / peak_gbs, 5),
               "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes, "traffic": None,
               "note": "contractual memory line; does not bind (DESIGN.md §4)"}
        roof = {"kernel": "merkle::leaf_hash_kernel", "bound": "hbm", "achieved": hbm["achieved"], "peak": peak_gbs, "unit": "GB/s",
                "frac": hbm["frac"], "traffic": None, "ms_per_launch": round(leaf_ms, 3), "hbm": hbm}
        try:
            prof = json.load(open(os.path.join(ROOT, "profiles", "leaf_hash_profile.json")))
            if prof.get("cols") == cols:
                ipp = prof["warp_inst_per_launch"] / (prof["rows"] * ((cols + 7) // 8) / 32)
                sm_mhz = (clocks or {}).get("sm_mhz") or peaks.get("sm_max_mhz", 1965.0)
                n_smsp = 148 * 4
                peak_issue = n_smsp * sm_mhz * 1e6
                perm_rate = perms_leaf / (leaf_ms * 1e-3)
                ach_issue = perm_rate / 32 * ipp
                clk_per_warp_perm = n_smsp * sm_mhz * 1e6 / (perm_rate / 32)
                wide_per_perm, wide_rate = prof.get("imad_wide_per_permutation", 1652), prof.get("imad_wide_warp_inst_per_clk_per_smsp", 0.175)
                if prof.get("rows") == rows_local:
                    hbm["traffic"] = prof["dram_bytes_per_launch"]
                roof = {"kernel": "merkle::leaf_hash_kernel", "bound": "sm-issue", "achieved": round(ach_issue, 1), "peak": peak_issue,
                        "unit": "warp-inst/s", "frac": round(ach_issue / peak_issue, 4), "traffic": hbm["traffic"],
                        "ms_per_launch": round(leaf_ms, 3), "permutations_per_s": round(perm_rate, 1),
                        "warp_inst_per_permutation": round(ipp, 1), "sm_mhz": sm_mhz,
                        "numerator": "executed warp instructions (ncu smsp__inst_executed / permutation x live permutation rate): issue-port "
                                     "occupancy, not efficiency",
                        "peak_source": "148 SMs x 4 sub-partitions x 1 warp-inst/clk x SM clock sampled during the run",
                        "profile": prof.get("source"),
                        "imad_wide_floor": {"frac": round(wide_per_perm / wide_rate / clk_per_warp_perm, 4),
                                            "imad_wide_per_permutation": wide_per_perm, "warp_inst_per_clk_per_smsp": wide_rate,
                                            "clk_per_warp_permutation": round(clk_per_warp_perm, 1),
                                            "note": "algorithmic floor: 118 S-boxes x 14 IMAD.WIDE.U32 at the measured multiplier rate "
                                                    "(profiles/r01_ubench2_issue_port.txt)"},
                        "hbm": hbm}
        except (OSError, KeyError):
            pass
        # the NTT passes (second kernel by time) against the HBM line: every pass reads and writes the matrix once
        pitch = (cols // world + 7) // 8 * 8 if world > 1 else (cols + 7) // 8 * 8
        n_pass = -(-log_n // 10) if log_n >= 3 else 1
        for stage, n_ntt in (("intt", 1), ("lde", 1 << r)):
            ms_st = stage_acc.get(stage, 0.0) / a.steps
            if ms_st > 0:
                b = 16 * n * pitch * n_pass * n_ntt
                roof.setdefault("ntt", {})[stage] = {"bound": "hbm", "achieved": round(b / (ms_st * 1e-3) / 1e9, 1), "peak": peak_gbs, "unit": "GB/s",
                                                     "frac": round(b / (ms_st * 1e-3) / 1e9 / peak_gbs, 4), "algorithmic_bytes": b,
                                                     "launches": n_pass * n_ntt, "ms": round(ms_st, 3)}

    cpu = None if (a.no_cpu_baseline or world > 1) else cpu_baseline(a)   # rank 0 at N=1 only

    line = {"metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": round(ms_per_step, 4), "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u64 (Goldilocks field, integer + exact fp64 limb arithmetic)", "data": "synthetic",
            "config": {"workload": workload_name(a), "log_n": log_n, "n_cols": cols, "rate_bits": r, "cap_height": h,
                       "sharding": "none" if world == 1 else (f"columns/{world} -> " + {
                           "coset": "iNTT -> coefficient blocks pulled over NVLink (one contiguous copy per peer, overlapped with the NTTs) -> own cosets of all columns",
                           "p2p": "LDE -> coset rows shipped to their owners by the copy engines behind the next coset's NTT",
                           "nccl": "LDE -> NCCL all-to-all + repack"}[state.exchange] + f" -> leaf ranges/{world}"),
                       "l2": "inputs (%.2f GB) and leaves (%.2f GB) exceed the 126 MB L2; no flush needed" % (cols * n * 8 / 1e9, R * cols * 8 / 1e9),
                       "permutations_per_step": perms_per_commit(log_n, cols, r, h)},
            "stage_ms": {k: round(v / a.steps, 4) for k, v in stage_acc.items()},
            "clocks": clocks, "gpu_launches": launches, "e2e": e2e, "roofline": roof, "cpu_baseline": cpu, "parity": parity}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    if parity["match"] is False or parity.get("e2e_cap_equals_device_cap") is False:
        raise SystemExit("PARITY MISMATCH: the Merkle cap differs from the oracle's golden (see the `parity` object)")


if __name__ == "__main__":
    main()
