"""Device time of OpeningSet::new (gl_batch_eval) against what a host-side OpeningSet::new would pay; prints one JSON line.

    python tools/opening_set_bench.py [--repeats 30] [--warmup 5]

Shapes: the wrapper's four commits at 2^16 (constants+sigmas 86, wires 135, Z/partial products 20, quotient chunks 16; r = 3, cap 4),
with the Z commit at zeta and g*zeta in one call, and one 2^20 x 135 commit at one point.  Per shape:
  device_ms         host clock around the synchronous calls, warmed up, median of the repeats (per_call_ms: the same per call).
                    L2 is overwritten (256 MB device write) before every timed window, so the coefficients come from HBM.
  bytes_read        the live coefficient words the evaluation needs (N x columns x 8 B; each matrix is read once per call),
                    gb_per_s and hbm_fraction against the 6 548 GB/s copy rate DESIGN.md quotes.
  host_copy_bytes   what a host-side OpeningSet::new would first copy back (the same coefficients).
  oracle_ms         the host Horner of tests/opening_set_oracle.py (C + OpenMP, oracle_threads host threads) on the same
                    evaluations, median of 3.
  parity            sha256 of the device values == sha256 of the oracle's.
The GPU's name and power limit are read in the same run.  Needs a CUDA device: there is no CPU fallback.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import plonky25_b200 as g  # noqa: E402
import opening_set_oracle as oso  # noqa: E402
from oracle_c import splitmix_columns  # noqa: E402
import wrapper_pipeline as wp  # noqa: E402

HBM_COPY_GBPS = 6548.0


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as e:   # the measurement stands without the query; say why the fields are missing
        import torch
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"unavailable ({type(e).__name__})"}


def median_ms(fn, flush, repeats, warmup):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(repeats):
        flush()
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts))


def sha(arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a, dtype=np.uint64).tobytes())
    return h.hexdigest()


def measure(flush, calls, repeats, warmup):
    """calls: [(batch, [points])] — one gl_batch_eval each"""
    per_call = [median_ms(lambda b=b, pts=pts: g.eval_commitment(b, pts), flush, repeats, warmup) for b, pts in calls]
    total = median_ms(lambda: [g.eval_commitment(b, pts) for b, pts in calls], flush, repeats, warmup)
    dev = [g.eval_commitment(b, pts) for b, pts in calls]
    coeffs = [b.polynomials for b, _ in calls]
    ora, ts = None, []
    for _ in range(3):
        t0 = time.perf_counter()
        ora = [np.stack([oso.eval_ext(c, z) for z in pts]) for c, (_, pts) in zip(coeffs, calls)]
        ts.append((time.perf_counter() - t0) * 1e3)
    nbytes = sum(8 * b.merkle_tree.leaf_len << b.degree_log for b, _ in calls)
    rate = nbytes / (total * 1e-3) / 1e9
    return {"device_ms": round(total, 4), "per_call_ms": [round(t, 4) for t in per_call], "bytes_read": nbytes,
            "gb_per_s": round(rate, 1), "hbm_fraction": round(rate / HBM_COPY_GBPS, 4), "host_copy_bytes": nbytes,
            "oracle_ms": round(float(np.median(ts)), 2), "oracle_threads": oso.num_threads(), "parity": sha(dev) == sha(ora),
            "sha256": sha(dev)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    import torch
    ctx = g.Context(0)
    scrub = torch.empty(1 << 25, dtype=torch.float64, device="cuda")   # 256 MB > the 126 MB L2

    def flush():
        scrub.zero_()
        torch.cuda.synchronize()

    out = {"tool": "opening_set_bench", **gpu_info()}
    log_n = 16
    cols = wp.make_columns(log_n)
    batches = [(g.PolynomialBatch.from_coeffs if wp.IS_COEFFS[k] else g.PolynomialBatch.from_values)(list(c), 3, False, 4, ctx=ctx)
               for k, c in enumerate(cols)]
    zeta = (0x1234_5678_9ABC_DEF0 % g.api.P, 0x0FED_CBA9_8765_4321 % g.api.P)
    gz = wp._g_times(zeta, log_n)
    calls = [(batches[0], [zeta]), (batches[1], [zeta]), (batches[2], [zeta, gz]), (batches[3], [zeta])]
    out["wrapper_2p16"] = {"widths": list(wp.WIDTHS), "points": [len(p) for _, p in calls],
                           **measure(flush, calls, args.repeats, args.warmup)}
    for b in batches:
        b.merkle_tree.free()
    big = g.PolynomialBatch.from_values(list(splitmix_columns(77, 135, 1 << 20)), 1, False, 4, ctx=ctx)
    out["single_2p20x135"] = {"points": [1], **measure(flush, [(big, [zeta])], args.repeats, args.warmup)}
    big.merkle_tree.free()
    print(json.dumps(out))
    ctx.close()
    return 0 if out["wrapper_2p16"]["parity"] and out["single_2p20x135"]["parity"] else 1


if __name__ == "__main__":
    sys.exit(main())
