"""Grouped search (``mlv_index_search_grouped``) against plain search on the headline data: 10M x 768 cosine rows from the
synthetic generator, k = 10, groups of 1, 16 and 1024 consecutive rows.

Both sides run in one process and alternate, call by call.  The plain side is forced onto the fp32 pass ("scan_half" 0,
"gemm" 0, staged host path) so that the same kernel family is compared; the plain search with default tuning (shadow
scans, tensor-core batch path, latency path) is reported for context.  Single queries and 8-query passes; host wall clock around each blocking call.  Prints
one JSON line per (group size, batch), and with --out appends them to that file.

    python scripts/bench_grouped.py [--rows 10000000] [--reps 40] [--out profiles/grouped_10Mx768.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_name_and_power():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--dim", type=int, default=768)
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--reps", type=int, default=40)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from mlvectordb_b200 import DeviceShard
    s = DeviceShard(a.dim, "cosine", capacity=a.rows)
    s.add_synthetic(42, 0, a.rows, scaled=True)
    Q = np.random.default_rng(43).standard_normal((8 * a.reps, a.dim), dtype=np.float32)
    card = gpu_name_and_power()
    lines = []

    def timed(fn, batches):
        fn(batches[0])                                     # warm the shape
        t = []
        for b in batches:
            t0 = time.perf_counter()
            fn(b)
            t.append(time.perf_counter() - t0)
        return float(np.median(t)) * 1e3

    def plain_fp32(q):
        s.set_tuning("scan_half", 0)
        s.set_tuning("gemm", 0)
        s.set_tuning("fast_host", 0)
        s.search(q, a.k)
        s.set_tuning("scan_half", -1)
        s.set_tuning("gemm", -1)
        s.set_tuning("fast_host", 1)

    for shift in (0, 4, 10):
        s.set_column(0, (np.arange(a.rows, dtype=np.int64) >> shift).astype(np.int32))
        for nq in (1, 8):
            batches = [Q[i * nq:(i + 1) * nq] for i in range(a.reps)]
            g_ms, p_ms = [], []
            for b in batches:                              # alternate the two, call by call
                g_ms.append(timed(lambda q: s.search_grouped(q, a.k, 0), [b]))
                p_ms.append(timed(plain_fp32, [b]))
            d_ms = timed(lambda q: s.search(q, a.k), batches)
            rec = {"rows": a.rows, "dim": a.dim, "space": "cosine", "k": a.k, "group_rows": 1 << shift, "nq": nq,
                   "grouped_ms": round(float(np.median(g_ms)), 4), "plain_fp32_ms": round(float(np.median(p_ms)), 4),
                   "plain_default_ms": round(d_ms, 4),
                   "grouped_over_plain_fp32": round(float(np.median(g_ms)) / float(np.median(p_ms)), 4),
                   "gpu": card, "timing": "host wall clock per blocking call, median of reps"}
            print(json.dumps(rec), flush=True)
            lines.append(rec)
    if a.out:
        with open(a.out, "a") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")
    s.close()


if __name__ == "__main__":
    main()
