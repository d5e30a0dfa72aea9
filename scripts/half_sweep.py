"""Launch-shape sweep of the shadow scan at the headline shape (dev tool): --tier fp16 (scan_kernel_half) or q8
(scan_kernel_q8, the int8 shadow)."""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mlvectordb_b200 import DeviceShard  # noqa: E402
from oracle import synthetic  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--rows", type=int, default=10_000_000)
ap.add_argument("--dim", type=int, default=768)
ap.add_argument("--reps", type=int, default=12)
ap.add_argument("--tier", default="fp16", choices=["fp16", "q8"])
a = ap.parse_args()
s = DeviceShard(a.dim, "cosine", capacity=a.rows)
s.add_synthetic(42, 0, a.rows, True)
Q = synthetic.queries(43, a.reps, a.dim)
s.set_timing(True)
DEFAULTS = {"cw": 0, "r": 0, "stage_kb": 0, "max_stages": 8, "tile_batch": 4}


def run(half, **kw):
    # half: 0 = the fp32 scan, 1 = the tier under test
    s.set_tuning("scan_half", 0 if not half else (1 if a.tier == "fp16" else -1))
    s.set_tuning("scan_q8", 1 if a.tier == "q8" else 0)
    for key, v in {**DEFAULTS, **kw}.items():
        s.set_tuning(key, v)
    try:
        s.search(Q[:1], 10)
        s.scan_time_ms()
        for i in range(a.reps):
            s.search(Q[i:i + 1], 10)
        ms, n = s.scan_time_ms()
    except Exception as e:  # noqa: BLE001
        return {"half": half, **kw, "error": str(e)[:80]}
    per = ms / n
    # the int8 pass reads rows of whole 128-byte chunks and one fp32 scale per row
    bytes_read = a.rows * (a.dim * 4 if not half else (a.dim * 2 if a.tier == "fp16" else (a.dim + 127) // 128 * 128 + 4))
    return {"half": half, "tier": a.tier if half else "fp32", **kw, "search_ms": round(per, 4), "bytes_read_GBps": round(bytes_read / per / 1e6, 1),
            "B_alg_GBps": round(a.rows * a.dim * 4 / per / 1e6, 1)}


print(json.dumps(run(0)), flush=True)
print(json.dumps(run(1)), flush=True)
for cw in ((2, 4, 6) if a.tier == "fp16" else (4, 5, 6, 7)):
    for r in (0,):
        for kb in (24, 48, 96):
            print(json.dumps(run(1, cw=cw, r=r, stage_kb=kb)), flush=True)
for ms_ in (4, 16):
    print(json.dumps(run(1, max_stages=ms_)), flush=True)
s.close()
