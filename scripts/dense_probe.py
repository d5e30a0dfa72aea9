import json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mlvectordb_b200 import DeviceShard
from oracle import synthetic
dim, nq, k = 768, 4096, 100
Q = synthetic.queries(43, nq, dim)
for rows in (256, 512, 2304, 20736):
    s = DeviceShard(dim, "l2", capacity=rows)
    s.add_synthetic(42, 0, rows, False)
    s.set_timing(True)
    s.set_tuning("gemm", 1)
    for wide in (3, 0):
        s.set_tuning("gemm_wide", wide)
        for predict in (1, 0):
            s.set_tuning("gemm_predict", predict)
            s.search(Q, k); s.gemm_stats()
            b = s.gemm_stats()
            for _ in range(5): s.search(Q, k)
            st = s.gemm_stats()
            print(json.dumps({"rows": rows, "wide": wide, "predict": predict, "gemm_us_per_batch": round(st["gemm_ms"] / 5 * 1e3, 1),
                              "rounds": (st["rounds"] - b["rounds"]) / 5}), flush=True)
    s.close()
