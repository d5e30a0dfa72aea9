"""Generate ``tests/golden/reference_wrappers.json``.

Runs the UNMODIFIED reference ``Index`` / ``QueryProcessor`` (imported from the original project's
checkout at ``BASELINE.json``'s ``reference_path`` or ``MLV_REFERENCE_ROOT``, reference
``src/mlvectordb/implementations/index.py`` and ``query_processor.py``) over the exact hnswlib stand-in (``oracle/hnswlib_exact.py``) and records what
they return.  The reference is not part of this repository, so the outputs are committed; the inputs are
regenerated from ``oracle/synthetic.py`` by the tests (only seeds are stored).

PARITY UNPINNED: the arithmetic under the wrappers is the oracle's restatement of hnswlib
0.8.0, not hnswlib itself (absent from this image) -- these fixtures pin the *wrapper*
behaviour (clamping, score transform, tombstones, rebuild, ordering), and the oracle's
numbers at the time of generation.

Usage:  python tests/golden/make_golden.py
"""
from __future__ import annotations

import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import refload, synthetic  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_wrappers.json")


def run_case(ref, case):
    """Execute one scripted case against the reference Index; returns the search records."""
    d, seed = case["dim"], case["seed"]
    index = ref.Index(space=case["space"])
    vec_of = {}      # (ns, ordinal) -> Vector
    ordinal_of = {}  # uuid -> (ns, ordinal)
    records = []
    for op in case["ops"]:
        kind = op["op"]
        if kind == "add":
            ns = op["ns"]
            data = synthetic.rows(seed, op["first"], op["n"], d, scaled=case.get("scaled", False))
            vs = [ref.Vector(values=row) for row in data]
            for i, v in enumerate(vs):
                vec_of[(ns, op["first"] + i)] = v
                ordinal_of[v.id] = (ns, op["first"] + i)
            index.add(vs, ns)
        elif kind == "remove":
            ns = op["ns"]
            ids = [vec_of[(ns, o)].id for o in op["ordinals"] if (ns, o) in vec_of]
            index.remove(ids, ns)
            records.append({"op": "rebuild_required", "ns": ns, "value": bool(index.is_rebuild_required(ns))})
        elif kind == "rebuild":
            source = {ns: [vec_of[(ns, o)] for o in ords] for ns, ords in op["source"].items()}
            index.rebuild(source, metric=op["metric"])
        elif kind == "search":
            ns = op["ns"]
            if "query_row" in op:     # planted: the query IS a stored row
                qv = synthetic.rows(seed, op["query_row"], 1, d, scaled=case.get("scaled", False))[0]
            else:
                qv = synthetic.queries(seed, op["query"] + 1, d)[op["query"]]
            if op.get("as_list"):
                qv = [float(x) for x in qv]
            res = index.search(ref.VectorDTO(values=qv, metadata={}), top_k=op["k"], namespace=ns, metric=op["metric"])
            records.append({
                "op": "search", "ns": ns, "k": op["k"], "metric": op["metric"],
                "ordinals": [ordinal_of[r.vector_id][1] for r in res],
                "scores": [float(r.score) for r in res],
            })
        else:
            raise ValueError(kind)
    return records


def cases():
    cs = []
    # config 1 (BASELINE.json configs[0]): 10k x 128 cosine k=10 single queries -- exactly the
    # reference's 10 000-row cap (index.py:37)
    cs.append({
        "name": "c1_cosine_10k_128", "space": "cosine", "dim": 128, "seed": 42, "scaled": True,
        "ops": [{"op": "add", "ns": "default", "first": 0, "n": 10000}]
        + [{"op": "search", "ns": "default", "k": 10, "metric": "cosine", "query": i} for i in range(6)]
        + [{"op": "search", "ns": "default", "k": 10, "metric": "cosine", "query_row": 4242},
           {"op": "search", "ns": "default", "k": 1, "metric": "cosine", "query": 6},
           {"op": "search", "ns": "default", "k": 100, "metric": "cosine", "query": 7}],
    })
    # l2 index searched with the REST default metric="cosine": score = 1 - squared L2 (quirk Q1)
    cs.append({
        "name": "l2_space_cosine_metric_quirk", "space": "l2", "dim": 16, "seed": 7,
        "ops": [{"op": "add", "ns": "a", "first": 0, "n": 300},
                {"op": "search", "ns": "a", "k": 5, "metric": "l2", "query": 0},
                {"op": "search", "ns": "a", "k": 5, "metric": "cosine", "query": 0},
                {"op": "search", "ns": "a", "k": 5, "metric": "l2", "query_row": 17, "as_list": True},
                {"op": "search", "ns": "missing", "k": 5, "metric": "l2", "query": 0}],
    })
    # inner product, odd dimension, incremental adds into two namespaces
    cs.append({
        "name": "ip_two_namespaces_incremental", "space": "ip", "dim": 37, "seed": 11,
        "ops": [{"op": "add", "ns": "x", "first": 0, "n": 50},
                {"op": "add", "ns": "y", "first": 1000, "n": 70},
                {"op": "add", "ns": "x", "first": 50, "n": 25},
                {"op": "search", "ns": "x", "k": 8, "metric": "ip", "query": 0},
                {"op": "search", "ns": "y", "k": 8, "metric": "ip", "query": 0},
                {"op": "search", "ns": "x", "k": 200, "metric": "ip", "query": 1}],   # k clamped to 75
    })
    # tombstones: remove below and above the 0.2 rebuild threshold, unknown ids, k > live
    cs.append({
        "name": "l2_remove_threshold_rebuild", "space": "l2", "dim": 24, "seed": 3,
        "ops": [{"op": "add", "ns": "r", "first": 0, "n": 40},
                {"op": "add", "ns": "keep", "first": 500, "n": 10},
                {"op": "remove", "ns": "r", "ordinals": [0, 1, 2]},               # 3/40 < 0.2
                {"op": "search", "ns": "r", "k": 5, "metric": "l2", "query_row": 1},
                {"op": "remove", "ns": "r", "ordinals": [1, 2, 999]},            # already gone / unknown: no-op
                {"op": "remove", "ns": "r", "ordinals": [3, 4, 5, 6, 7]},        # 8/40 = 0.2 -> flag
                {"op": "search", "ns": "r", "k": 40, "metric": "l2", "query": 2},  # clamped to 32
                {"op": "rebuild", "metric": "l2", "source": {"r": list(range(8, 40))}},
                {"op": "search", "ns": "r", "k": 3, "metric": "l2", "query": 2},
                {"op": "search", "ns": "keep", "k": 3, "metric": "l2", "query": 2}],  # Q6: wiped -> []
    })
    # everything removed -> []
    cs.append({
        "name": "cosine_remove_all", "space": "cosine", "dim": 8, "seed": 5,
        "ops": [{"op": "add", "ns": "z", "first": 0, "n": 2},
                {"op": "remove", "ns": "z", "ordinals": [0, 1]},
                {"op": "search", "ns": "z", "k": 5, "metric": "cosine", "query": 0}],
    })
    return cs


def query_processor_case(ref):
    """reference tests/test_query_processor.py:52-67 restated with recorded outputs."""
    qp = ref.QueryProcessor(ref.StorageEngineInMemory(), ref.Index(space="cosine"))
    vs = [([1, 0, 0], "A"), ([0, 1, 0], "B"), ([0.8, 0.2, 0], "C")]
    qp.upsert_many([ref.VectorDTO(values=v, metadata={"label": l}) for v, l in vs])
    res = qp.find_similar(ref.VectorDTO(values=[0.9, 0.1, 0], metadata={}), top_k=3)
    return {"vectors": vs, "query": [0.9, 0.1, 0], "k": 3,
            "labels": [r["metadata"]["label"] for r in res],
            "scores": [float(r["score"]) for r in res]}


def main():
    ref = refload.load()
    out = {"generator": "tests/golden/make_golden.py", "parity": "unpinned (oracle restates hnswlib 0.8.0)",
           "cases": [], "query_processor": query_processor_case(ref)}
    for c in cases():
        out["cases"].append({**c, "records": run_case(ref, c)})
    with open(OUT, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    main()
