"""CPU: the oracle against the committed golden fixtures (what the reference wrappers returned) and against itself
(C port vs numpy)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import cscan, exact, hnswlib_exact, synthetic

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "reference_wrappers.json")


def _golden():
    with open(GOLDEN) as f:
        return json.load(f)


@pytest.mark.parametrize("case", _golden()["cases"], ids=lambda c: c["name"])
def test_oracle_reproduces_golden_searches(case):
    """Replay each scripted case with plain oracle calls (no reference code): the live set is
    tracked here, the expected hits come from the committed reference-wrapper outputs."""
    d, seed, space = case["dim"], case["seed"], case["space"]
    ns_rows, ns_space = {}, {}            # ns -> {ordinal: row}
    records = iter(case["records"])
    for op in case["ops"]:
        kind = op["op"]
        if kind == "add":
            data = synthetic.rows(seed, op["first"], op["n"], d, scaled=case.get("scaled", False))
            ns_rows.setdefault(op["ns"], {}).update({op["first"] + i: data[i] for i in range(op["n"])})
            ns_space.setdefault(op["ns"], space)
        elif kind == "remove":
            next(records)
            for o in op["ordinals"]:
                ns_rows.get(op["ns"], {}).pop(o, None)
        elif kind == "rebuild":
            all_rows = {o: r for rows in ns_rows.values() for o, r in rows.items()}
            ns_rows = {ns: {o: all_rows[o] for o in ords} for ns, ords in op["source"].items()}
            ns_space = {ns: op["metric"] for ns in op["source"]}
        else:
            rec = next(records)
            rows = ns_rows.get(op["ns"], {})
            if not rows:
                assert rec["ordinals"] == []
                continue
            ords = np.array(sorted(rows))
            X = np.stack([rows[o] for o in ords])
            if "query_row" in op:
                q = synthetic.rows(seed, op["query_row"], 1, d, scaled=case.get("scaled", False))[0]
            else:
                q = synthetic.queries(seed, op["query"] + 1, d)[op["query"]]
            k = min(op["k"], len(ords))
            L, D = exact.knn(X, q, k, ns_space[op["ns"]])
            got_scores = D[0].astype(np.float64)
            exp_scores = np.array(rec["scores"], dtype=np.float64)
            if op["metric"] == "cosine":
                exp_scores = 1 - exp_scores
            assert exact.check_topk_parity(ords[L[0]], got_scores, rec["ordinals"], exp_scores) is None


def test_stand_in_follows_hnswlib_error_semantics():
    idx = hnswlib_exact.Index(space="l2", dim=3)
    idx.init_index(max_elements=4)
    idx.add_items(np.eye(3, dtype=np.float32), np.arange(3))
    with pytest.raises(RuntimeError):
        idx.knn_query(np.zeros((1, 2), np.float32), k=1)          # wrong dimension
    with pytest.raises(RuntimeError):
        idx.knn_query(np.zeros((1, 3), np.float32), k=4)          # cannot fill k
    with pytest.raises(RuntimeError):
        idx.add_items(np.ones((2, 3), np.float32), np.array([10, 11]))  # exceeds max_elements
    idx.mark_deleted(1)
    with pytest.raises(RuntimeError):
        idx.mark_deleted(1)
    labels, dists = idx.knn_query(np.array([[0, 1, 0]], np.float32), k=2)
    assert 1 not in labels[0].tolist() and labels.dtype == np.uint64 and dists.dtype == np.float32
    assert idx.get_current_count() == 3                            # deleted rows still count (index.py:56)
    lab2, _ = idx.knn_query(np.array([[1, 0, 0]], np.float32), k=1, filter=lambda l: l != 0)
    assert lab2[0].tolist() == [2]                                 # 0 filtered, 1 deleted
    with pytest.raises(RuntimeError):
        idx.knn_query(np.array([[1, 0, 0]], np.float32), k=2, filter=lambda l: l != 0)


def test_distance_definitions_known_answers():
    """Hand-computed values of the three hnswlib spaces (also reference README.md probe, SURVEY Q1)."""
    X = np.array([[1, 0, 0], [0, 2, 0]], np.float32)
    q = np.array([1, 0, 0], np.float32)
    assert exact.distances(X, q, "l2").tolist() == [0.0, 5.0]
    assert exact.distances(X, q, "ip").tolist() == [0.0, 1.0]
    L, D = exact.knn(X, q, 2, "cosine")
    assert L[0].tolist() == [0, 1] and D[0].tolist() == pytest.approx([0.0, 1.0], abs=1e-7)
    # l2 index searched with metric="cosine": 1 - squared L2 -> [1, -4]  (SURVEY.md Q1 probe)
    assert [1 - float(x) for x in exact.distances(X, q, "l2")] == [1.0, -4.0]
    n = exact.normalize_rows(np.array([[3, 4]], np.float32))
    assert n[0].tolist() == pytest.approx([0.6, 0.8], rel=1e-6)
    assert exact.normalize_rows(np.zeros((1, 4), np.float32))[0].tolist() == [0, 0, 0, 0]   # 1e-30 guard


@pytest.mark.parametrize("space", ["l2", "ip", "cosine"])
@pytest.mark.parametrize("dim", [3, 16, 37, 768])
def test_c_port_matches_numpy_oracle(space, dim):
    X = synthetic.rows(3, 0, 3000, dim, scaled=True)
    Q = synthetic.queries(3, 4, dim)
    Xn = cscan.normalize(X) if space == "cosine" else X
    Qn = cscan.normalize(Q) if space == "cosine" else Q
    if space == "cosine":
        np.testing.assert_allclose(Xn, exact.normalize_rows(X), rtol=1e-6, atol=1e-9)
    for simd16 in (False, True):
        l, d, c = cscan.knn(Xn, Qn, 10, space, simd16=simd16)
        L, D = exact.knn(X, Q, 10, space)
        for i in range(4):
            assert c[i] == 10
            assert exact.check_topk_parity(l[i], d[i], L[i], D[i]) is None
    # filter bitmap path of the C port
    mask = synthetic.buckets(3, 0, 3000) < 10
    l, d, c = cscan.knn(Xn, Qn, 10, space, allow_bitmap=synthetic.bitmap_from_mask(mask))
    L, D = exact.knn(X, Q, 10, space, allow=mask)
    for i in range(4):
        assert exact.check_topk_parity(l[i][:c[i]], d[i][:c[i]], L[i], D[i]) is None


def test_synthetic_generator_c_equals_numpy():
    for seed, first, n, d, scaled in ((42, 0, 64, 128, True), (7, 10**12, 33, 5, False), (1, 999, 10, 770, True)):
        assert np.array_equal(cscan.fill_synthetic(seed, first, n, d, scaled), synthetic.rows(seed, first, n, d, scaled))
    x = synthetic.rows(42, 0, 2000, 64)
    assert -1.0 <= x.min() < -0.99 and 0.99 < x.max() < 1.0 and abs(float(x.mean())) < 0.01
    b = synthetic.buckets(42, 0, 100000)
    assert b.min() == 0 and b.max() == 99 and abs((b < 10).mean() - 0.10) < 0.01
    m = np.zeros(70, bool)
    m[[0, 31, 32, 69]] = True
    w = synthetic.bitmap_from_mask(m)
    assert w.dtype == np.uint32 and w.tolist() == [0x80000001, 0x1, 0x20]


def test_streaming_knn_equals_in_memory_and_range_semantics():
    X = synthetic.rows(9, 0, 5000, 24)
    Q = synthetic.queries(9, 3, 24)
    L1, D1 = exact.knn(X, Q, 25, "l2", chunk_rows=700)
    L2, D2 = exact.knn(X, Q, 25, "l2", chunk_rows=10**6)
    for a, b, c, d in zip(L1, L2, D1, D2):
        assert a.tolist() == b.tolist() and np.array_equal(c, d)
    radius = float(D1[0][9])
    Lr, Dr = exact.range_search(X, Q[:1], radius, "l2")
    assert Lr[0].tolist() == L1[0][:10].tolist()           # d <= radius is inclusive
    assert exact.check_topk_parity([1, 2], [0.5, 0.5 + 1e-9], [2, 1], [0.5, 0.5]) is None   # tie swap allowed
    assert exact.check_topk_parity([1, 3], [0.5, 0.9], [1, 2], [0.5, 0.6]) is not None


@pytest.mark.parametrize("space,scaled", [("l2", False), ("ip", True), ("cosine", True)])
def test_streamed_synthetic_oracle_equals_the_materialised_one(space, scaled):
    """orc_knn_synthetic / orc_range_synthetic regenerate rows on the fly; they must be bit-identical to
    fill_synthetic -> normalize -> knn on the same rows (that is what lets full-size GPU tests use them)."""
    n, d, k, first = 20_000, 96, 10, 1000
    Q = synthetic.queries(7, 5, d)
    X = cscan.fill_synthetic(42, first, n, d, scaled)
    Xn = cscan.normalize(X) if space == "cosine" else X
    Qn = cscan.normalize(Q) if space == "cosine" else Q
    L0, D0, C0 = cscan.knn(Xn, Qn, k, space, first_label=first)
    L1, D1, C1 = cscan.knn_synthetic(42, first, n, d, scaled, Q, k, space)
    assert np.array_equal(L0, L1) and np.array_equal(D0, D1) and np.array_equal(C0, C1)
    mask = synthetic.buckets(3, 0, n) < 10
    L2, D2, C2 = cscan.knn_synthetic(42, first, n, d, scaled, Q, k, space, allow=mask)
    L3, D3, C3 = cscan.knn(Xn, Qn, k, space, allow_bitmap=synthetic.bitmap_from_mask(mask), first_label=first)
    assert np.array_equal(L2, L3) and np.array_equal(D2, D3) and np.array_equal(C2, C3)
    Lr, Dr = exact.knn(X, Q, k, space, allow=mask)      # and within tolerance of the numpy restatement
    for i in range(5):
        assert exact.check_topk_parity(L2[i] - first, D2[i], Lr[i], Dr[i]) is None
    radius = float(D1[0, -1])
    hits = cscan.range_synthetic(42, first, n, d, scaled, Q, radius, space, max_hits=4)   # forces the retry
    assert hits[0][0].tolist() == L1[0].tolist() and np.array_equal(hits[0][1], D1[0])
    Lx, Dx = exact.range_search(X, Q, radius, space)
    for i in range(5):
        assert len(hits[i][0]) == len(Lx[i]) or abs(len(hits[i][0]) - len(Lx[i])) <= 2   # ties at the radius
    assert cscan.check_knn_synthetic(L1, D1, C1, 42, first, n, d, scaled, Q, k, space) is None
    bad = L1.copy()
    bad[2, 3] = first + n - 1
    assert cscan.check_knn_synthetic(bad, D1, C1, 42, first, n, d, scaled, Q, k, space) is not None
    assert np.array_equal(cscan.distances_synthetic(42, L1[1], d, scaled, Q[1], space), D1[1])


def test_oracle_thread_count_ignores_omp_num_threads():
    """torchrun exports OMP_NUM_THREADS=1; the reference arm must still use every core it may run on."""
    code = ("import os, sys; sys.path.insert(0, %r); from oracle import cscan; "
            "print(cscan.num_threads(), cscan.use_all_cores(), cscan.host_threads())" % ROOT)
    out = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, OMP_NUM_THREADS="1"),
                         capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr[-1000:]
    before, after, cores = (int(x) for x in out.stdout.split())
    assert before == 1 and after == cores
