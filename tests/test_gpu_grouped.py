"""GPU: grouped search (``mlv_index_search_grouped``, ``scan_kernel_grouped``) against the existing device path.

The reference is the plain search itself: ``search`` with k = every live row (<= 1024), or ``range_search`` with radius
+inf, gives every candidate row's exact fp32-scan distance in (distance, row) order; walking that list as the contract
says (first row of every group not seen yet, up to k) must give the grouped answer bit for bit -- distances, rows,
groups and counts."""
import math
import zlib

import numpy as np
import pytest

from _grouped_oracle import grouped_topk
from oracle import exact, synthetic

pytestmark = pytest.mark.gpu

MISSING = exact.COLUMN_MISSING
KS = (1, 7, 10, 16, 32)
NQS = (1, 3, 8, 13)


def _shard(dim, space, capacity=0):
    from mlvectordb_b200 import DeviceShard
    return DeviceShard(dim, space, capacity=capacity)


def _all_rows(shard, Q, filt=None):
    """Every candidate row of every query ascending by (distance, row), from the plain device path."""
    live = shard.live
    if live <= 1024:
        d, r, c = shard.search(Q, max(live, 1), filt)
        return [(d[i, : c[i]], r[i, : c[i]]) for i in range(Q.shape[0])]
    return shard.range_search(Q, float("inf"), filt, max_hits=live)


def _walk(d, r, groups, k):
    """The contract's walk over one query's ascending (d, row) list; groups: code per row."""
    g = groups[r] if r.size else np.empty(0, np.int32)
    keep = g != MISSING
    d, r, g = d[keep], r[keep], g[keep]
    _, first = np.unique(g, return_index=True)
    sel = np.sort(first)[:k]
    return d[sel], r[sel], g[sel]


def _check(shard, Q, k, groups, filt=None, ref=None, got=None):
    ref = _all_rows(shard, Q, filt) if ref is None else ref
    dists, rows, grp, counts = shard.search_grouped(Q, k, 0, filt) if got is None else got
    for i in range(Q.shape[0]):
        ed, er, eg = _walk(ref[i][0], ref[i][1], groups, k)
        c = int(counts[i])
        assert c == len(er), (i, c, len(er))
        assert np.array_equal(rows[i, :c], er), (i, rows[i, :c], er)
        assert np.array_equal(dists[i, :c].view(np.uint32), ed.astype(np.float32).view(np.uint32)), i
        assert np.array_equal(grp[i, :c], eg), i
        assert np.all(np.isposinf(dists[i, c:])) and np.all(rows[i, c:] == -1) and np.all(grp[i, c:] == MISSING)
    return dists, rows, grp, counts


def _data(n, dim, seed):
    rng = np.random.default_rng(seed)
    return rng.standard_normal((n, dim)).astype(np.float32), rng.standard_normal((13, dim)).astype(np.float32), rng


def _layout(name, n, rng, X, Q, space):
    i = np.arange(n)
    if name == "own":
        return i.astype(np.int32)
    if name == "block16":
        return (i // 16).astype(np.int32)
    if name == "mod37":
        return (i % 37).astype(np.int32)
    if name == "one":
        return np.full(n, 5, np.int32)
    if name == "few":
        return (i % 5).astype(np.int32)
    if name == "huge_near":
        Xn, q = (exact.normalize_rows(X), exact.normalize_rows(Q[:1])[0]) if space == "cosine" else (X, Q[0])
        near = np.argsort(exact.distances(Xn, q, space), kind="stable")[: n // 3]
        g = i.astype(np.int32) + 1000
        g[near] = 7
        return g
    if name == "zipf":
        return (rng.zipf(1.6, n) % 211).astype(np.int32)
    raise ValueError(name)


LAYOUTS = ("own", "block16", "mod37", "one", "few", "huge_near", "zipf")


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("dim", [3, 100, 768])
@pytest.mark.parametrize("space", ["l2", "ip", "cosine"])
def test_grouped_matches_the_walk(space, dim, layout):
    n = 3000
    X, Q, rng = _data(n, dim, zlib.crc32(f"{space}/{dim}/{layout}".encode()))
    s = _shard(dim, space)
    s.add(X)
    groups = _layout(layout, n, rng, X, Q, space)
    s.set_column(0, groups)
    ref = _all_rows(s, Q)
    for k in KS:
        for nq in NQS:
            got = _check(s, Q[:nq], k, groups, ref=ref[:nq])
            if layout == "own":   # every row its own group: the plain search's answer
                d, r, c = s.search(Q[:nq], k)
                assert np.array_equal(got[1], r) and np.array_equal(got[0].view(np.uint32), d.view(np.uint32))
                assert np.array_equal(got[3], c)
    s.close()


def test_missing_values_and_rows_appended_after_the_column():
    n, dim = 2000, 64
    X, Q, rng = _data(n + 700, dim, 11)
    s = _shard(dim, "l2", capacity=n)
    s.add(X[:n])
    groups = (np.arange(n) % 50).astype(np.int32)
    groups[rng.random(n) < 0.3] = MISSING
    s.set_column(0, groups)
    s.add(X[n:])                                  # the matrix grows past the column: these rows have no group
    full = np.concatenate([groups, np.full(700, MISSING, np.int32)])
    assert np.array_equal(s.get_column(0), full)
    for k in (1, 10, 32):
        _check(s, Q[:8], k, full)
    # the appended rows are nearest: they must still not appear
    s2 = _shard(dim, "l2", capacity=n)
    s2.add(X[:n])
    s2.set_column(0, groups)
    s2.add(np.repeat(Q[:1], 300, axis=0))
    full2 = np.concatenate([groups, np.full(300, MISSING, np.int32)])
    _, rows, _, _ = _check(s2, Q[:1], 10, full2)
    assert rows.max() < n


def test_tombstones_filters_and_gathered_scans():
    n, dim = 6000, 48
    X, Q, rng = _data(n, dim, 12)
    s = _shard(dim, "cosine")
    s.add(X)
    groups = (rng.integers(0, 400, n)).astype(np.int32)
    s.set_column(0, groups)
    s.set_column(1, (np.arange(n) % 20).astype(np.int32))
    s.mark_deleted(np.flatnonzero(rng.random(n) < 0.2).astype(np.uint64))
    for k in (7, 32):
        _check(s, Q[:8], k, groups)
        mask = rng.random(n) < 0.5                       # per-call bitmap (gathered scan)
        _check(s, Q[:8], k, groups, filt=mask)
        sparse = rng.random(n) < 0.03                    # prepared and selective: gathered
        pf = s.prepare_filter(sparse)
        _check(s, Q[:8], k, groups, filt=pf)
        dense = rng.random(n) < 0.95                     # prepared and dense: streamed with a mask
        _check(s, Q[:8], k, groups, filt=s.prepare_filter(dense))
        wf = s.where([(1, "==", 3)])                     # 5 %: a device `where` filter, gathered
        _check(s, Q[:8], k, groups, filt=wf)
        pf.close()


def test_bound_filter_applies():
    n, dim = 3000, 32
    X, Q, rng = _data(n, dim, 13)
    s = _shard(dim, "l2")
    s.add(X)
    groups = (np.arange(n) // 7).astype(np.int32)
    s.set_column(0, groups)
    pf = s.prepare_filter(rng.random(n) < 0.1)
    from mlvectordb_b200.shard import _bound
    ref = _all_rows(s, Q[:3], pf)
    with _bound(s, pf):
        got = s.search_grouped(Q[:3], 10, 0)
    _check(s, Q[:3], 10, groups, ref=ref, got=got)


def test_compaction_moves_the_column():
    n, dim = 4000, 16
    X, Q, rng = _data(n, dim, 14)
    s = _shard(dim, "ip")
    s.add(X)
    groups = (rng.integers(0, 300, n)).astype(np.int32)
    s.set_column(0, groups)
    s.mark_deleted(np.flatnonzero(rng.random(n) < 0.4).astype(np.uint64))
    mapping = s.compact()
    keep = mapping >= 0
    moved = np.empty(int(keep.sum()), np.int32)
    moved[mapping[keep]] = groups[keep]
    assert np.array_equal(s.get_column(0), moved)
    for k in (1, 16, 32):
        _check(s, Q[:13], k, moved)


def test_exact_duplicates_inside_and_across_groups():
    n, dim = 2500, 24
    X, Q, rng = _data(n, dim, 15)
    near = X[0] * 0.0 + Q[0]
    X[100:140] = near                                  # 40 identical rows at distance 0 ...
    X[900:910] = near
    groups = (np.arange(n) % 90).astype(np.int32)
    groups[100:120] = 3                                # ... 20 of them in one group, the others across groups
    groups[905:910] = 3
    s = _shard(dim, "l2")
    s.add(X)
    s.set_column(0, groups)
    for k in (1, 7, 32):
        d, r, g, c = _check(s, Q[:4], k, groups)
        assert r[0, 0] == 100                           # the tie goes to the lowest row


@pytest.mark.parametrize("space", ["l2", "cosine"])
def test_list_stress_worst_member_first_under_tuning(space):
    """Rows ordered so the scan meets every group's members from worst to best; every group spread over all tiles."""
    n, dim = 24000, 100
    X, Q, rng = _data(n, dim, 16)
    Xn, q0 = (exact.normalize_rows(X), exact.normalize_rows(Q[:1])[0]) if space == "cosine" else (X, Q[0])
    X = X[np.argsort(-exact.distances(Xn, q0, space), kind="stable")]
    groups = (np.arange(n) % 61).astype(np.int32)
    s = _shard(dim, space)
    s.add(X)
    s.set_column(0, groups)
    Qs = np.concatenate([Q[:1], Q[1:8]])
    ref = _all_rows(s, Qs)
    base = {k: _check(s, Qs, k, groups, ref=ref) for k in (10, 32)}
    for key, values in (("ctas", (1, 7, 37)), ("cw", (2, 5, 16)), ("tile_batch", (1, 16))):
        for v in values:
            s.set_tuning(key, v)
            for k in (10, 32):
                got = _check(s, Qs, k, groups, ref=ref)
                assert all(np.array_equal(a, b) for a, b in zip(got, base[k])), (key, v, k)
        s.set_tuning(key, 0 if key != "tile_batch" else 4)


def test_argument_errors_and_a_column_never_written():
    from mlvectordb_b200 import _capi
    X, Q, _ = _data(500, 8, 17)
    s = _shard(8, "l2")
    s.add(X)
    s.set_column(0, np.arange(500, dtype=np.int32))
    for k, col, status in ((0, 0, _capi.MLV_E_INVALID), (33, 0, _capi.MLV_E_UNSUPPORTED), (5, 16, _capi.MLV_E_INVALID)):
        with pytest.raises(_capi.MlvError) as e:
            s.search_grouped(Q[:2], k, col)
        assert e.value.status == status
    d, r, g, c = s.search_grouped(Q[:3], 5, 4)          # never written: no groups, not an error
    assert (c == 0).all() and np.isposinf(d).all() and (r == -1).all() and (g == MISSING).all()
    for key in ("dynamic", "fused"):
        s.set_tuning(key, 0)
        with pytest.raises(_capi.MlvError) as e:
            s.search_grouped(Q[:1], 5, 0)
        assert e.value.status == _capi.MLV_E_UNSUPPORTED
        s.set_tuning(key, 1)
    _check(s, Q[:2], 5, np.arange(500, dtype=np.int32))
    s.mark_deleted(np.arange(500, dtype=np.uint64))      # nothing live
    d, r, g, c = s.search_grouped(Q[:2], 5, 0)
    assert (c == 0).all() and (g == MISSING).all()


def test_gpu_index_processor_and_rest_group_by():
    from fastapi.testclient import TestClient

    from _refshim import Storage
    from mlvectordb_b200 import GpuIndex, GpuQueryProcessor, VectorDTO
    from mlvectordb_b200.index import NotDeviceEvaluable
    from mlvectordb_b200.rest_api import GpuRestAPI

    class _Storage(Storage):
        @property
        def list_namespaces(self):
            return list(self._data)

        def get_storage_info(self):
            return {}

    rng = np.random.default_rng(18)
    n, dim = 400, 16
    X = rng.standard_normal((n, dim)).astype(np.float32)
    docs = [f"doc{int(v)}.pdf" for v in rng.integers(0, 30, n)]
    mds = [{"doc": docs[i], "page": i % 9, "tags": ["x"]} if i % 10 else {"page": i % 9} for i in range(n)]
    qp = GpuQueryProcessor(_Storage(), GpuIndex(space="cosine"))
    qp.upsert_matrix(X, "ns", metadata=mds)
    index = qp._index
    q = rng.standard_normal(dim).astype(np.float32)
    dto = VectorDTO(values=q.tolist(), metadata={})
    plain = index.search(dto, n, "ns", "cosine")
    by_id = {v.id: v.metadata for v in qp._storage.namespace_map["ns"]}
    want, seen = [], set()
    for hit in plain:
        doc = by_id[hit.vector_id].get("doc")
        if doc is not None and doc not in seen:
            seen.add(doc)
            want.append((hit.vector_id, hit.score))
    got = index.search(dto, 10, "ns", "cosine", group_by="doc")
    assert [(h.vector_id, h.score) for h in got] == want[:10]
    rows, scores, counts = index.search_batch(np.stack([q, q]), 32, "ns", metric="cosine", group_by="doc")
    assert counts.tolist() == [min(32, len(want))] * 2
    assert np.array_equal(scores[0, : counts[0]], np.array([s for _, s in want[:32]], np.float32))
    assert index.search(dto, 5, "ns", "cosine", group_by="never_seen") == []
    with pytest.raises(NotDeviceEvaluable):
        index.search(dto, 5, "ns", "cosine", group_by="tags")
    with pytest.raises(ValueError):
        index.search(dto, 33, "ns", "cosine", group_by="doc")
    # the processor composes group_by with filters, on the device and on the host
    hits = qp.find_similar(dto, 5, "ns", group_by="doc", filter={"page": 3})
    exp_pf, seen = [], set()
    for hit in plain:
        md = by_id[hit.vector_id]
        if md.get("page") == 3 and md.get("doc") is not None and md["doc"] not in seen:
            seen.add(md["doc"])
            exp_pf.append(hit.vector_id)
    assert [h["id"] for h in hits] == exp_pf[:5]
    assert len({h["metadata"]["doc"] for h in hits}) == len(hits)
    host = qp.find_similar(dto, 5, "ns", group_by="doc", filter=lambda md: md.get("page", 0) < 4)
    assert len({h["metadata"]["doc"] for h in host}) == len(host) and all(h["metadata"]["page"] < 4 for h in host)
    batch = qp.find_similar_batch([q, q], 10, "ns", group_by="doc", enrich=False)
    assert [h["id"] for h in batch[1]] == [v for v, _ in want[:10]]
    client = TestClient(GpuRestAPI(qp).get_app())
    r = client.post("/search?namespace=ns", json={"query": q.tolist(), "top_k": 10, "group_by": "doc"})
    assert r.status_code == 200 and [h["id"] for h in r.json()] == [str(v) for v, _ in want[:10]]
    assert client.post("/search?namespace=ns", json={"query": q.tolist(), "top_k": 5, "group_by": "tags"}).status_code == 400
    r = client.post("/query/knn", json={"vector": q.tolist(), "k": 3, "namespace": "ns", "group_by": "doc"})
    assert r.status_code == 200 and r.json()["count"] == 3


def test_scale_1m_cosine_1000_groups_against_the_oracle():
    n, dim, seed = 1_000_000, 768, 5
    from mlvectordb_b200 import DeviceShard
    s = DeviceShard(dim, "cosine", capacity=n)
    s.add_synthetic(seed, 0, n, scaled=True)
    groups = np.random.default_rng(19).integers(0, 1000, n).astype(np.int32)
    s.set_column(0, groups)
    Q = synthetic.queries(seed + 1, 3, dim)
    X = exact.normalize_rows(synthetic.rows(seed, 0, n, dim, scaled=True))
    Qn = exact.normalize_rows(Q)
    for k in (10, 32):
        d, r, g, c = s.search_grouped(Q, k, 0)
        for i in range(3):
            od = exact.distances(X, Qn[i], "cosine")
            er, ed, eg = grouped_topk(od, groups, k)
            best_of = lambda grp, od=od: float(od[groups == grp].min())   # noqa: E731
            msg = exact.check_topk_parity(g[i, : c[i]], d[i, : c[i]], eg, ed, all_ref_scores=best_of)
            assert msg is None, msg
            assert np.array_equal(groups[r[i, : c[i]]], g[i, : c[i]])
            assert exact.scores_close(od[r[i, : c[i]]], d[i, : c[i]]).all()
    s.close()


def test_headline_10m_groups_of_16_and_paths_not_taken():
    n, dim, seed = 10_000_000, 768, 42
    from mlvectordb_b200 import DeviceShard
    s = DeviceShard(dim, "cosine", capacity=n)
    s.add_synthetic(seed, 0, n, scaled=True)
    groups = (np.arange(n, dtype=np.int64) >> 4).astype(np.int32)
    s.set_column(0, groups)
    Q = np.random.default_rng(seed + 1).standard_normal((13, dim), dtype=np.float32)
    d, r, c = s.search(Q[:4], 1024)                      # plain, deduplicated by group on the host
    before = s.gemm_stats()
    gd, gr, gg, gc = s.search_grouped(Q[:4], 10, 0)
    for i in range(4):
        ed, er, eg = _walk(d[i, : c[i]], r[i, : c[i]], groups, 10)
        assert len(er) >= 10                             # the 1024 rows hold enough groups: the check is decisive
        assert np.array_equal(gr[i], er) and np.array_equal(gd[i].view(np.uint32), ed.view(np.uint32))
        assert np.array_equal(gg[i], eg) and gc[i] == 10
    # a grouped batch never takes the tensor-core path or a shadow scan, and each pass is one timed launch
    s.search_grouped(Q[:8], 10, 0)
    s.scan_time_ms()
    s.set_timing(True)
    s.search_grouped(Q, 32, 0)
    ms, launches = s.scan_time_ms()
    s.set_timing(False)
    assert launches == math.ceil(13 / 8) and ms > 0
    after = s.gemm_stats()
    for key in ("searches", "queries", "half_scan_queries", "q8_scan_queries", "half_queries"):
        assert after[key] == before[key], key
    s.close()
