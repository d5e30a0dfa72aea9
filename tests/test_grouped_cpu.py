"""CPU: grouped search (``mlv_index_search_grouped``) -- the oracle's restatement of the contract on hand-made cases,
the argument checks that need no device, and the REST mapping of ``group_by`` (a recording processor stands in)."""
import uuid

import numpy as np
import pytest

from _grouped_oracle import grouped_topk
from oracle import exact

MISSING = exact.COLUMN_MISSING


def _walk(d, g, k, allow=None):
    rows, dists, groups = grouped_topk(np.asarray(d, np.float32), np.asarray(g, np.int32), k, allow)
    return rows.tolist(), dists.tolist(), groups.tolist()


def test_oracle_best_member_per_group_ascending():
    d = [5.0, 1.0, 3.0, 2.0, 4.0, 0.5]
    g = [1, 1, 2, 2, 3, 3]
    assert _walk(d, g, 3) == ([5, 1, 3], [0.5, 1.0, 2.0], [3, 1, 2])
    assert _walk(d, g, 2) == ([5, 1], [0.5, 1.0], [3, 1])


def test_oracle_ties_inside_a_group_go_to_the_lower_row():
    d = [2.0, 1.0, 1.0, 1.0]
    g = [9, 9, 9, 4]
    rows, dists, groups = _walk(d, g, 5)
    assert rows == [1, 3] and groups == [9, 4] and dists == [1.0, 1.0]


def test_oracle_ties_across_groups_order_by_row():
    d = [1.0, 1.0, 1.0, 0.0]
    g = [3, 2, 1, 3]
    # row 3 is group 3's best; then rows 1 and 2 (tied at 1.0) in row order
    assert _walk(d, g, 3) == ([3, 1, 2], [0.0, 1.0, 1.0], [3, 2, 1])
    assert _walk(d, g, 2) == ([3, 1], [0.0, 1.0], [3, 2])


def test_oracle_missing_values_are_no_group():
    d = [0.0, 1.0, 2.0, 3.0]
    g = [MISSING, 5, MISSING, 6]
    assert _walk(d, g, 4) == ([1, 3], [1.0, 3.0], [5, 6])
    assert _walk([0.0], [MISSING], 3) == ([], [], [])


def test_oracle_fewer_groups_than_k():
    rng = np.random.default_rng(1)
    d = rng.standard_normal(200).astype(np.float32)
    g = (np.arange(200) % 3).astype(np.int32)
    rows, dists, groups = _walk(d, g, 10)
    assert len(rows) == 3 and sorted(groups) == [0, 1, 2]
    for r, grp in zip(rows, groups):
        members = np.flatnonzero(g == grp)
        assert r == members[np.argmin(d[members])]


def test_oracle_allow_mask_applies_before_grouping():
    d = [0.0, 1.0, 2.0]
    g = [1, 1, 2]
    assert _walk(d, g, 2, np.array([False, True, True])) == ([1, 2], [1.0, 2.0], [1, 2])


def test_oracle_every_row_its_own_group_is_the_plain_topk():
    rng = np.random.default_rng(7)
    X = rng.standard_normal((500, 16)).astype(np.float32)
    q = rng.standard_normal(16).astype(np.float32)
    X[10] = X[11]                                   # an exact tie: ordered by row
    d = exact.distances(X, q, "l2")
    for k in (1, 7, 32):
        L, D = exact.knn(X, q[None, :], k, "l2")
        rows, dists, groups = grouped_topk(d, np.arange(500, dtype=np.int32), k)
        assert rows.tolist() == L[0].tolist() and np.array_equal(dists, D[0]) and groups.tolist() == rows.tolist()


def test_group_by_rejects_k_above_32_before_any_device_work():
    from mlvectordb_b200 import _capi
    from mlvectordb_b200.index import GpuIndex
    from mlvectordb_b200.interfaces import VectorDTO
    assert _capi.MAX_GROUP_K == 32
    idx = GpuIndex.__new__(GpuIndex)                 # no namespace, no device: the check comes first
    with pytest.raises(ValueError):
        idx.search(VectorDTO(values=[0.0, 1.0], metadata={}), 33, "nowhere", "l2", group_by="doc")
    with pytest.raises(ValueError):
        idx.search_batch(np.zeros((2, 2), np.float32), 33, "nowhere", group_by="doc")


def test_capi_declares_the_grouped_entries():
    from mlvectordb_b200 import _capi
    assert "mlv_index_search_grouped" in _capi.SIGNATURES
    assert "mlv_index_search_grouped_device" in _capi.SIGNATURES
    assert len(_capi.SIGNATURES["mlv_index_search_grouped"][1]) == 10
    assert len(_capi.SIGNATURES["mlv_index_search_grouped_device"][1]) == 11


# ---- REST ---------------------------------------------------------------------------------------------------------
fastapi = pytest.importorskip("fastapi")
from fastapi.testclient import TestClient  # noqa: E402

from mlvectordb_b200.index import NotDeviceEvaluable  # noqa: E402
from mlvectordb_b200.rest_api import GpuRestAPI  # noqa: E402


class _GroupingRecorder:
    """Records what reaches the processor; a ``group_by`` of "host_only" behaves like a key kept on the host."""

    def __init__(self):
        self.calls = []
        self.ids = [uuid.uuid4() for _ in range(3)]

    def _hits(self, n):
        return [{"id": self.ids[i], "score": 0.1 * i} for i in range(n)]

    def _check(self, extra):
        if extra.get("group_by") == "host_only":
            raise NotDeviceEvaluable("metadata key 'host_only' is not held as a device column")

    def find_similar(self, query, top_k, namespace="default", metric="cosine", **extra):
        self.calls.append(("find_similar", top_k, extra))
        self._check(extra)
        return self._hits(min(top_k, 3))

    def find_similar_batch(self, queries, top_k, namespace="default", metric="cosine", **extra):
        self.calls.append(("find_similar_batch", top_k, extra))
        self._check(extra)
        return [self._hits(2) for _ in queries]

    def find_in_range(self, query, radius, namespace="default", metric="cosine", **extra):
        self.calls.append(("find_in_range", radius, extra))
        return self._hits(2)


@pytest.fixture()
def rest():
    rec = _GroupingRecorder()
    return rec, TestClient(GpuRestAPI(rec).get_app())


def test_rest_group_by_reaches_the_processor(rest):
    rec, client = rest
    r = client.post("/search", json={"query": [1, 0], "top_k": 5, "group_by": "doc", "include_values": False})
    assert r.status_code == 200 and len(r.json()) == 3
    assert rec.calls[-1] == ("find_similar", 5, {"enrich": False, "group_by": "doc"})
    r = client.post("/search/batch", json={"queries": [[1, 0], [0, 1]], "top_k": 4, "group_by": "doc"})
    assert r.status_code == 200 and len(r.json()) == 2
    assert rec.calls[-1][0] == "find_similar_batch" and rec.calls[-1][2]["group_by"] == "doc"
    r = client.post("/query/knn", json={"vector": [1, 0], "k": 32, "group_by": "page"})
    assert r.status_code == 200 and r.json()["count"] == 3
    assert rec.calls[-1][2]["group_by"] == "page"
    r = client.post("/query/hybrid", json={"vector": [1, 0], "k": 3, "filter": {"lang": "en"}, "group_by": "doc"})
    assert r.status_code == 200
    assert rec.calls[-1][2]["group_by"] == "doc" and rec.calls[-1][2]["filter"] == {"lang": "en"}


def test_rest_without_group_by_passes_nothing_new(rest):
    rec, client = rest
    assert client.post("/search", json={"query": [1, 0], "top_k": 50}).status_code == 200
    assert "group_by" not in rec.calls[-1][2]
    assert client.post("/search/batch", json={"queries": [[1, 0]], "top_k": 50}).status_code == 200
    assert "group_by" not in rec.calls[-1][2]


@pytest.mark.parametrize("route,body", [
    ("/search", {"query": [1, 0], "top_k": 5, "radius": 0.5, "group_by": "doc"}),
    ("/search", {"query": [1, 0], "top_k": 33, "group_by": "doc"}),
    ("/search", {"query": [1, 0], "top_k": 5, "group_by": "host_only"}),
    ("/search/batch", {"queries": [[1, 0]], "top_k": 100, "group_by": "doc"}),
    ("/search/batch", {"queries": [[1, 0]], "top_k": 5, "group_by": "host_only"}),
    ("/query/knn", {"vector": [1, 0], "k": 33, "group_by": "doc"}),
    ("/query/knn", {"vector": [1, 0], "k": 3, "group_by": "host_only"}),
    ("/query/hybrid", {"vector": [1, 0], "k": 3, "filter": {"a": 1}, "group_by": "host_only"}),
    ("/query/range", {"vector": [1, 0], "radius": 0.3, "group_by": "doc"}),
    ("/query/similarity", {"vector": [1, 0], "threshold": 0.7, "group_by": "doc"}),
])
def test_rest_group_by_client_errors_are_400(rest, route, body):
    rec, client = rest
    r = client.post(route, json=body)
    assert r.status_code == 400, r.text
    assert "group_by" in r.json()["detail"] or "host" in r.json()["detail"]
    assert all(c[0] != "find_in_range" for c in rec.calls)
