"""``GpuIndex``: drop-in for the reference ``Index`` backed by the B200 exact-search library.

Mirrors reference ``src/mlvectordb/implementations/index.py:17-165`` method for method
(constructor signature, ``add`` / ``remove`` / ``search`` / ``rebuild`` /
``is_rebuild_required``, attribute ``_space``), so ``QueryProcessor(storage, GpuIndex(...))``
(reference ``api/server.py:54``, ``query_processor.py:19,24,33,56-61``) works unchanged.  What
differs underneath: every namespace is one contiguous device-resident fp32 row matrix scanned
exactly by hand-written sm_100a kernels (``csrc/scan_kernel.cuh``) instead of an hnswlib graph.

Behaviour kept from the reference (SURVEY.md section 3, Q1-Q10):
  * the space is fixed at construction; ``search(metric=...)`` only toggles ``score = 1 - d`` when
    ``metric == "cosine"`` (``index.py:23,55,126-127``);
  * scores are hnswlib-form distances: squared L2, ``1 - dot``, cosine similarity after the toggle;
  * ``top_k`` is clamped to the live count; unknown namespace / nothing live / wrong dimension
    -> ``[]`` (``index.py:98-119``); ``remove`` of unknown ids is a no-op (``:70-84``);
  * ``rebuild(source, metric)`` replaces every namespace by ``source`` (``:136-162``).
Deliberate differences:
  * no 10 000-row cap (``index.py:37``); results are exact, ties ordered by row;
  * with ``auto_compact=True`` (default) a namespace whose deleted ratio reaches
    ``rebuild_threshold`` is compacted on the device and ``is_rebuild_required`` stays False, so
    ``QueryProcessor.delete`` never takes the reference's rebuild path that wipes the *other*
    namespaces (Q6).  ``auto_compact=False`` restores the reference's flag behaviour.
Additive (no reference code; README-only intent): ``search_batch``, ``filter=``, ``group_by=``,
``range_search``, ``dimension``, ``add_matrix``, ``info``.
"""
from __future__ import annotations

import os
from typing import Callable, Dict, Iterable, List, Mapping, Optional, Sequence, Union
from uuid import UUID

import numpy as np

from . import _capi
from .columns import ColumnCodec
from .interfaces import SearchResult, VectorDTO, VectorProtocol
from .shard import DeviceShard, PreparedFilter, canonical_space

# row mask / packed bitmap, callable(uuid) -> bool, prepared filter, or a mapping of metadata constraints
# ({key: value} equality, {key: (op, a)} / {key: ("between", a, b)}) evaluated on the device columns
FilterArg = Union[None, np.ndarray, Callable[[UUID], bool], PreparedFilter, Mapping]


class NotDeviceEvaluable(ValueError):
    """A metadata constraint the device columns cannot decide (see ``columns.py``); evaluate it on the host
    and pass a row mask / ``callable(uuid)`` instead (``GpuQueryProcessor`` does)."""


from uuid import SafeUUID as _SafeUUID   # noqa: E402

_uuid_new, _uuid_set, _int_from_bytes, _UNKNOWN = object.__new__, object.__setattr__, int.from_bytes, _SafeUUID.unknown


def uuid_from_bytes(raw: bytes) -> UUID:
    """``UUID(bytes=raw)`` without the constructor's argument checks (1.7 us -> 0.4 us): a search builds one UUID per
    hit, which at k = 10 is half of ``GpuIndex.search``'s host time on a small namespace.  ``raw`` is always 16 bytes
    taken from the id table, which only holds bytes of valid UUIDs."""
    u = _uuid_new(UUID)
    _uuid_set(u, "int", _int_from_bytes(raw, "big"))
    _uuid_set(u, "is_safe", _UNKNOWN)
    return u


def _random_uuid_bytes(n: int) -> np.ndarray:
    ids = np.frombuffer(os.urandom(16 * n), dtype=np.uint8).reshape(n, 16).copy()
    ids[:, 6] = (ids[:, 6] & 0x0F) | 0x40  # version 4
    ids[:, 8] = (ids[:, 8] & 0x3F) | 0x80  # RFC 4122 variant
    return ids


class _Namespace:
    """Per-namespace state: reference ``index.py:19-30`` (index, dim, id maps, counters)."""

    def __init__(self, dim: int, space: str, device: int, capacity: int):
        self.dim = dim
        self.space = space
        self.shard = DeviceShard(dim, space, capacity=capacity, device=device)
        self.ids = np.empty((max(capacity, 16), 16), dtype=np.uint8)  # row -> uuid bytes (label_to_uuid)
        self.n = 0                                                    # rows stored incl. tombstoned
        self.gone = np.zeros(max(capacity, 16), dtype=bool)           # host mirror of the tombstones
        self.uuid_to_row: Optional[Dict[bytes, int]] = {}             # None = not built (bulk loaded)
        self.total = 0
        self.deleted = 0
        self.rebuild_required = False
        self.codec = ColumnCodec()                                    # metadata key -> device column
        self.version = 0                                              # bumped by every mutation
        self.where_cache: Dict[tuple, PreparedFilter] = {}            # constraints -> filter, valid for `version`

    def touch(self) -> None:
        self.version += 1
        for f in self.where_cache.values():
            f.close()
        self.where_cache.clear()

    def reserve(self, extra: int) -> None:
        need = self.n + extra
        if need > self.ids.shape[0]:
            cap = max(need, self.ids.shape[0] * 2)
            ids = np.empty((cap, 16), dtype=np.uint8)
            ids[: self.n] = self.ids[: self.n]
            self.ids = ids
            gone = np.zeros(cap, dtype=bool)
            gone[: self.n] = self.gone[: self.n]
            self.gone = gone

    def lookup(self) -> Dict[bytes, int]:
        if self.uuid_to_row is None:
            live = np.flatnonzero(~self.gone[: self.n])
            raw = self.ids[: self.n].tobytes()
            self.uuid_to_row = {raw[16 * r: 16 * r + 16]: int(r) for r in live.tolist()}
        return self.uuid_to_row

    def uuid_of(self, row: int) -> UUID:
        return uuid_from_bytes(self.ids[row].tobytes())


class PendingResults:
    """``GpuIndex.search_async`` in flight."""

    def __init__(self, pending, ns, metric: str):
        self._pending, self._ns, self._metric = pending, ns, metric

    def result(self) -> List[SearchResult]:
        if self._pending is None:
            return []
        dists, rows, counts = self._pending.result()
        out = []
        for row, dist in zip(rows[0, : counts[0]].tolist(), dists[0, : counts[0]].tolist()):
            score = float(dist)
            if self._metric == "cosine":
                score = 1 - score
            out.append(SearchResult(vector_id=self._ns.uuid_of(row), score=score))
        return out


class GpuIndex:
    def __init__(self, space: str = "l2", ef_construction: int = 200, M: int = 16, rebuild_threshold: float = 0.2,
                 device: int = 0, capacity: int = 0, auto_compact: bool = True):
        # ef_construction / M are accepted for signature compatibility (reference index.py:18);
        # an exact scan has no graph parameters.
        canonical_space(space)            # validate early (hnswlib raises at first add instead)
        self._space = space
        self._ef_construction = ef_construction
        self._M = M
        self._rebuild_threshold = float(rebuild_threshold)
        self._device = int(device)
        self._capacity_hint = int(capacity)
        self._auto_compact = bool(auto_compact)
        self._ns: Dict[str, _Namespace] = {}
        _capi.lib()                       # fail loudly now if the CUDA library is missing

    # ------------------------------------------------------------------ internals
    def _get_or_create(self, namespace: str, dim: int, metric: str, capacity: int = 0) -> _Namespace:
        ns = self._ns.get(namespace)
        if ns is None:
            ns = _Namespace(dim, canonical_space(metric), self._device, capacity or self._capacity_hint)
            self._ns[namespace] = ns
        return ns

    def _append(self, ns: _Namespace, data: np.ndarray, ids: np.ndarray) -> np.ndarray:
        n = data.shape[0]
        first = ns.shard.add(data)
        assert first == ns.n, "host id map out of step with the device matrix"
        ns.reserve(n)
        ns.ids[first:first + n] = ids
        ns.gone[first:first + n] = False
        ns.n += n
        ns.total += n
        ns.touch()
        return np.arange(first, first + n, dtype=np.int64)

    @staticmethod
    def _ingest_metadata(ns: _Namespace, first_row: int, vectors) -> None:
        """Metadata mappings of freshly appended rows -> device columns (``columns.py``)."""
        mds = [getattr(v, "metadata", None) for v in vectors]
        if not any(mds):
            return
        for column, codes in ns.codec.encode_rows(mds).items():
            ns.shard.set_column(column, codes, first_row)

    def _maybe_compact(self, ns: _Namespace) -> None:
        ratio = ns.deleted / max(1, ns.total)
        if ratio < self._rebuild_threshold:
            return
        if not self._auto_compact:
            ns.rebuild_required = True
            return
        self._compact(ns)

    def _compact(self, ns: _Namespace) -> None:
        mapping = ns.shard.compact()
        keep = mapping >= 0
        live = int(keep.sum())
        ns.ids[:live] = ns.ids[: ns.n][keep]
        ns.gone[: ns.n] = False
        ns.n = live
        ns.total = live
        ns.deleted = 0
        ns.rebuild_required = False
        ns.uuid_to_row = None
        ns.touch()

    def _filter_mask(self, ns: _Namespace, filt: FilterArg):
        if filt is None:
            return None
        if isinstance(filt, PreparedFilter):
            return filt
        if isinstance(filt, Mapping):
            return self._where(ns, filt)
        if callable(filt):
            return np.fromiter((bool(filt(ns.uuid_of(r))) for r in range(ns.n)), dtype=bool, count=ns.n)
        return filt

    @staticmethod
    def _order_columns(ns, constraints: Mapping) -> None:
        """An ordered constraint on a dictionary-coded key needs codes that ascend with the values: re-code the column
        by rank (one read + one write of 4 bytes per row; again only after new values broke the order)."""
        from . import _capi
        try:
            names = ns.codec.unordered_columns(constraints)
        except TypeError:
            return
        for name in names:
            perm = ns.codec.reorder(name)
            if perm is None or ns.n == 0:
                continue
            column = ns.codec.column_index(name)
            codes = ns.shard.get_column(column, 0, ns.n)
            has = codes != _capi.COLUMN_MISSING
            codes[has] = perm[codes[has]]
            ns.shard.set_column(column, codes, 0)

    def _where(self, ns: _Namespace, constraints: Mapping) -> PreparedFilter:
        try:
            key = tuple(sorted(constraints.items(), key=lambda kv: kv[0]))
            cached = ns.where_cache.get(key)
        except TypeError:
            key, cached = None, None
        if cached is not None:
            return cached
        self._order_columns(ns, constraints)
        preds = ns.codec.predicates(constraints)
        if preds is None:
            raise NotDeviceEvaluable(f"constraints {dict(constraints)!r} cannot be evaluated on the device columns")
        prepared = ns.shard.where(preds)
        if key is not None:
            ns.where_cache[key] = prepared
        return prepared

    @staticmethod
    def _group_column(ns: _Namespace, group_by: str) -> Optional[int]:
        """Device column of metadata key ``group_by``, or None when no row ever had the key (no groups at all).  A key
        kept on the host only cannot be grouped on the device, and there is no host grouping."""
        if ns.codec.kind(group_by) == "host":
            raise NotDeviceEvaluable(f"metadata key {group_by!r} is not held as a device column; it cannot be grouped by")
        return ns.codec.column_index(group_by)

    @staticmethod
    def _check_group_k(top_k: int) -> None:
        if int(top_k) > _capi.MAX_GROUP_K:
            raise ValueError(f"group_by supports top_k <= {_capi.MAX_GROUP_K}, got {top_k}")

    # ------------------------------------------------------------------ IndexProtocol
    def add(self, vectors: Iterable[VectorProtocol], namespace: str) -> None:
        """reference index.py:50-67"""
        vectors = list(vectors)
        if not vectors:
            return
        dim = vectors[0].values.shape[0]
        ns = self._get_or_create(namespace, dim, self._space)
        data = np.array([v.values for v in vectors], dtype=np.float32)
        if data.ndim != 2 or data.shape[1] != ns.dim:
            raise RuntimeError("Wrong dimensionality of the vectors")  # hnswlib's add_items error
        ids = np.frombuffer(b"".join(v.id.bytes for v in vectors), dtype=np.uint8).reshape(-1, 16)
        rows = self._append(ns, data, ids)
        self._ingest_metadata(ns, int(rows[0]), vectors)
        if ns.uuid_to_row is not None:
            for v, r in zip(vectors, rows.tolist()):
                ns.uuid_to_row[v.id.bytes] = r

    def remove(self, ids: Sequence[UUID], namespace: str) -> None:
        """reference index.py:69-89"""
        ns = self._ns.get(namespace)
        if ns is None:
            return
        lookup = ns.lookup()
        rows = []
        for uid in ids:
            r = lookup.pop(uid.bytes, None)
            if r is not None:
                rows.append(r)
        if rows:
            changed = ns.shard.mark_deleted(np.asarray(rows, dtype=np.uint64))
            assert changed == len(rows), "device tombstones out of step with the host id map"
            ns.gone[rows] = True
            ns.touch()
        ns.deleted += len(rows)
        self._maybe_compact(ns)

    def search(self, query: VectorDTO, top_k: int, namespace: str, metric: str,
               filter: FilterArg = None, group_by: Optional[str] = None) -> List[SearchResult]:
        """reference index.py:91-129 (``filter`` and ``group_by`` are additive).

        ``group_by``: a metadata key; the result is then the ``top_k`` (<= 32) nearest *groups* -- rows with equal
        values of the key (Python equality) -- each reported by its nearest row, nearest group first.  Rows without the
        key belong to no group (``mlv_index_search_grouped``)."""
        if group_by is not None:
            self._check_group_k(top_k)
        ns = self._ns.get(namespace)
        if ns is None:
            return []
        active = ns.total - ns.deleted
        if active == 0:
            return []
        top_k = min(int(top_k), active)
        if top_k < 1:
            return []
        q = np.asarray(query.values, dtype=np.float32).reshape(-1)
        if q.shape[0] != ns.dim:
            return []  # the reference swallows hnswlib's dimension RuntimeError into [] (index.py:110-119)
        if group_by is None:
            dists, rows, counts = ns.shard.search(q[None, :], top_k, self._filter_mask(ns, filter))
        else:
            column = self._group_column(ns, group_by)
            if column is None:
                return []
            dists, rows, _, counts = ns.shard.search_grouped(q[None, :], top_k, column, self._filter_mask(ns, filter))
        c = int(counts[0])
        raw = ns.ids[rows[0, :c]].tobytes()          # the hits' uuid bytes in one gather (label -> UUID, reference index.py:123)
        scores = dists[0, :c].tolist()
        if metric == "cosine":
            return [SearchResult(vector_id=uuid_from_bytes(raw[16 * i: 16 * i + 16]), score=1 - scores[i]) for i in range(c)]
        return [SearchResult(vector_id=uuid_from_bytes(raw[16 * i: 16 * i + 16]), score=scores[i]) for i in range(c)]

    def search_async(self, query: VectorDTO, top_k: int, namespace: str, metric: str,
                     filter: FilterArg = None) -> "PendingResults":
        """``search`` that returns at once; ``.result()`` gives the ``List[SearchResult]``.  A server that keeps
        two requests in flight overlaps one request's copies / launch latency with the other's scan.
        ``filter``: metadata constraints or a prepared filter (row masks / callables: prepare them first with
        ``prepare_filter`` -- the submit must not wait for a host-side evaluation); it stays bound to this search only."""
        ns = self._ns.get(namespace)
        active = (ns.total - ns.deleted) if ns is not None else 0
        k = min(int(top_k), active)
        q = np.asarray(query.values, dtype=np.float32).reshape(-1)
        if ns is None or k < 1 or q.shape[0] != ns.dim:
            return PendingResults(None, None, metric)
        prepared = self._filter_mask(ns, filter)
        if prepared is not None and not isinstance(prepared, PreparedFilter):
            prepared = ns.shard.prepare_filter(prepared)
            ns.where_cache[("async", id(prepared))] = prepared   # kept alive until the namespace changes
        from .shard import _bound
        with _bound(ns.shard, prepared):      # the launch captures the filter's row list; the binding ends with the submit
            pending = ns.shard.submit(q[None, :], k)
        return PendingResults(pending, ns, metric)

    def rebuild(self, source: Mapping[str, Iterable[VectorProtocol]], metric: str) -> None:
        """reference index.py:131-162: drop everything, re-add ``source`` with ``space=metric``."""
        for ns in self._ns.values():
            ns.touch()
            ns.shard.close()
        self._ns.clear()
        for namespace, vectors in source.items():
            vectors = list(vectors)
            if not vectors:
                continue
            dim = vectors[0].values.shape[0]
            ns = self._get_or_create(namespace, dim, metric, capacity=len(vectors))
            data = np.array([v.values for v in vectors], dtype=np.float32)
            ids = np.frombuffer(b"".join(v.id.bytes for v in vectors), dtype=np.uint8).reshape(-1, 16)
            rows = self._append(ns, data, ids)
            self._ingest_metadata(ns, 0, vectors)
            ns.uuid_to_row = {v.id.bytes: r for v, r in zip(vectors, rows.tolist())}
            ns.total = len(vectors)
            ns.deleted = 0
            ns.rebuild_required = False

    def is_rebuild_required(self, namespace: str) -> bool:
        """reference index.py:164-165"""
        ns = self._ns.get(namespace)
        return bool(ns.rebuild_required) if ns is not None else False

    # ------------------------------------------------------------------ additive surface
    def dimension(self, namespace: str) -> Optional[int]:
        ns = self._ns.get(namespace)
        return ns.dim if ns is not None else None

    def add_matrix(self, matrix: np.ndarray, namespace: str, ids: Optional[Sequence[UUID]] = None,
                   columns: Optional[Mapping[str, Sequence]] = None,
                   metadata: Optional[Sequence[Optional[Mapping]]] = None) -> np.ndarray:
        """Bulk ingest without per-row ``Vector`` objects (SURVEY.md H4).  Returns the rows' UUID bytes [n, 16].
        ``columns``: metadata as whole columns ``{key: values[n]}`` (integer arrays are stored as they are, other
        values dictionary coded) for ``filter={key: ...}`` searches evaluated on the device; ``metadata``: the same
        as one mapping per row (what ``add`` reads from ``v.metadata``)."""
        data = np.ascontiguousarray(matrix, dtype=np.float32)
        if data.ndim != 2:
            raise ValueError("matrix must be [n, dim]")
        if data.shape[0] == 0:
            return np.empty((0, 16), dtype=np.uint8)
        ns = self._get_or_create(namespace, data.shape[1], self._space, capacity=data.shape[0])
        if data.shape[1] != ns.dim:
            raise RuntimeError("Wrong dimensionality of the vectors")
        if ids is None:
            id_bytes = _random_uuid_bytes(data.shape[0])
        else:
            id_bytes = np.frombuffer(b"".join(u.bytes for u in ids), dtype=np.uint8).reshape(-1, 16)
            if id_bytes.shape[0] != data.shape[0]:
                raise ValueError("len(ids) != rows")
        if columns:
            for name, values in columns.items():
                if len(values) != data.shape[0]:
                    raise ValueError(f"column {name!r} has {len(values)} values for {data.shape[0]} rows")
        rows = self._append(ns, data, id_bytes)
        for name, values in (columns or {}).items():
            self.set_column(namespace, name, values, first_row=int(rows[0]))
        if metadata is not None:
            if len(metadata) != data.shape[0]:
                raise ValueError("len(metadata) != rows")
            for column, codes in ns.codec.encode_rows(metadata).items():
                ns.shard.set_column(column, codes, int(rows[0]))
        if data.shape[0] > 100_000:
            ns.uuid_to_row = None          # rebuilt lazily from ns.ids by the first remove()
        elif ns.uuid_to_row is not None:
            raw = id_bytes.tobytes()
            for i, r in enumerate(rows.tolist()):
                ns.uuid_to_row[raw[16 * i: 16 * i + 16]] = r
        return id_bytes

    def add_synthetic(self, namespace: str, n: int, dim: int, seed: int, scaled: bool = False,
                      first_gen_row: int = 0) -> None:
        """Benchmark / parity input: rows generated on the device (``mlv_index_add_synthetic``)."""
        ns = self._get_or_create(namespace, dim, self._space, capacity=n)
        if dim != ns.dim:
            raise RuntimeError("Wrong dimensionality of the vectors")
        first = ns.shard.add_synthetic(seed, first_gen_row, n, scaled)
        assert first == ns.n
        ns.reserve(n)
        ns.ids[first:first + n] = _random_uuid_bytes(n)
        ns.gone[first:first + n] = False
        ns.n += n
        ns.total += n
        ns.uuid_to_row = None
        ns.touch()

    def search_batch(self, queries: np.ndarray, top_k: int, namespace: str, metric: Optional[str] = None,
                     filter: FilterArg = None, group_by: Optional[str] = None):
        """Batched search -> (rows i64 [nq,k] (-1 padded), scores f32 [nq,k], counts i32 [nq]).

        Scores follow ``search``: hnswlib-form distances, ``1 - d`` when ``metric == "cosine"``.  ``group_by`` as in
        ``search``: row i of the result holds query i's nearest groups, one row each.
        """
        if group_by is not None:
            self._check_group_k(top_k)
        q = np.ascontiguousarray(queries, dtype=np.float32)
        if q.ndim == 1:
            q = q[None, :]
        nq = q.shape[0]
        ns = self._ns.get(namespace)
        active = (ns.total - ns.deleted) if ns is not None else 0
        k = min(int(top_k), active)
        if ns is None or k < 1 or q.shape[1] != ns.dim:
            return (np.full((nq, 0), -1, np.int64), np.empty((nq, 0), np.float32), np.zeros(nq, np.int32))
        if group_by is None:
            dists, rows, counts = ns.shard.search(q, k, self._filter_mask(ns, filter))
        else:
            column = self._group_column(ns, group_by)
            if column is None:
                return (np.full((nq, 0), -1, np.int64), np.empty((nq, 0), np.float32), np.zeros(nq, np.int32))
            dists, rows, _, counts = ns.shard.search_grouped(q, k, column, self._filter_mask(ns, filter))
        if (metric if metric is not None else self._space) == "cosine":
            dists = (1.0 - dists.astype(np.float64)).astype(np.float32)
        return rows, dists, counts

    def uuids_of(self, namespace: str, rows: np.ndarray) -> List[Optional[UUID]]:
        ns = self._ns[namespace]
        return [ns.uuid_of(int(r)) if r >= 0 else None for r in np.asarray(rows).reshape(-1)]

    def range_search(self, query: VectorDTO, radius: float, namespace: str, metric: str,
                     filter: FilterArg = None) -> List[SearchResult]:
        """Every live row with hnswlib-form distance <= radius, ascending; same score toggle as ``search``.

        For ``metric == "cosine"`` on a cosine index that is cosine similarity >= 1 - radius (the
        stale client's ``threshold`` query, reference ``examples/api_client.py:50-63``).
        """
        ns = self._ns.get(namespace)
        if ns is None or ns.total - ns.deleted == 0:
            return []
        q = np.asarray(query.values, dtype=np.float32).reshape(-1)
        if q.shape[0] != ns.dim:
            return []
        (dists, rows), = ns.shard.range_search(q[None, :], float(radius), self._filter_mask(ns, filter))
        out = []
        for row, dist in zip(rows.tolist(), dists.tolist()):
            score = float(dist)
            if metric == "cosine":
                score = 1 - score
            out.append(SearchResult(vector_id=ns.uuid_of(row), score=score))
        return out

    def set_column(self, namespace: str, name: str, values, first_row: int = 0) -> bool:
        """Write metadata key ``name`` for rows ``first_row ..`` as one column.  False when the key cannot live on
        the device (``columns.py``: more than 16 keys, unhashable values) -- constraints on it then raise
        ``NotDeviceEvaluable``."""
        ns = self._ns[namespace]
        if first_row < 0 or first_row + len(values) > ns.n:
            raise ValueError("column values beyond the stored rows")
        enc = ns.codec.encode_column(name, values)
        ns.touch()
        if enc is None:
            return False
        ns.shard.set_column(enc[0], enc[1], first_row)
        return True

    def where(self, namespace: str, constraints: Mapping) -> Optional[PreparedFilter]:
        """Prepared filter for metadata constraints evaluated on the device columns, or None when they cannot be
        (then evaluate on the host and use ``prepare_filter``).  Cached until the namespace changes."""
        ns = self._ns.get(namespace)
        if ns is None:
            return None
        try:
            return self._where(ns, constraints)
        except NotDeviceEvaluable:
            return None

    def metadata_columns(self, namespace: str) -> List[str]:
        ns = self._ns.get(namespace)
        return ns.codec.names() if ns is not None else []

    def prepare_filter(self, namespace: str, filter: FilterArg) -> PreparedFilter:
        """Evaluate a filter (row mask or ``callable(uuid) -> bool``) once and keep it on the device;
        pass the result as ``filter=`` to ``search`` / ``search_batch`` / ``range_search``.  It follows later
        adds / removes of the namespace (rows added afterwards do not pass); compaction renumbers rows, so
        prepare it again after the namespace was compacted."""
        ns = self._ns[namespace]
        resolved = self._filter_mask(ns, filter)
        if isinstance(resolved, PreparedFilter):      # already prepared (or metadata constraints decided on the device)
            return resolved
        return ns.shard.prepare_filter(resolved)

    def info(self, namespace: str) -> dict:
        ns = self._ns[namespace]
        inf = ns.shard.info()
        return {"rows": int(inf.rows), "live": int(inf.live), "capacity": int(inf.capacity), "dim": int(inf.dim),
                "device": int(inf.device), "device_bytes": int(inf.device_bytes), "space": ns.space,
                "tombstones": int(inf.rows - inf.live)}

    def namespaces(self) -> List[str]:
        return list(self._ns)

    def save(self, path: str) -> dict:
        """Snapshot every namespace under directory ``path`` (``snapshot.py``)."""
        from .snapshot import save_index
        return save_index(self, path)

    @classmethod
    def load(cls, path: str, device: int = 0) -> "GpuIndex":
        """Index restored from ``save``'s directory; searches return what they returned before the save."""
        from .snapshot import load_index
        return load_index(path, device=device, index_cls=cls)

    def close(self) -> None:
        for ns in self._ns.values():
            ns.touch()
            ns.shard.close()
        self._ns.clear()
