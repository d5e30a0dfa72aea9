"""``GpuQueryProcessor``: the caller of the index (SURVEY.md section 8f, ranks 1-3).

Mirrors the reference ``QueryProcessor`` (``src/mlvectordb/implementations/query_processor.py:11-82``)
method for method -- ``insert``, ``upsert_many``, ``find_similar``, ``delete``, ``list_namespaces``,
``get_namespace_vectors``, ``get_namespace_count``, ``get_storage_info`` keep their names, arguments
and results, so ``RestAPI(GpuQueryProcessor(storage, GpuIndex(...)))`` works where the reference
builds ``RestAPI(QueryProcessor(...))`` (``api/server.py:54-57``) -- and adds the entry points the
reference only sketches, so the GPU index's abilities are reachable from the product surface:

* ``find_similar(..., filter=...)``        metadata-filtered search (``README.md:123,477``; request shape
                                           ``examples/api_client.py:65-74``: a dict of equality constraints)
* ``find_similar_batch(queries, ...)``     many queries in one call (tensor-core path from 5 queries on a >= 1 GB matrix)
* ``find_in_range(query, radius, ...)``    radius query (``README.md:121,215``; ``examples/api_client.py:38-48``)
* ``upsert_matrix(matrix, ...)``           bulk ingest without one ``Vector`` + ``uuid4()`` per row (SURVEY H4)
* ``enrich=False``                         ids + scores only: skips the per-hit storage lookup and the k x d
                                           float payload that dominates a response at GPU speeds (rank 2)

Works with any storage that implements the reference ``StorageEngine`` protocol
(``interfaces/storage_engine.py:16-53``); the storage stays the source of truth for values and metadata.
"""
from __future__ import annotations

from typing import Any, Callable, Dict, Iterable, List, Mapping, Optional, Sequence, Union
from uuid import UUID, uuid4

import numpy as np

from .columns import host_predicate
from .index import GpuIndex, _random_uuid_bytes
from .interfaces import VectorDTO
from .shard import PreparedFilter

MetadataFilter = Union[None, Mapping[str, Any], Callable[[Mapping[str, Any]], bool], PreparedFilter]


class StoredVector:
    """What ``Vector`` is in the reference (``implementations/vector.py:10-42``): ``id`` (uuid4), ``values``
    (an fp32 copy), ``metadata``.  ``upsert_matrix`` builds these with ids minted in bulk."""

    __slots__ = ("id", "values", "metadata")

    def __init__(self, values, metadata: Optional[Mapping[str, Any]] = None, id: Optional[UUID] = None):  # noqa: A002
        self.id = id if id is not None else uuid4()
        self.values = np.array(values, dtype=np.float32)
        self.metadata = metadata or {}

    def __eq__(self, other):
        return isinstance(other, StoredVector) and self.id == other.id

    @classmethod
    def rows_of(cls, matrix: np.ndarray, ids: Sequence[UUID], metadata: Optional[Sequence[Optional[Mapping[str, Any]]]]):
        """One ``StoredVector`` per row of ``matrix`` whose ``values`` are row views of ONE fp32 copy of the matrix
        (the per-row ``np.array`` copy of ``__init__`` is what makes per-object bulk ingest slow, SURVEY H4)."""
        own = np.array(matrix, dtype=np.float32)
        out = []
        for i in range(own.shape[0]):
            v = cls.__new__(cls)
            v.id = ids[i]
            v.values = own[i]
            v.metadata = (metadata[i] if metadata is not None else None) or {}
            out.append(v)
        return out


class GpuQueryProcessor:
    def __init__(self, storage_engine, index: GpuIndex):
        self._storage = storage_engine
        self._index = index
        # prepared filters per (namespace, predicate key), valid while the namespace is unchanged
        self._filters: Dict[tuple, tuple] = {}
        self._mutations: Dict[str, int] = {}

    # ------------------------------------------------------------------ reference surface
    def insert(self, vector: VectorDTO, namespace: str = "default") -> None:
        """reference query_processor.py:16-19"""
        new_vec = StoredVector(vector.values, vector.metadata)
        self._storage.write(new_vec, namespace)
        self._index.add([new_vec], namespace)
        self._touch(namespace)

    def upsert_many(self, vectors: Iterable[VectorDTO], namespace: str = "default") -> None:
        """reference query_processor.py:21-24 (no upsert semantics there either: every call mints new ids)"""
        vectors = list(vectors)
        raw = _random_uuid_bytes(len(vectors)).tobytes()          # ids minted in one go (uuid4 layout)
        vecs = [StoredVector(v.values, v.metadata, id=UUID(bytes=raw[16 * i:16 * i + 16])) for i, v in enumerate(vectors)]
        self._storage.write_vectors(vecs, namespace)
        self._index.add(vecs, namespace)
        self._touch(namespace)

    def find_similar(self, query: VectorDTO, top_k: int, namespace: str = "default", metric: str = "cosine",
                     filter: MetadataFilter = None, enrich: bool = True,  # noqa: A002
                     group_by: Optional[str] = None) -> List[dict]:
        """reference query_processor.py:26-49; ``filter`` / ``enrich`` / ``group_by`` are additive.  ``group_by``: the
        ``top_k`` (<= 32) nearest groups of that metadata key, each as its nearest vector (``GpuIndex.search``)."""
        grouped = {"group_by": group_by} if group_by is not None else {}
        results = self._index.search(query, top_k=top_k, namespace=namespace, metric=metric,
                                     filter=self._resolve_filter(namespace, filter), **grouped)
        if not results:
            return []
        return self._enrich([(r.vector_id, r.score) for r in results], namespace, enrich)

    def delete(self, ids: Sequence[UUID], namespace: str = "default") -> Sequence[UUID]:
        """reference query_processor.py:51-62"""
        deleted = [vid for vid in ids if self._storage.delete(vid, namespace)]
        self._index.remove(ids, namespace)
        if self._index.is_rebuild_required(namespace):   # only with GpuIndex(auto_compact=False)
            source = {namespace: self._storage.namespace_map.get(namespace, [])}
            self._index.rebuild(source, metric=self._index._space)
        self._touch(namespace)
        return deleted

    def list_namespaces(self) -> List[str]:
        return self._storage.list_namespaces

    def get_namespace_vectors(self, namespace: str) -> List[Dict[str, Any]]:
        return [{"id": v.id, "values": v.values, "metadata": v.metadata}
                for v in self._storage.namespace_map.get(namespace, [])]

    def get_namespace_count(self, namespace: str) -> int:
        return len(self._storage.namespace_map.get(namespace, []))

    def get_storage_info(self) -> Dict[str, Any]:
        return self._storage.get_storage_info()

    # ------------------------------------------------------------------ additive surface
    def find_similar_batch(self, queries: Sequence[Union[VectorDTO, Sequence[float]]], top_k: int,
                           namespace: str = "default", metric: str = "cosine", filter: MetadataFilter = None,  # noqa: A002
                           enrich: bool = True, group_by: Optional[str] = None) -> List[List[dict]]:
        """One result list per query, each exactly what ``find_similar`` returns for that query."""
        q = np.asarray([getattr(v, "values", v) for v in queries], dtype=np.float32)
        if q.ndim != 2 or q.shape[0] == 0:
            return [[] for _ in range(len(queries))]
        grouped = {"group_by": group_by} if group_by is not None else {}
        rows, scores, counts = self._index.search_batch(q, top_k, namespace, metric=metric,
                                                        filter=self._resolve_filter(namespace, filter), **grouped)
        out = []
        for i in range(q.shape[0]):
            n = int(counts[i])
            ids = self._index.uuids_of(namespace, rows[i, :n]) if n else []
            out.append(self._enrich(list(zip(ids, (float(s) for s in scores[i, :n]))), namespace, enrich))
        return out

    def find_in_range(self, query: VectorDTO, radius: float, namespace: str = "default", metric: str = "cosine",
                      filter: MetadataFilter = None, enrich: bool = True) -> List[dict]:  # noqa: A002
        """Every stored vector with hnswlib-form distance <= ``radius`` (cosine: similarity >= 1 - radius),
        nearest first; same result dicts as ``find_similar``."""
        results = self._index.range_search(query, radius, namespace, metric,
                                           filter=self._resolve_filter(namespace, filter))
        return self._enrich([(r.vector_id, r.score) for r in results], namespace, enrich)

    def upsert_matrix(self, matrix: np.ndarray, namespace: str = "default",
                      metadata: Optional[Sequence[Mapping[str, Any]]] = None) -> List[UUID]:
        """Bulk ingest: one H2D append for the whole matrix, ids minted in bulk.  Returns the new ids."""
        data = np.ascontiguousarray(matrix, dtype=np.float32)
        if data.ndim != 2:
            raise ValueError("matrix must be [n, dim]")
        n = data.shape[0]
        if metadata is not None and len(metadata) != n:
            raise ValueError("len(metadata) != rows")
        id_bytes = _random_uuid_bytes(n)
        ids = [UUID(bytes=id_bytes[i].tobytes()) for i in range(n)]
        vecs = StoredVector.rows_of(data, ids, metadata)
        # index first: it is the step that can refuse the block (wrong dimension, out of device memory); a block the
        # index refused never reaches the storage, so the two cannot disagree
        self._index.add_matrix(data, namespace, ids=ids, metadata=metadata)
        try:
            self._storage.write_vectors(vecs, namespace)
        except Exception:
            self._index.remove(ids, namespace)
            raise
        self._touch(namespace)
        return ids

    # ------------------------------------------------------------------ internals
    def _touch(self, namespace: str) -> None:
        self._mutations[namespace] = self._mutations.get(namespace, 0) + 1
        for key in [k for k in self._filters if k[0] == namespace]:
            self._filters.pop(key)[0].close()

    def _enrich(self, hits, namespace: str, enrich: bool) -> List[dict]:
        if not enrich:
            return [{"id": vid, "score": score} for vid, score in hits]
        stored = {v.id: v for v in self._storage.read_vectors([vid for vid, _ in hits], namespace) if v}
        out = []
        for vid, score in hits:   # hit order kept, ids missing from storage dropped (query_processor.py:38-48)
            v = stored.get(vid)
            if v:
                out.append({"id": v.id, "values": v.values, "metadata": v.metadata, "score": score})
        return out

    def _resolve_filter(self, namespace: str, flt: MetadataFilter):
        """dict of equality constraints / predicate over metadata -> prepared device filter (cached until the
        namespace changes).  Constraints over keys the index holds as device columns are evaluated by
        ``mlv_filter_create_where``; anything else (callables, unhashable / ``None`` values, keys beyond the
        column limit) is evaluated on the host against the storage's metadata (SURVEY H5)."""
        if flt is None or isinstance(flt, PreparedFilter):
            return flt
        if self._index.dimension(namespace) is None:
            return None
        if isinstance(flt, Mapping):
            on_device = self._index.where(namespace, flt)   # metadata columns on the device (columns.py)
            if on_device is not None:
                return on_device
            items = tuple(sorted(flt.items(), key=lambda kv: kv[0]))
            try:
                key = (namespace, hash(items), items)
            except TypeError:
                key = None
            pred = host_predicate(flt)
        else:
            key, pred = None, flt
        if key is not None and key in self._filters:
            return self._filters[key][0]
        by_id = {v.id: v.metadata for v in self._storage.namespace_map.get(namespace, [])}

        def passes(uid):
            md = by_id.get(uid)
            return md is not None and bool(pred(md))

        prepared = self._index.prepare_filter(namespace, passes)
        if key is not None:
            self._filters[key] = (prepared, self._mutations.get(namespace, 0))
        return prepared
