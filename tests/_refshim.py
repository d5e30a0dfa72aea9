"""Test-only stand-ins for the reference's CALLERS of the index (not part of the product).

The original project is not part of this repository, so the drop-in tests need a thin
restatement of what sits around the index: ``Vector`` (reference
``src/mlvectordb/implementations/vector.py:10-42``), an in-memory storage
(``storage_engine_in_memory.py:10-86``, only the calls ``QueryProcessor`` makes) and
``QueryProcessor`` (``query_processor.py:11-62``).  Behaviour restated, not copied: uuid4 ids,
fp32 value copies, hit enrichment in hit order dropping ids missing from storage, delete ->
remove -> rebuild-if-flagged.
"""
from __future__ import annotations

import uuid
from collections import defaultdict

import numpy as np


class Vector:
    def __init__(self, values, metadata=None):
        self.id = uuid.uuid4()
        self.values = np.array(values, dtype=np.float32)
        self.metadata = metadata or {}


class Storage:
    def __init__(self):
        self._data = defaultdict(dict)

    def write_vectors(self, vectors, namespace):
        for v in vectors:
            self._data[namespace][v.id] = v

    def write(self, vector, namespace):
        self._data[namespace][vector.id] = vector

    def read_vectors(self, ids, namespace):
        return [self._data[namespace].get(i) for i in ids]

    def delete(self, vid, namespace):
        return self._data[namespace].pop(vid, None) is not None

    @property
    def namespace_map(self):
        return {ns: list(d.values()) for ns, d in self._data.items()}


class InMemoryStorage(Storage):
    """plus the two storage calls ``GpuQueryProcessor`` forwards (``storage_engine_in_memory.py:22-30,61-69``)"""

    @property
    def list_namespaces(self):
        return list(self._data)

    def get_storage_info(self):
        return {"total_vectors": sum(len(d) for d in self._data.values())}


class QueryProcessor:
    def __init__(self, storage, index):
        self._storage = storage
        self._index = index

    def insert(self, dto, namespace="default"):
        v = Vector(dto.values, dto.metadata)
        self._storage.write(v, namespace)
        self._index.add([v], namespace)

    def upsert_many(self, dtos, namespace="default"):
        vs = [Vector(d.values, d.metadata) for d in dtos]
        self._storage.write_vectors(vs, namespace)
        self._index.add(vs, namespace)

    def find_similar(self, query, top_k, namespace="default", metric="cosine"):
        hits = self._index.search(query, top_k=top_k, namespace=namespace, metric=metric)
        if not hits:
            return []
        stored = {v.id: v for v in self._storage.read_vectors([h.vector_id for h in hits], namespace) if v}
        out = []
        for h in hits:
            v = stored.get(h.vector_id)
            if v:
                out.append({"id": v.id, "values": v.values, "metadata": v.metadata, "score": h.score})
        return out

    def delete(self, ids, namespace="default"):
        done = [i for i in ids if self._storage.delete(i, namespace)]
        self._index.remove(ids, namespace)
        if getattr(self._index, "is_rebuild_required", None) and self._index.is_rebuild_required(namespace):
            self._index.rebuild({namespace: self._storage.namespace_map.get(namespace, [])}, metric=self._index._space)
        return done
