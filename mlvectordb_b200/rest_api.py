"""``GpuRestAPI``: the reference's HTTP surface over ``GpuQueryProcessor`` (SURVEY.md section 8f rank 1).

The nine routes the reference server really has keep their paths, request / response models, status codes
and messages (``src/mlvectordb/api/rest_api.py:17-46`` models, ``:96-311`` routes), so existing clients of
``RestAPI`` work unchanged against ``GpuRestAPI(GpuQueryProcessor(storage, GpuIndex(...)))``:

    POST /vectors . PUT /vectors/batch . POST /search . DELETE /vectors . GET /namespaces .
    GET /namespaces/vectors . GET /storage/info . GET /health . POST /log/level

What the GPU index can do beyond the reference becomes reachable from the product surface:

* ``POST /search`` takes three optional fields on top of the reference's ``query / top_k / metric``
  (``rest_api.py:22-25``): ``filter`` (metadata constraints, evaluated on the device columns when possible),
  ``radius`` (range search instead of top-k) and ``include_values`` (``false`` skips the k x d float payload
  that dominates a response at GPU speeds -- rank 2);
* ``POST /search/batch``: many queries per request (tensor-core path from 5 queries on a >= 1 GB matrix);
* ``group_by`` (a metadata key) on ``POST /search``, ``POST /search/batch``, ``POST /query/knn`` and ``POST /query/hybrid``:
  the ``top_k`` (<= 32) nearest groups of rows sharing the key's value, each reported by its nearest row.  Combined with
  ``radius``, with ``top_k`` > 32 or with a key the index keeps on the host only, the request gets 400;
* the routes the reference only documents (``README.md:325-333``) with the request shapes of its example
  client (``examples/api_client.py:26-74``): ``POST /query/knn`` (``vector``, ``k``), ``POST /query/range``
  (``vector``, ``radius``), ``POST /query/similarity`` (``vector``, ``threshold``, ``metric``: cosine
  similarity >= threshold, i.e. radius = 1 - threshold), ``POST /query/hybrid`` (``vector``, ``k``,
  ``filter``), ``GET /statistics`` (per-namespace device rows / tombstones / bytes / metadata columns).

Like the reference, handlers are ``async def`` that call the synchronous processor inline, so the event
loop serialises every index call (``rest_api.py:163-193``; SURVEY 8b "Threading").
"""
from __future__ import annotations

import json
import logging
import math
import time
from contextlib import asynccontextmanager
from typing import Any, Dict, List, Optional
from uuid import UUID

from fastapi import FastAPI, HTTPException, Query, Request, Response, status
from pydantic import BaseModel, Field

from ._capi import MAX_GROUP_K, format_f32_json
from .index import NotDeviceEvaluable
from .interfaces import VectorDTO


# ---- the reference's models (rest_api.py:17-46), field for field ------------------------------------
class VectorCreateRequest(BaseModel):
    values: List[float]
    metadata: Dict[str, Any] = Field(default_factory=dict)


class VectorSearchRequest(BaseModel):
    query: List[float]
    top_k: int = Field(10, ge=1, le=1000)
    metric: str = "cosine"
    # additive
    filter: Optional[Dict[str, Any]] = None
    radius: Optional[float] = None
    include_values: bool = True
    group_by: Optional[str] = None


class VectorSearchResult(BaseModel):
    id: UUID
    values: List[float] = Field(default_factory=list)
    metadata: Dict[str, Any] = Field(default_factory=dict)
    score: float


class VectorDeleteRequest(BaseModel):
    ids: List[UUID]


class BatchVectorRequest(BaseModel):
    vectors: List[VectorCreateRequest]


class VectorInfo(BaseModel):
    id: UUID
    values: List[float]
    metadata: Dict[str, Any]


# ---- additive models ---------------------------------------------------------------------------------
class BatchSearchRequest(BaseModel):
    queries: List[List[float]]
    top_k: int = Field(10, ge=1, le=1000)
    metric: str = "cosine"
    filter: Optional[Dict[str, Any]] = None
    include_values: bool = False
    group_by: Optional[str] = None


class QueryRequest(BaseModel):
    """Request shape of the reference's example client (``examples/api_client.py:26-74``)."""
    vector: List[float]
    k: int = Field(10, ge=1, le=1000)
    radius: Optional[float] = None
    threshold: Optional[float] = None
    metric: str = "cosine"
    filter: Optional[Dict[str, Any]] = None
    namespace: str = "default"
    include_values: bool = True
    type: Optional[str] = None
    group_by: Optional[str] = None


def _constraints(raw: Optional[Dict[str, Any]]) -> Optional[Dict[str, Any]]:
    """JSON has no tuples: ``{"key": ["<", 5]}`` / ``{"key": ["between", 1, 9]}`` become operator constraints
    (``columns.py``); every other value is an equality constraint, as in the reference's sketch."""
    if not raw:
        return None
    from ._capi import PRED_OPS
    out = {}
    for key, want in raw.items():
        if isinstance(want, list) and len(want) in (2, 3) and isinstance(want[0], str) and want[0] in PRED_OPS:
            want = tuple(want)
        out[key] = want
    return out


def _encode_hits(hits) -> bytes:
    """The ``List[VectorSearchResult]`` JSON of the reference (rest_api.py:28-32,163), written directly: the k x d
    stored values go through ``mlv_format_f32_json`` (shortest float32 text, C speed) instead of pydantic
    validation + ``json.dumps`` of k x d Python floats, which costs several ms per response at d = 768."""
    parts = []
    for h in hits:
        values = h.get("values")
        metadata = h.get("metadata")
        score = float(h["score"])
        parts.append(b'{"id":"%s","values":%s,"metadata":%s,"score":%s}' % (
            str(h["id"]).encode(), format_f32_json(values) if values is not None and len(values) else b"[]",
            json.dumps(metadata, default=str).encode() if metadata else b"{}",
            repr(score).encode() if math.isfinite(score) else json.dumps(score).encode()))
    return b"[" + b",".join(parts) + b"]"


def _check_group_by(group_by: Optional[str], radius: Optional[float], top_k: int) -> None:
    """400 for the ``group_by`` requests the index cannot answer."""
    if group_by is None:
        return
    if radius is not None:
        raise HTTPException(status_code=status.HTTP_400_BAD_REQUEST, detail="group_by cannot be combined with radius")
    if top_k > MAX_GROUP_K:
        raise HTTPException(status_code=status.HTTP_400_BAD_REQUEST, detail=f"group_by supports top_k <= {MAX_GROUP_K}")


def _json(payload: bytes) -> Response:
    return Response(content=payload, media_type="application/json")


class GpuRestAPI:
    def __init__(self, query_processor, title: str = "Vector DB API", enable_file_logging: bool = False,
                 log_level: str = "INFO"):
        """Same constructor as the reference ``RestAPI`` (``rest_api.py:49-56``)."""
        self.query_processor = query_processor
        self.title = title
        self.enable_file_logging = enable_file_logging
        self.logger = logging.getLogger("vector_db_api")
        self.logger.setLevel(log_level)
        if enable_file_logging and not any(isinstance(h, logging.FileHandler) for h in self.logger.handlers):
            self.logger.addHandler(logging.FileHandler("vector_db_api.log", encoding="utf-8"))

        @asynccontextmanager
        async def lifespan(app: FastAPI):
            self.logger.info("Vector DB API (GPU index) started")
            yield
            self.logger.info("Vector DB API (GPU index) stopped")

        self.app = FastAPI(title=title, lifespan=lifespan)
        self._setup_middleware()
        self._setup_routes()

    def get_app(self) -> FastAPI:
        return self.app

    # ------------------------------------------------------------------ helpers
    def _fail(self, what: str, exc: Exception):
        self.logger.error("%s: %s", what, exc, exc_info=True)
        raise HTTPException(status_code=status.HTTP_500_INTERNAL_SERVER_ERROR, detail=f"{what}: {exc}")

    def _search(self, query: List[float], top_k: int, namespace: str, metric: str, flt, radius, include_values: bool,
                group_by: Optional[str] = None):
        qp = self.query_processor
        dto = VectorDTO(values=query, metadata={})
        extra = {}
        if flt is not None:
            extra["filter"] = flt
        if not include_values:
            extra["enrich"] = False
        if group_by is not None:
            extra["group_by"] = group_by
        if radius is not None:
            return qp.find_in_range(dto, radius, namespace=namespace, metric=metric, **extra)
        # without additive fields this is exactly the reference's call (rest_api.py:178-183), so any
        # QueryProcessorProtocol implementation works behind the reference routes
        return qp.find_similar(query=dto, top_k=top_k, namespace=namespace, metric=metric, **extra)

    def _bad_group_by(self, group_by: Optional[str], what: str, exc: Exception):
        """A grouped request over a key the device cannot group by is the client's error (400); anything else is not."""
        if group_by is None:
            self._fail(what, exc)
        raise HTTPException(status_code=status.HTTP_400_BAD_REQUEST, detail=str(exc))

    # ------------------------------------------------------------------ routes
    def _setup_routes(self):
        app, qp = self.app, self.query_processor

        @app.post("/vectors", status_code=status.HTTP_201_CREATED)
        async def insert_vector(vector: VectorCreateRequest, namespace: str = Query("default")):
            try:
                qp.insert(VectorDTO(values=vector.values, metadata=vector.metadata), namespace)
                return {"status": "success", "message": "Vector inserted"}
            except Exception as e:  # noqa: BLE001 -- the reference maps everything to 500 (rest_api.py:116-124)
                self._fail("Insert failed", e)

        @app.put("/vectors/batch")
        async def upsert_vectors(batch_request: BatchVectorRequest, namespace: str = Query("default")):
            try:
                dtos = [VectorDTO(values=v.values, metadata=v.metadata) for v in batch_request.vectors]
                qp.upsert_many(dtos, namespace)
                return {"status": "success", "message": f"{len(dtos)} vectors upserted"}
            except Exception as e:  # noqa: BLE001
                self._fail("Batch upsert failed", e)

        @app.post("/search", response_model=List[VectorSearchResult])
        async def search_similar(search_request: VectorSearchRequest, namespace: str = Query("default")):
            r = search_request
            _check_group_by(r.group_by, r.radius, r.top_k)
            try:
                return _json(_encode_hits(self._search(r.query, r.top_k, namespace, r.metric, _constraints(r.filter), r.radius,
                                                       r.include_values, r.group_by)))
            except NotDeviceEvaluable as e:
                self._bad_group_by(r.group_by, "Search failed", e)
            except Exception as e:  # noqa: BLE001
                self._fail("Search failed", e)

        @app.post("/search/batch", response_model=List[List[VectorSearchResult]])
        async def search_batch(batch: BatchSearchRequest, namespace: str = Query("default")):
            _check_group_by(batch.group_by, None, batch.top_k)
            grouped = {"group_by": batch.group_by} if batch.group_by is not None else {}
            try:
                per_query = qp.find_similar_batch(batch.queries, batch.top_k, namespace=namespace, metric=batch.metric,
                                                  filter=_constraints(batch.filter), enrich=batch.include_values, **grouped)
                return _json(b"[" + b",".join(_encode_hits(hits) for hits in per_query) + b"]")
            except NotDeviceEvaluable as e:
                self._bad_group_by(batch.group_by, "Batch search failed", e)
            except Exception as e:  # noqa: BLE001
                self._fail("Batch search failed", e)

        @app.delete("/vectors")
        async def delete_vectors(delete_request: VectorDeleteRequest, namespace: str = Query("default")):
            if not delete_request.ids:
                raise HTTPException(status_code=status.HTTP_400_BAD_REQUEST, detail="No IDs provided")
            try:
                gone = qp.delete(delete_request.ids, namespace)
                return {"status": "success" if len(gone) else "error", "message": f"{len(gone)} vectors deleted"}
            except Exception as e:  # noqa: BLE001
                self._fail("Delete failed", e)

        @app.get("/namespaces")
        async def list_namespaces():
            try:
                return {"namespaces": qp.list_namespaces()}
            except Exception as e:  # noqa: BLE001
                self._fail("Failed to list namespaces", e)

        @app.get("/namespaces/vectors", response_model=List[VectorInfo])
        async def get_namespace_vectors(namespace: str = Query("default")):
            try:
                return qp.get_namespace_vectors(namespace)
            except Exception as e:  # noqa: BLE001
                self._fail("Failed to get vectors", e)

        @app.get("/storage/info")
        async def get_storage_info():
            try:
                return qp.get_storage_info()
            except Exception as e:  # noqa: BLE001
                self._fail("Failed to get storage info", e)

        @app.get("/health")
        async def health_check():
            return {"status": "healthy"}

        @app.post("/log/level")
        async def set_log_level(level: str):
            valid = ["DEBUG", "INFO", "WARNING", "ERROR"]
            if level.upper() not in valid:
                raise HTTPException(status_code=status.HTTP_400_BAD_REQUEST, detail=f"Invalid level. Must be one of: {valid}")
            logging.getLogger().setLevel(level.upper())
            self.logger.setLevel(level.upper())
            return {"status": "success", "message": f"Log level set to {level.upper()}"}

        # ---- the routes the reference documents but never built (README.md:325-333) --------------------
        def _query(kind: str):
            async def handler(req: QueryRequest):
                try:
                    radius = req.radius
                    if kind == "range" and radius is None:
                        raise HTTPException(status_code=status.HTTP_400_BAD_REQUEST, detail="radius is required")
                    if kind == "similarity":
                        if req.threshold is None:
                            raise HTTPException(status_code=status.HTTP_400_BAD_REQUEST, detail="threshold is required")
                        radius = 1.0 - req.threshold     # cosine similarity >= threshold
                    if kind in ("knn", "hybrid"):
                        radius = None
                    if kind == "hybrid" and not req.filter:
                        raise HTTPException(status_code=status.HTTP_400_BAD_REQUEST, detail="filter is required")
                    _check_group_by(req.group_by, radius, req.k)
                    hits = self._search(req.vector, req.k, req.namespace, req.metric, _constraints(req.filter), radius,
                                        req.include_values, req.group_by)
                    return _json(b'{"type":"%s","count":%d,"results":%s}' % (kind.encode(), len(hits), _encode_hits(hits)))
                except HTTPException:
                    raise
                except NotDeviceEvaluable as e:
                    self._bad_group_by(req.group_by, f"{kind} query failed", e)
                except Exception as e:  # noqa: BLE001
                    self._fail(f"{kind} query failed", e)
            handler.__name__ = f"query_{kind}"
            return handler

        for kind in ("knn", "range", "similarity", "hybrid"):
            app.post(f"/query/{kind}")(_query(kind))

        @app.get("/statistics")
        async def statistics():
            try:
                index = getattr(qp, "_index", None)
                out = {}
                if index is not None and hasattr(index, "namespaces"):
                    for ns in index.namespaces():
                        out[ns] = dict(index.info(ns), metadata_columns=index.metadata_columns(ns))
                return {"namespaces": out}
            except Exception as e:  # noqa: BLE001
                self._fail("Failed to get statistics", e)

    def _setup_middleware(self):
        @self.app.middleware("http")
        async def log_requests(request: Request, call_next):
            t0 = time.time()
            response = await call_next(request)
            self.logger.info("%s %s -> %d in %.2f ms", request.method, request.url.path, response.status_code,
                             (time.time() - t0) * 1000)
            return response
