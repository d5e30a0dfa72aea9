"""Import the UNMODIFIED reference wrappers over the exact hnswlib stand-in.  TEST ORACLE.

Needs a checkout of the original MLVectorDB project at ``BASELINE.json``'s ``reference_path``
(``MLV_REFERENCE_ROOT`` overrides it).
The reference modules import each other as ``src.mlvectordb...`` and need the reference
root on ``sys.path`` (reference ``storage_engine_in_memory.py:6-7``, ``pyproject.toml:6``);
``src/mlvectordb/__init__.py:19`` imports ``Index`` eagerly, which imports ``hnswlib`` --
so ``sys.modules['hnswlib']`` is pre-seeded with ``oracle.hnswlib_exact``.

Used by ``tests/golden/make_golden.py`` to generate the committed fixtures, which the tests replay
without the reference.
"""
from __future__ import annotations

import importlib
import json
import os
import sys
from types import SimpleNamespace

with open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "BASELINE.json")) as _f:
    REFERENCE_ROOT = os.environ.get("MLV_REFERENCE_ROOT", json.load(_f)["reference_path"])


def available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "src", "mlvectordb"))


def load(lift_cap: bool = False) -> SimpleNamespace:
    """Return the reference's classes, running over the exact stand-in."""
    if not available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT}")
    from . import hnswlib_exact

    hnswlib_exact.ENFORCE_MAX_ELEMENTS = not lift_cap
    sys.modules["hnswlib"] = hnswlib_exact
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    idx = importlib.import_module("src.mlvectordb.implementations.index")
    qp = importlib.import_module("src.mlvectordb.implementations.query_processor")
    vec = importlib.import_module("src.mlvectordb.implementations.vector")
    ivec = importlib.import_module("src.mlvectordb.interfaces.vector")
    st = importlib.import_module("src.mlvectordb.implementations.storage_engine_in_memory")
    return SimpleNamespace(
        Index=idx.Index,
        SearchResult=idx.SearchResult,
        QueryProcessor=qp.QueryProcessor,
        Vector=vec.Vector,
        VectorDTO=ivec.VectorDTO,
        StorageEngineInMemory=st.StorageEngineInMemory,
        hnswlib=hnswlib_exact,
    )
