"""Grouped search (``mlv_index_search_grouped``): the contract restated in numpy.  TEST ORACLE.

No reference code exists (group-by search as Qdrant, Milvus and Vespa offer it); the semantics are *defined* here, over
the distances of ``oracle/exact.py``.
"""
from typing import Optional

import numpy as np

from oracle.exact import COLUMN_MISSING


def grouped_topk(dists, groups, k: int, allow: Optional[np.ndarray] = None):
    """The k nearest groups of one query, one best row per group.

    ``dists``: the query's distance to every row (the scan's fp32 arithmetic); ``groups``: every row's int32 group code
    (``COLUMN_MISSING`` = no group); ``allow``: optional bool mask (live AND passing).  Rows that are allowed and have a
    group, ordered by ``(distance, row)``; the first row of every group not seen yet is kept, up to k of them.
    Returns ``(rows int64, dists, groups int32)`` of length ``min(k, distinct groups)``, ascending.
    """
    d = np.asarray(dists)
    g = np.asarray(groups, dtype=np.int32)
    cand = g != COLUMN_MISSING
    if allow is not None:
        cand &= np.asarray(allow, dtype=bool)
    rows = np.flatnonzero(cand).astype(np.int64)
    order = rows[np.lexsort((rows, d[rows]))]
    _, first = np.unique(g[order], return_index=True)   # first occurrence of each group along the walk
    keep = order[np.sort(first)][:k]
    return keep, d[keep], g[keep]
