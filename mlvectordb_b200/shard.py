"""``DeviceShard``: one namespace's (or one row shard's) device-resident row matrix.

Thin object wrapper over the C ABI (``include/mlv_index.h``); holds no search logic of its own.
It plays the role the per-namespace ``hnswlib.Index`` object plays in the reference
(``src/mlvectordb/implementations/index.py:19,32-48``): rows are addressed by local row number
(hnswlib labels, ``index.py:56-63``), ``add`` = ``add_items`` (``:65``), ``mark_deleted`` (``:80``),
``search`` = ``knn_query`` (``:111``).
"""
from __future__ import annotations

import ctypes as C
import weakref
from typing import Optional, Tuple

import numpy as np

from . import _capi
from ._capi import METRIC_CODE, IndexInfo, check

ALIASES = {"euclidean": "l2", "dot": "ip", "inner_product": "ip"}


def canonical_space(space: str) -> str:
    s = ALIASES.get(space, space)
    if s not in METRIC_CODE:
        raise ValueError(f"unknown space {space!r}; expected one of l2, ip, cosine")
    return s


def pack_bitmap(mask: np.ndarray) -> np.ndarray:
    """bool[rows] -> uint32 words, bit (r & 31) of word (r >> 5) = mask[r]."""
    mask = np.ascontiguousarray(mask, dtype=bool)
    n = mask.shape[0]
    words = (n + 31) // 32
    if n != words * 32:
        padded = np.zeros(words * 32, dtype=bool)
        padded[:n] = mask
        mask = padded
    return np.packbits(mask, bitorder="little").view(np.uint32)


def key_parts(keys: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
    """Candidate keys (uint64: f32_orderable(distance) << 32 | row, csrc/common.cuh) -> (distance float32, row uint32)."""
    k = np.asarray(keys, dtype=np.uint64)
    o = (k >> np.uint64(32)).astype(np.uint32)
    bits = np.where(o & np.uint32(0x80000000), o & np.uint32(0x7FFFFFFF), ~o).astype(np.uint32)
    return bits.view(np.float32), (k & np.uint64(0xFFFFFFFF)).astype(np.uint32)


def make_keys(dist: np.ndarray, rows: np.ndarray) -> np.ndarray:
    """(distance float32, row) -> the kernels' uint64 keys, whose unsigned order is (distance, row) ascending."""
    b = np.ascontiguousarray(dist, dtype=np.float32).view(np.uint32)
    o = np.where(b & np.uint32(0x80000000), ~b, b | np.uint32(0x80000000)).astype(np.uint64)
    return (o << np.uint64(32)) | np.asarray(rows, dtype=np.uint64)


class DeviceShard:
    def __init__(self, dim: int, space: str = "l2", capacity: int = 0, device: int = 0, row_base: int = 0):
        self.space = canonical_space(space)
        self.dim = int(dim)
        self.device = int(device)
        self._lib = _capi.lib()
        self._h = C.c_void_p()
        check(self._lib.mlv_index_create(self.dim, METRIC_CODE[self.space], int(capacity), self.device, C.byref(self._h)))
        self._filters = weakref.WeakSet()   # prepared filters of this shard: released with it (they hold device buffers)
        if row_base:
            self.set_row_base(row_base)

    # -- lifecycle ------------------------------------------------------------------------
    def close(self) -> None:
        if getattr(self, "_h", None) and self._h.value:
            for f in list(getattr(self, "_filters", ())):
                f.close()
            self._lib.mlv_index_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, status: int) -> None:
        check(status, self._h)

    def set_row_base(self, row_base: int) -> None:
        self._ck(self._lib.mlv_index_set_row_base(self._h, int(row_base)))

    def info(self) -> IndexInfo:
        inf = IndexInfo()
        self._ck(self._lib.mlv_index_info(self._h, C.byref(inf)))
        return inf

    @property
    def rows(self) -> int:
        return int(self.info().rows)

    @property
    def live(self) -> int:
        return int(self.info().live)

    # -- mutation -------------------------------------------------------------------------
    def add(self, rows: np.ndarray) -> int:
        x = np.ascontiguousarray(rows, dtype=np.float32)
        if x.ndim == 1:
            x = x[None, :]
        if x.ndim != 2 or x.shape[1] != self.dim:
            raise ValueError(f"expected rows of dimension {self.dim}, got shape {x.shape}")
        first = C.c_uint64()
        self._ck(self._lib.mlv_index_add(self._h, x.ctypes.data, x.shape[0], C.byref(first)))
        return int(first.value)

    def add_device(self, ptr: int, n: int) -> int:
        first = C.c_uint64()
        self._ck(self._lib.mlv_index_add_device(self._h, C.c_void_p(ptr), int(n), C.byref(first)))
        return int(first.value)

    def add_synthetic(self, seed: int, first_gen_row: int, n: int, scaled: bool = False) -> int:
        first = C.c_uint64()
        self._ck(self._lib.mlv_index_add_synthetic(self._h, int(seed), int(first_gen_row), int(n), int(bool(scaled)),
                                                   C.byref(first)))
        return int(first.value)

    def mark_deleted(self, rows) -> int:
        r = np.ascontiguousarray(rows, dtype=np.uint64)
        changed = C.c_uint64()
        self._ck(self._lib.mlv_index_mark_deleted(self._h, r.ctypes.data, r.shape[0], C.byref(changed)))
        return int(changed.value)

    def compact(self) -> np.ndarray:
        """Drop tombstoned rows; returns old_to_new (int64, -1 for dropped rows)."""
        n = self.rows
        mapping = np.empty(n, dtype=np.int64)
        new_rows = C.c_uint64()
        self._ck(self._lib.mlv_index_compact(self._h, mapping.ctypes.data if n else None, C.byref(new_rows)))
        return mapping

    def clear(self) -> None:
        self._ck(self._lib.mlv_index_clear(self._h))

    # -- query ----------------------------------------------------------------------------
    def prepare_filter(self, filt) -> "PreparedFilter":
        """Upload a filter once (bool mask per row, or packed uint32 words) for repeated searches."""
        words = self._filter_words(filt)
        return PreparedFilter(self, words)

    def _filter_words(self, filt) -> Optional[np.ndarray]:
        if filt is None or isinstance(filt, PreparedFilter):
            return None
        f = np.asarray(filt)
        n = self.rows
        if f.dtype == np.uint32:
            if f.shape[0] < (n + 31) // 32:
                raise ValueError("filter bitmap shorter than ceil(rows/32) words")
            return np.ascontiguousarray(f)
        if f.shape[0] != n:
            raise ValueError(f"filter mask has {f.shape[0]} entries for {n} rows")
        return pack_bitmap(f.astype(bool))

    def search(self, queries: np.ndarray, k: int, filt=None) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
        """-> (dists f32 [nq,k] hnswlib-form ascending, rows i64 [nq,k], counts i32 [nq])."""
        q = np.ascontiguousarray(queries, dtype=np.float32)
        if q.ndim == 1:
            q = q[None, :]
        if q.ndim != 2 or q.shape[1] != self.dim:
            raise ValueError(f"expected queries of dimension {self.dim}, got shape {q.shape}")
        nq = q.shape[0]
        dists = np.empty((nq, k), dtype=np.float32)
        rows = np.empty((nq, k), dtype=np.int64)
        counts = np.empty(nq, dtype=np.int32)
        if filt is None:      # the batch-1 latency path: nothing between the caller and the one launch but this call
            st = self._lib.mlv_index_search(self._h, q.ctypes.data, nq, int(k), None, dists.ctypes.data, rows.ctypes.data,
                                            counts.ctypes.data)
            if st:
                self._ck(st)
            return dists, rows, counts
        fw = self._filter_words(filt)
        with _bound(self, filt):
            self._ck(self._lib.mlv_index_search(self._h, q.ctypes.data, nq, int(k), fw.ctypes.data if fw is not None else None,
                                                dists.ctypes.data, rows.ctypes.data, counts.ctypes.data))
        return dists, rows, counts

    def search_device(self, q_ptr: int, nq: int, k: int, out_d_ptr: int, out_r_ptr: int, out_c_ptr: int,
                      filter_ptr: int = 0, stream: int = 0) -> None:
        """All pointers are device addresses (e.g. ``tensor.data_ptr()``); enqueues on ``stream``
        (a ``cudaStream_t`` value such as ``torch.cuda.current_stream().cuda_stream``; 0 = the
        legacy default stream) and does not synchronise."""
        self._ck(self._lib.mlv_index_search_device(
            self._h, C.c_void_p(q_ptr), int(nq), int(k), C.c_void_p(filter_ptr) if filter_ptr else None,
            C.c_void_p(out_d_ptr), C.c_void_p(out_r_ptr), C.c_void_p(out_c_ptr), C.c_void_p(stream)))

    # -- fused multi-GPU exchange (include/mlv_index.h: mlv_exchange_*) ---------------------
    def attach_exchange(self, exchange: "Exchange", row_bases) -> None:
        rb = np.ascontiguousarray(row_bases, dtype=np.uint64)
        assert rb.shape[0] == exchange.world
        self._ck(self._lib.mlv_index_attach_exchange(self._h, exchange._x, rb.ctypes.data))
        self._exchange = exchange  # keep it alive as long as the shard uses it

    def exchange_supported(self, k: int) -> bool:
        return bool(self._lib.mlv_index_exchange_supported(self._h, int(k)))

    def search_exchange_device(self, q_ptr: int, nq: int, k: int, out_d_ptr: int, out_r_ptr: int, out_c_ptr: int,
                               filter_ptr: int = 0, stream: int = 0) -> None:
        """Collective: local scan + peer-memory exchange + merge in one kernel; outputs hold the GLOBAL top-k."""
        self._ck(self._lib.mlv_index_search_exchange_device(
            self._h, C.c_void_p(q_ptr), int(nq), int(k), C.c_void_p(filter_ptr) if filter_ptr else None,
            C.c_void_p(out_d_ptr), C.c_void_p(out_r_ptr), C.c_void_p(out_c_ptr), C.c_void_p(stream)))

    def submit(self, queries: np.ndarray, k: int, exchange: bool = False) -> "PendingSearch":
        """Start a search and return at once (``mlv_index_submit``); ``.result()`` blocks for the answer.
        Up to four may be in flight per shard."""
        q = np.ascontiguousarray(queries, dtype=np.float32).reshape(-1, self.dim)
        ticket = C.c_uint32()
        self._ck(self._lib.mlv_index_submit(self._h, q.ctypes.data, q.shape[0], int(k), int(bool(exchange)), C.byref(ticket)))
        return PendingSearch(self, int(ticket.value), q.shape[0], int(k))

    def search_exchange(self, queries: np.ndarray, k: int):
        """Collective, host buffers: like ``search`` but the outputs hold the GLOBAL top-k of all row shards."""
        q = np.ascontiguousarray(queries, dtype=np.float32).reshape(-1, self.dim)
        nq = q.shape[0]
        dists = np.empty((nq, k), dtype=np.float32)
        rows = np.empty((nq, k), dtype=np.int64)
        counts = np.empty(nq, dtype=np.int32)
        self._ck(self._lib.mlv_index_search_exchange(self._h, q.ctypes.data, nq, int(k), None, dists.ctypes.data,
                                                     rows.ctypes.data, counts.ctypes.data))
        return dists, rows, counts

    RANGE_OVERFLOW = 1 << 63

    def range_exchange_supported(self) -> bool:
        return bool(self._lib.mlv_index_range_exchange_supported(self._h))

    def range_search_exchange(self, queries: np.ndarray, radius: float, max_hits: int = 8192):
        """Collective: the GLOBAL hit lists of a row-sharded range search from one fused kernel per query
        (``mlv_index_range_search_exchange``).  -> list per query of (dists, global rows), or None when some rank's list
        did not fit its share of the exchange slot (every rank gets None: take the all-gather path)."""
        q = np.ascontiguousarray(queries, dtype=np.float32).reshape(-1, self.dim)
        nq = q.shape[0]
        dists = np.empty((nq, max_hits), dtype=np.float32)
        rows = np.empty((nq, max_hits), dtype=np.int64)
        counts = np.zeros(nq, dtype=np.uint64)
        self._ck(self._lib.mlv_index_range_search_exchange(self._h, q.ctypes.data, nq, C.c_float(radius), None, int(max_hits),
                                                           dists.ctypes.data, rows.ctypes.data, counts.ctypes.data))
        if (counts == np.uint64(0xFFFFFFFFFFFFFFFF)).any():
            raise RuntimeError("sharded range search: a peer rank did not post its hits within the exchange timeout")
        if (counts >= np.uint64(self.RANGE_OVERFLOW)).any():
            return None
        return [(dists[i, : int(counts[i])].copy(), rows[i, : int(counts[i])].copy()) for i in range(nq)]

    def range_search(self, queries: np.ndarray, radius: float, filt=None, max_hits: int = 1024):
        """-> list per query of (dists f32 [hits], rows i64 [hits]) ascending (d, row)."""
        q = np.ascontiguousarray(queries, dtype=np.float32)
        if q.ndim == 1:
            q = q[None, :]
        if q.ndim != 2 or q.shape[1] != self.dim:
            raise ValueError(f"expected queries of dimension {self.dim}, got shape {q.shape}")
        nq = q.shape[0]
        fw = self._filter_words(filt)
        while True:
            dists = np.empty((nq, max_hits), dtype=np.float32)
            rows = np.empty((nq, max_hits), dtype=np.int64)
            counts = np.zeros(nq, dtype=np.uint64)
            with _bound(self, filt):
                self._ck(self._lib.mlv_index_range_search(
                    self._h, q.ctypes.data, nq, C.c_float(radius), fw.ctypes.data if fw is not None else None, int(max_hits),
                    dists.ctypes.data, rows.ctypes.data, counts.ctypes.data))
            most = int(counts.max()) if nq else 0
            if most <= max_hits:
                return [(dists[i, : int(counts[i])].copy(), rows[i, : int(counts[i])].copy()) for i in range(nq)]
            max_hits = most  # the call reports the total: one retry with an exact buffer

    # -- columnar metadata + device-evaluated predicates (include/mlv_index.h: mlv_index_set_column ...) ----
    def set_column(self, column: int, values, first_row: int = 0) -> None:
        """int32 codes for rows ``first_row ..`` of ``column`` (``_capi.COLUMN_MISSING`` = no value)."""
        v = np.ascontiguousarray(values, dtype=np.int32)
        self._ck(self._lib.mlv_index_set_column(self._h, int(column), int(first_row), v.ctypes.data, v.shape[0]))

    def get_column(self, column: int, first_row: int = 0, n: Optional[int] = None) -> np.ndarray:
        n = self.rows - first_row if n is None else int(n)
        out = np.empty(n, dtype=np.int32)
        self._ck(self._lib.mlv_index_get_column(self._h, int(column), int(first_row), n, out.ctypes.data))
        return out

    def where(self, predicates) -> "PreparedFilter":
        """Prepared filter from a conjunction of ``(column, op, a[, b])`` with op in
        ``== != < <= > >= between``, evaluated on the device over the columns."""
        preds = (_capi.Predicate * max(len(predicates), 1))()
        for i, p in enumerate(predicates):
            column, op, a = p[0], p[1], p[2]
            preds[i] = _capi.Predicate(int(column), _capi.PRED_OPS[op], int(a), int(p[3]) if len(p) > 3 else 0)
        f = C.c_void_p()
        self._ck(self._lib.mlv_filter_create_where(self._h, preds, len(predicates), C.byref(f)))
        return PreparedFilter._adopt(self, f)

    # -- snapshot (include/mlv_index.h: mlv_index_export_rows / export_live / import_rows) ------------------
    def export_rows(self, first_row: int = 0, n: Optional[int] = None, out: Optional[np.ndarray] = None) -> np.ndarray:
        """Rows as stored (cosine: normalised), tombstoned ones included."""
        n = self.rows - first_row if n is None else int(n)
        if out is None:
            out = np.empty((n, self.dim), dtype=np.float32)
        assert out.shape == (n, self.dim) and out.dtype == np.float32 and out.flags.c_contiguous
        self._ck(self._lib.mlv_index_export_rows(self._h, int(first_row), n, out.ctypes.data))
        return out

    def export_live(self) -> np.ndarray:
        """Tombstone bitmap, uint32 words, bit set = live."""
        words = np.zeros((self.rows + 31) // 32, dtype=np.uint32)
        self._ck(self._lib.mlv_index_export_live(self._h, words.ctypes.data, words.shape[0]))
        return words

    def import_rows(self, rows: np.ndarray, live_words: Optional[np.ndarray] = None) -> int:
        """Append stored-form rows without normalising them again; ``live_words`` restores tombstones."""
        x = np.ascontiguousarray(rows, dtype=np.float32)
        if x.ndim != 2 or x.shape[1] != self.dim:
            raise ValueError(f"expected rows of dimension {self.dim}, got shape {x.shape}")
        lw = None
        if live_words is not None:
            lw = np.ascontiguousarray(live_words, dtype=np.uint32)
            if lw.shape[0] < (x.shape[0] + 31) // 32:
                raise ValueError("live bitmap shorter than ceil(rows/32) words")
        first = C.c_uint64()
        self._ck(self._lib.mlv_index_import_rows(self._h, x.ctypes.data, x.shape[0], lw.ctypes.data if lw is not None else None,
                                                 C.byref(first)))
        return int(first.value)

    def order_pairs_device(self, d_ptr: int, r_ptr: int, n: int, out_d_ptr: int, out_r_ptr: int, stream: int = 0) -> None:
        """Order n (distance f32, global row i64) pairs in device memory ascending by (distance, row); entries with
        row < 0 sort last (``mlv_index_order_pairs_device``)."""
        self._ck(self._lib.mlv_index_order_pairs_device(self._h, C.c_void_p(d_ptr), C.c_void_p(r_ptr), int(n), C.c_void_p(out_d_ptr),
                                                        C.c_void_p(out_r_ptr), C.c_void_p(stream)))

    def get_rows(self, rows) -> np.ndarray:
        r = np.ascontiguousarray(rows, dtype=np.uint64)
        out = np.empty((r.shape[0], self.dim), dtype=np.float32)
        self._ck(self._lib.mlv_index_get_rows(self._h, r.ctypes.data, r.shape[0], out.ctypes.data))
        return out

    # -- measurement hooks ------------------------------------------------------------------
    def set_timing(self, enabled: bool) -> None:
        self._ck(self._lib.mlv_index_set_timing(self._h, int(enabled)))

    def scan_time_ms(self) -> Tuple[float, int]:
        ms, n = C.c_double(), C.c_uint64()
        self._ck(self._lib.mlv_index_scan_time_ms(self._h, C.byref(ms), C.byref(n)))
        return float(ms.value), int(n.value)

    def set_tuning(self, key: str, value: int) -> None:
        self._ck(self._lib.mlv_index_set_tuning(self._h, key.encode(), int(value)))

    def debug_timeline(self, max_ctas: int = 1024) -> np.ndarray:
        """[n_ctas, 16] globaltimer ns stamps of the last scan (needs set_tuning('timeline', 1)): 0 start, 1 first tile,
        2 last tile consumed, 3 lists folded, 4 ticket taken, for the last CTA 5 final select / 6 outputs / 7 flag, and finer
        ones: 8 own lists sorted, 9 all lists sorted, last CTA 10 past the fence / 11 threshold / 12 survivors (0 = not taken)."""
        out = np.zeros((max_ctas, 16), dtype=np.uint64)
        n = C.c_uint32()
        self._ck(self._lib.mlv_index_debug_timeline(self._h, out.ctypes.data_as(C.POINTER(C.c_uint64)), max_ctas, C.byref(n)))
        return out[: n.value]

    def gemm_stats(self) -> dict:
        """Counters of the tensor-core batch path (``mlv_index_gemm_stats``)."""
        st = _capi.GemmStats()
        self._ck(self._lib.mlv_index_gemm_stats(self._h, C.byref(st)))
        return {f: getattr(st, f) for f, _ in st._fields_}

    def debug_gemm(self, queries: np.ndarray) -> np.ndarray:
        """Approximate (3xTF32 GEMM-form) distances [nq, rows] of the tensor-core kernel (tests only)."""
        q = np.ascontiguousarray(queries, dtype=np.float32).reshape(-1, self.dim)
        out = np.empty((q.shape[0], self.rows), dtype=np.float32)
        self._ck(self._lib.mlv_index_debug_gemm(self._h, q.ctypes.data_as(C.c_void_p), q.shape[0],
                                                out.ctypes.data_as(C.c_void_p)))
        return out

    def debug_gemm_rounds(self, queries: np.ndarray, passes: int, bn: int, cap: int, rounds=None, kprime: int = 0,
                          thresholds: Optional[np.ndarray] = None, mask: Optional[np.ndarray] = None, max_ctas: int = 0) -> dict:
        """GEMM rounds as a batch search runs them (``mlv_index_debug_gemm_rounds``; tests only).  bn 64 / 128 / 256 =
        single-tile kernel, 0 = CTA pair; rounds = [(end_tile, jrank), ...] (default: one round over every tile);
        thresholds[nq] initial (None = +inf); mask = bool[rows] filter.  -> dict of keys [nq, cap] uint64, counts
        (uncapped), thr, flags, pad_count."""
        q = np.ascontiguousarray(queries, dtype=np.float32).reshape(-1, self.dim)
        nq = q.shape[0]
        if rounds is None:
            rounds = [(-(-self.rows // 128), kprime)]
        ends = np.ascontiguousarray([r[0] for r in rounds], dtype=np.uint32)
        jr = np.ascontiguousarray([r[1] for r in rounds], dtype=np.uint32)
        cfg = _capi.GemmRoundsCfg(int(passes), int(bn), int(max_ctas), int(cap), int(kprime), len(rounds),
                                  ends.ctypes.data_as(C.POINTER(C.c_uint32)), jr.ctypes.data_as(C.POINTER(C.c_uint32)))
        thr = None if thresholds is None else np.ascontiguousarray(thresholds, dtype=np.float32).reshape(nq)
        bm = None if mask is None else pack_bitmap(mask)
        out = {"keys": np.empty((nq, int(cap)), np.uint64), "counts": np.empty(nq, np.uint32),
               "thr": np.empty(nq, np.float32), "flags": np.empty(nq, np.uint32)}
        pad = C.c_uint64()
        self._ck(self._lib.mlv_index_debug_gemm_rounds(
            self._h, q.ctypes.data_as(C.c_void_p), nq, None if thr is None else thr.ctypes.data_as(C.c_void_p),
            None if bm is None else bm.ctypes.data_as(C.c_void_p), C.byref(cfg), out["keys"].ctypes.data_as(C.c_void_p),
            out["counts"].ctypes.data_as(C.c_void_p), out["thr"].ctypes.data_as(C.c_void_p),
            out["flags"].ctypes.data_as(C.c_void_p), C.byref(pad)))
        out["pad_count"] = int(pad.value)
        return out

    def debug_half_scan(self, query: np.ndarray) -> Tuple[np.ndarray, dict]:
        """Approximate distances [rows] the shadow scan's consumers compute for one query (+inf for tombstoned rows) and
        what its certificate is computed from (``mlv_half_scan_debug_t`` as a dict; tests only)."""
        q = np.ascontiguousarray(query, dtype=np.float32).reshape(self.dim)
        out = np.empty(self.rows, dtype=np.float32)
        info = _capi.HalfScanDebug()
        self._ck(self._lib.mlv_index_debug_half_scan(self._h, q.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p),
                                                     C.byref(info)))
        return out, {f: getattr(info, f) for f, _ in info._fields_}

    def debug_q8_scan(self, query: np.ndarray) -> Tuple[np.ndarray, dict]:
        """Approximate distances [rows] the int8 shadow scan's consumers compute for one query (+inf for tombstoned rows)
        and what its certificate is computed from (``mlv_q8_scan_debug_t`` as a dict; tests only)."""
        q = np.ascontiguousarray(query, dtype=np.float32).reshape(self.dim)
        out = np.empty(self.rows, dtype=np.float32)
        info = _capi.Q8ScanDebug()
        self._ck(self._lib.mlv_index_debug_q8_scan(self._h, q.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p),
                                                   C.byref(info)))
        return out, {f: getattr(info, f) for f, _ in info._fields_}

    def kernel_launches(self) -> int:
        n = C.c_uint64()
        self._ck(self._lib.mlv_index_kernel_launches(self._h, C.byref(n)))
        return int(n.value)


class PendingSearch:
    """A search in flight (``DeviceShard.submit``)."""

    def __init__(self, shard: "DeviceShard", ticket: int, nq: int, k: int):
        self._shard, self._ticket, self._nq, self._k = shard, ticket, nq, k
        self._out = None

    def result(self):
        """-> (dists f32 [nq,k], rows i64 [nq,k], counts i32 [nq]); blocks until the search is done."""
        if self._out is None:
            dists = np.empty((self._nq, self._k), dtype=np.float32)
            rows = np.empty((self._nq, self._k), dtype=np.int64)
            counts = np.empty(self._nq, dtype=np.int32)
            s = self._shard
            s._ck(s._lib.mlv_index_collect(s._h, self._ticket, dists.ctypes.data, rows.ctypes.data, counts.ctypes.data))
            self._out = (dists, rows, counts)
        return self._out


class PreparedFilter:
    """A filter bitmap resident on the device with its passing-row list (``mlv_filter_*``)."""

    def __init__(self, shard: DeviceShard, words: np.ndarray):
        self._lib = _capi.lib()
        self._shard = shard
        self._f = C.c_void_p()
        w = np.ascontiguousarray(words, dtype=np.uint32)
        check(self._lib.mlv_filter_create(shard._h, w.ctypes.data, w.shape[0], C.byref(self._f)), shard._h)
        shard._filters.add(self)

    @classmethod
    def _adopt(cls, shard: DeviceShard, handle) -> "PreparedFilter":
        self = cls.__new__(cls)
        self._lib, self._shard, self._f = _capi.lib(), shard, handle
        shard._filters.add(self)
        return self

    def bitmap(self, n_words: Optional[int] = None) -> np.ndarray:
        """The filter's bitmap words as the searches see them."""
        n_words = (self._shard.rows + 31) // 32 if n_words is None else int(n_words)
        out = np.zeros(max(n_words, 1), dtype=np.uint32)
        check(self._lib.mlv_filter_get_bitmap(self._f, out.ctypes.data, n_words), self._shard._h)
        return out[:n_words]

    @property
    def passing(self) -> int:
        n = C.c_uint64()
        check(self._lib.mlv_filter_passing(self._f, C.byref(n)), self._shard._h)
        return int(n.value)

    def close(self) -> None:
        if getattr(self, "_f", None) and self._f.value:
            if self._shard._h.value:          # the shard may already be gone
                self._lib.mlv_filter_destroy(self._f)
            self._f = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class _bound:
    """Context manager: bind a PreparedFilter to the shard for the duration of one call."""

    def __init__(self, shard: DeviceShard, filt):
        self.shard, self.f = shard, filt if isinstance(filt, PreparedFilter) else None

    def __enter__(self):
        if self.f is not None:
            if not self.f._f.value:
                raise RuntimeError("prepared filter was closed (its namespace changed since it was made); prepare it again")
            check(self.shard._lib.mlv_index_set_filter(self.shard._h, self.f._f), self.shard._h)

    def __exit__(self, *exc):
        if self.f is not None:
            self.shard._lib.mlv_index_set_filter(self.shard._h, None)
        return False


class Exchange:
    """Peer-memory exchange buffers of one rank (``mlv_exchange_*``); see ``csrc/exchange.cuh``."""

    HANDLE_BYTES = 64

    def __init__(self, device: int, world: int, rank: int):
        self._lib = _capi.lib()
        self._x = C.c_void_p()
        self.world, self.rank, self.device = int(world), int(rank), int(device)
        hb = (C.c_ubyte * self.HANDLE_BYTES)()
        check(self._lib.mlv_exchange_create(self.device, self.world, self.rank, C.byref(self._x), hb))
        self.handle = bytes(hb)

    def connect(self, all_handles) -> None:
        """``all_handles``: the ``handle`` of every rank, rank-major."""
        blob = b"".join(all_handles)
        assert len(blob) == self.world * self.HANDLE_BYTES
        buf = (C.c_ubyte * len(blob)).from_buffer_copy(blob)
        check(self._lib.mlv_exchange_connect(self._x, buf))

    def check(self) -> None:
        st = self._lib.mlv_exchange_check(self._x)
        if st != _capi.MLV_OK:
            raise RuntimeError("exchange: a peer rank did not post its candidates within the timeout")

    def close(self) -> None:
        if getattr(self, "_x", None) and self._x.value:
            self._lib.mlv_exchange_destroy(self._x)
            self._x = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
