/*
 * mlv_index.h -- C ABI of the B200-native exact-search index (libmlvindex.so).
 *
 * This is the drop-in boundary for the hot path of SudYar/MLVectorDB: everything the
 * reference does through `hnswlib.Index` inside
 * `src/mlvectordb/implementations/index.py` is replaced by the calls below.  Plain pointers
 * and sizes only; no torch / C++ types cross this boundary.  Every function returns an
 * `mlv_status` and never throws or aborts across the ABI (SURVEY.md section 8b).
 *
 * Arithmetic contract (hnswlib 0.8.0 form, reference index.py:36 selects it):
 *   MLV_L2      d = sum_i (x_i - q_i)^2        (squared, no sqrt)
 *   MLV_IP      d = 1 - sum_i x_i q_i
 *   MLV_COSINE  rows are normalised when added and queries when searched with
 *               1/(sqrt(sum v_i^2) + 1e-30) in fp32, then d = 1 - sum_i x_i q_i
 * All results are ascending by (d, row).  The Python shim applies the reference's
 * `score = 1 - d` for metric == "cosine" (reference index.py:126-127).
 *
 * Rows are addressed by their LOCAL row number inside the index (the role hnswlib labels
 * play at reference index.py:56-63); results carry `row_base + local row` so that shards of
 * one namespace report global rows.
 */
#ifndef MLV_INDEX_H
#define MLV_INDEX_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MLV_ABI_VERSION 6

typedef struct mlv_index *mlv_index_t;

enum mlv_metric { MLV_L2 = 0, MLV_IP = 1, MLV_COSINE = 2 };

enum mlv_status {
    MLV_OK = 0,
    MLV_E_INVALID = 1,      /* bad argument (NULL handle, k == 0, unknown metric ...) */
    MLV_E_CUDA = 2,         /* a CUDA runtime call failed; see mlv_last_error() */
    MLV_E_NOMEM = 3,        /* device or host allocation failed */
    MLV_E_UNSUPPORTED = 4,  /* valid request outside this build's limits (k > MLV_MAX_K, dim too large) */
    MLV_E_NO_DEVICE = 5     /* no usable CUDA device: there is NO CPU fallback */
};

#define MLV_MAX_K 1024u   /* reference REST bound is top_k <= 1000 (rest_api.py:24) */

typedef struct mlv_index_info {
    uint64_t rows;          /* stored rows including tombstoned ones (hnswlib get_current_count, index.py:56) */
    uint64_t live;          /* rows - tombstoned */
    uint64_t capacity;      /* rows the current device allocation can hold */
    uint64_t row_base;      /* added to local rows in every result */
    uint64_t device_bytes;  /* bytes of HBM held by this index */
    uint32_t dim;           /* logical dimension d */
    uint32_t ld;            /* floats per stored row (d rounded up to 4 -> 16-byte aligned rows) */
    int32_t metric;
    int32_t device;
} mlv_index_info_t;

/* ABI version of the loaded library (== MLV_ABI_VERSION of the header it was built from). */
int mlv_abi_version(void);
/* Number of visible CUDA devices, or 0.  Never fails. */
int mlv_device_count(void);
/* Text for a status code. */
const char *mlv_status_string(int status);
/* Last error text of this handle (valid until the next call on it); "" when none. */
const char *mlv_last_error(mlv_index_t h);

/*
 * Create an empty index for `dim`-dimensional fp32 rows on CUDA device `device`.
 * Replaces hnswlib.Index(space, dim) + init_index(...) (reference index.py:36-38); there is
 * no max_elements cap -- `capacity_hint` rows are pre-allocated and the matrix grows by
 * doubling.  Fails with MLV_E_NO_DEVICE when no GPU is present.
 */
int mlv_index_create(uint32_t dim, int metric, uint64_t capacity_hint, int device, mlv_index_t *out);
int mlv_index_destroy(mlv_index_t h);

/* Global row number of local row 0 (row shards of one namespace).  Default 0. */
int mlv_index_set_row_base(mlv_index_t h, uint64_t row_base);

/*
 * Append n rows (host memory, row-major [n, dim] fp32).  Replaces add_items (reference
 * index.py:65,158).  The data is copied (ownership stays with the caller, like
 * np.array(data, dtype=float32) at index.py:65); cosine rows are normalised on the device.
 * *first_row receives the local row of rows[0]; rows are numbered consecutively and never
 * reused until mlv_index_compact (reference labels: index.py:56-60).
 */
int mlv_index_add(mlv_index_t h, const float *rows, uint64_t n, uint64_t *first_row);
/* Same, rows already in device memory of this index's device. */
int mlv_index_add_device(mlv_index_t h, const float *rows_dev, uint64_t n, uint64_t *first_row);
/*
 * Append n rows produced on the device by the deterministic counter-based generator that
 * oracle/exact_scan.c::orc_fill_synthetic and oracle/synthetic.py restate bit for bit
 * (generator row numbers first_gen_row .. first_gen_row+n-1; `scaled` != 0 multiplies each
 * row by its per-row scale).  Benchmark / parity-test input path: 10M x 768 rows are
 * produced in HBM without a 30 GB host copy.
 */
int mlv_index_add_synthetic(mlv_index_t h, uint64_t seed, uint64_t first_gen_row, uint64_t n, int scaled,
                            uint64_t *first_row);

/*
 * Tombstone rows.  Replaces mark_deleted (reference index.py:80).  Rows >= info.rows or already
 * tombstoned are ignored (the reference never passes them: index.py:77-82 pops the id map
 * first).  *newly_deleted (nullable) receives how many rows changed state.
 */
int mlv_index_mark_deleted(mlv_index_t h, const uint64_t *rows, uint64_t n, uint64_t *newly_deleted);

/*
 * Drop tombstoned rows and renumber the survivors 0..live-1 in their old order (the
 * per-namespace part of reference Index.rebuild, index.py:131-162, without re-uploading).
 * old_to_new (nullable, host, info.rows entries) receives the new local row of every old
 * row, or -1 for dropped rows.
 */
int mlv_index_compact(mlv_index_t h, int64_t *old_to_new, uint64_t *new_rows);
/* Remove all rows (keeps the allocation). */
int mlv_index_clear(mlv_index_t h);

/*
 * Exact k-nearest-neighbour search of nq queries (host memory, [nq, dim] fp32).  Replaces
 * knn_query (reference index.py:111,115) and extends it with batches and a filter.
 *   filter_bitmap  nullable; host uint32 words, bit (r & 31) of word (r >> 5) set = local row r
 *                  may be returned (hnswlib-0.8 `filter=` semantics).  ceil(rows/32) words.
 *   out_dists      [nq, k] hnswlib-form distances ascending; +inf padding
 *   out_rows       [nq, k] row_base + local row; -1 padding
 *   out_counts     [nq]    min(k, live-and-passing rows): the clamp the reference applies at
 *                          index.py:103-107 falls out of the scan, hnswlib's "cannot fill k"
 *                          RuntimeError (index.py:110-119) cannot occur.
 * 1 <= k <= MLV_MAX_K.  Blocks until the results are in the host buffers.
 * A single query without a per-call bitmap takes the latency path: the raw query rides in the launch parameters,
 * the kernel writes the final top-k into pinned host memory and raises a flag the call polls -- one launch, no
 * copies, no preparation launch (set_tuning("fast_host", 0) disables it).
 */
int mlv_index_search(mlv_index_t h, const float *queries, uint32_t nq, uint32_t k, const uint32_t *filter_bitmap,
                     float *out_dists, int64_t *out_rows, int32_t *out_counts);
/*
 * Same with every pointer in device memory, enqueued on `stream` (a cudaStream_t; NULL = the
 * legacy default stream, as everywhere in CUDA) without synchronising.  Queries must hold
 * nq * dim floats.  The handle's scratch buffers are reused in stream order: use one stream
 * at a time per handle.  Batches that take the tensor-core path (see mlv_index_gemm_stats)
 * synchronise `stream` once before returning.
 */
int mlv_index_search_device(mlv_index_t h, const float *queries_dev, uint32_t nq, uint32_t k,
                            const uint32_t *filter_bitmap_dev, float *out_dists_dev, int64_t *out_rows_dev,
                            int32_t *out_counts_dev, void *stream);

/*
 * Asynchronous host-buffer search: mlv_index_submit copies the queries, enqueues the search on a stream
 * of its own and returns a ticket at once; mlv_index_collect blocks until that search is done and
 * copies the results out (same buffers and meaning as mlv_index_search).  Up to four searches may
 * be in flight per handle, each on its own scratch lane, so a server overlaps one request's copies,
 * launch latency and tail with the next request's scan.  exchange != 0 makes it the collective
 * mlv_index_search_exchange (every rank submits the same sequence of searches).
 */
int mlv_index_submit(mlv_index_t h, const float *queries, uint32_t nq, uint32_t k, int exchange, uint32_t *ticket);
int mlv_index_collect(mlv_index_t h, uint32_t ticket, float *out_dists, int64_t *out_rows, int32_t *out_counts);

/*
 * Range (radius) search: every live (and passing) row with d <= radius, ascending (d, row).
 * No reference code exists for it (README.md:121,215 only); semantics are defined by
 * oracle/exact.py::range_stream.  Each query owns max_hits slots of out_dists / out_rows;
 * out_counts[q] receives the TOTAL number of hits, which may exceed max_hits -- in that
 * case the max_hits slots hold an unspecified subset and the caller retries with a larger
 * buffer (the Python shim does).
 */
int mlv_index_range_search(mlv_index_t h, const float *queries, uint32_t nq, float radius,
                           const uint32_t *filter_bitmap, uint64_t max_hits, float *out_dists, int64_t *out_rows,
                           uint64_t *out_counts);

/*
 * Same with every pointer in device memory, enqueued on `stream` without synchronising.  Hit lists
 * of at most 8192 entries come back ordered; longer ones hold the right hits in unspecified order
 * (the host entry point above orders those itself).  One range search at a time per handle.
 */
int mlv_index_range_search_device(mlv_index_t h, const float *queries_dev, uint32_t nq, float radius,
                                  const uint32_t *filter_bitmap_dev, uint64_t max_hits, float *out_dists_dev,
                                  int64_t *out_rows_dev, uint64_t *out_counts_dev, void *stream);

/*
 * Order n (distance, row) pairs in device memory ascending by (distance, row): the last step of a sharded range
 * search, whose per-shard hit lists arrive concatenated (and padded with row = -1 entries, which sort last and
 * come back as distance +inf / row 2^32-1).  Rows are GLOBAL rows < 2^32; any n up to 2^31 (a bitonic network
 * over the whole list on the device).  Uses the handle's scratch: one ordering at a time per handle.
 */
int mlv_index_order_pairs_device(mlv_index_t h, const float *dists_dev, const int64_t *rows_dev, uint64_t n,
                                 float *out_dists_dev, int64_t *out_rows_dev, void *stream);

/* Copy stored rows (as stored: normalised for cosine) back to the host, [n, dim]. */
int mlv_index_get_rows(mlv_index_t h, const uint64_t *rows, uint64_t n, float *out);

int mlv_index_info(mlv_index_t h, mlv_index_info_t *info);

/*
 * Merge the per-shard results of one sharded search (SURVEY.md section 8e): `n_lists`
 * candidate lists per query, each k entries ascending, laid out [n_lists, nq, k] in device
 * memory exactly as an NCCL all-gather of every rank's (out_dists, out_rows) leaves them
 * (rank-major = ascending row_base).  Writes the global top-k per query.  Enqueued on
 * `stream` of device `device`; does not synchronise.
 */
int mlv_merge_topk(int device, const float *dists_dev, const int64_t *rows_dev, uint32_t n_lists, uint32_t nq,
                   uint32_t k, float *out_dists_dev, int64_t *out_rows_dev, int32_t *out_counts_dev, void *stream);

/*
 * Prepared filters.  A filter bitmap passed per call (filter_bitmap above) is turned into a list
 * of passing-and-live rows on the device before every search, and the scan then copies ONLY
 * those rows out of HBM (row-granular bulk copies), so a selective filter costs
 * selectivity x the bytes of an unfiltered scan.  For a predicate that is searched repeatedly,
 * mlv_filter_create uploads the bitmap and builds the list once; mlv_index_set_filter binds
 * it, and every search / range search on the handle whose own filter_bitmap argument is NULL is
 * restricted to it until mlv_index_set_filter(h, NULL).  The list follows later adds, deletes
 * and compaction automatically (rows appended after creation do not pass).  Dense filters
 * (>= 75 % passing) stream all rows and mask instead.  No reference code exists for filters
 * (README.md:123,477 only); semantics = hnswlib-0.8 knn_query(filter=...) restated in
 * oracle/exact.py (`allow`).
 */
typedef struct mlv_filter *mlv_filter_t;
int mlv_filter_create(mlv_index_t h, const uint32_t *bitmap, uint64_t n_words, mlv_filter_t *out);
/* live rows that pass (synchronises when the count is not known yet) */
int mlv_filter_passing(mlv_filter_t f, uint64_t *passing);
int mlv_filter_destroy(mlv_filter_t f);
int mlv_index_set_filter(mlv_index_t h, mlv_filter_t f);

/* The filter's bitmap as the searches see it (host, n_words uint32 words; words beyond the filter are 0). */
int mlv_filter_get_bitmap(mlv_filter_t f, uint32_t *out_words, uint64_t n_words);

/*
 * Columnar metadata (csrc/column_kernels.cuh; SURVEY.md H5 / section 8f rank 3).  The reference keeps
 * metadata as a host mapping per vector (implementations/vector.py:15) and sketches filters only as a dict of
 * equality constraints (README.md:123,477; examples/api_client.py:65-74).  An index may carry up to
 * MLV_MAX_COLUMNS int32 columns, one value per local row, in device memory beside the rows (how strings or
 * other values map to codes is the caller's business); rows never written hold MLV_COLUMN_MISSING.  Columns
 * follow compaction (values move with their rows) and are dropped by mlv_index_clear.
 * mlv_filter_create_where evaluates a conjunction of comparisons on the device into a prepared filter --
 * the same object mlv_filter_create builds from a host bitmap: a row passes when, for every predicate, its
 * value is not MLV_COLUMN_MISSING and `value op a` holds (MLV_OP_BETWEEN: a <= value <= b).  The filter is
 * the predicate's result at creation: rows appended or columns rewritten afterwards do not change it.
 * Semantics restated in oracle/exact.py::where_mask.
 */
#define MLV_MAX_COLUMNS 16u
#define MLV_MAX_PREDICATES 8u
#define MLV_COLUMN_MISSING INT32_MIN
enum mlv_pred_op { MLV_OP_EQ = 0, MLV_OP_NE = 1, MLV_OP_LT = 2, MLV_OP_LE = 3, MLV_OP_GT = 4, MLV_OP_GE = 5, MLV_OP_BETWEEN = 6 };
typedef struct mlv_predicate {
    uint32_t column;
    int32_t op;      /* enum mlv_pred_op */
    int32_t a, b;    /* b is used by MLV_OP_BETWEEN only */
} mlv_predicate_t;
/* Write values[0..n) of `column` for local rows first_row .. first_row+n-1 (host memory; rows must exist). */
int mlv_index_set_column(mlv_index_t h, uint32_t column, uint64_t first_row, const int32_t *values, uint64_t n);
/* Same, values already in device memory of this index's device. */
int mlv_index_set_column_device(mlv_index_t h, uint32_t column, uint64_t first_row, const int32_t *values_dev, uint64_t n);
/* Read a column back (MLV_COLUMN_MISSING where never written). */
int mlv_index_get_column(mlv_index_t h, uint32_t column, uint64_t first_row, uint64_t n, int32_t *out);
int mlv_filter_create_where(mlv_index_t h, const mlv_predicate_t *preds, uint32_t n_preds, mlv_filter_t *out);

/*
 * Snapshot support (SURVEY.md section 8f rank 4; the reference has no persistence, README.md:240-241 only):
 * rows exactly as stored (cosine: already normalised), tombstoned ones included, and the tombstone bitmap
 * (bit set = live).  mlv_index_import_rows appends stored-form rows WITHOUT normalising them again, so an
 * export -> import round trip reproduces the matrix bit for bit; live_words == NULL marks every row live.
 */
int mlv_index_export_rows(mlv_index_t h, uint64_t first_row, uint64_t n, float *out);
int mlv_index_export_live(mlv_index_t h, uint32_t *out_words, uint64_t n_words);
int mlv_index_import_rows(mlv_index_t h, const float *rows, uint64_t n, const uint32_t *live_words, uint64_t *first_row);

/*
 * Response path (SURVEY.md section 8f rank 2): the reference answers a search with the k stored vectors as
 * JSON number lists (rest_api.py:28-32,163), and at GPU search rates encoding k x d floats is the slowest
 * step of a request.  Writes n fp32 values as a JSON array "[v0,v1,...]" using the shortest decimal text that
 * round-trips each float32 (non-finite values as NaN / Infinity / -Infinity, like Python's json module).
 * Host-only helper, no device work.  cap >= 16 * n + 2 always suffices; *len receives the bytes written (no NUL).
 * MLV_E_INVALID when the buffer is too small.
 */
int mlv_format_f32_json(const float *values, uint64_t n, char *out, uint64_t cap, uint64_t *len);

/*
 * Fused multi-GPU exchange (csrc/exchange.cuh): the exchange step of a row-sharded search done
 * over NVLink peer memory by the search kernel itself.  One process per GPU: every rank creates
 * an exchange object, the ranks swap the 64-byte CUDA IPC handles (any transport; the Python
 * host uses torch.distributed.all_gather), connect, and attach the exchange to their shard
 * together with every rank's row_base.  mlv_index_search_exchange_device then returns the
 * GLOBAL top-k on every rank from a single kernel launch per group of <= 8 queries: local scan,
 * last CTA folds the block lists, stores its k best into every peer's buffer, waits for the
 * peers' lists (release/acquire flags at system scope) and merges.  Collective: every rank must
 * make the same sequence of calls.  Supported when mlv_index_exchange_supported(h, k) != 0
 * (k <= 55 on a 148-SM part); larger k uses the all-gather + mlv_merge_topk path.
 * A peer that does not arrive within the exchange timeout (5 s by default; MLV_EXCHANGE_TIMEOUT_MS in the
 * environment or mlv_exchange_set_timeout_ms) raises an error flag (mlv_exchange_check) instead of hanging
 * the GPU; the searches of that launch report count -1.  After a timeout the ranks' sequence numbers are out
 * of step: destroy and re-create the exchange on every rank.  At most four exchange searches may be in flight
 * per handle (mlv_index_submit refuses a fifth).
 */
typedef struct mlv_exchange *mlv_exchange_t;
#define MLV_EXCHANGE_HANDLE_BYTES 64
int mlv_exchange_create(int device, uint32_t world, uint32_t rank, mlv_exchange_t *out, unsigned char *handle_out);
/* all_handles: world * MLV_EXCHANGE_HANDLE_BYTES bytes, rank-major (this rank's own entry is ignored). */
int mlv_exchange_connect(mlv_exchange_t x, const unsigned char *all_handles);
/* MLV_OK, or MLV_E_CUDA when a peer timed out in an earlier search (synchronises the device; reported once). */
int mlv_exchange_check(mlv_exchange_t x);
/* How long a search waits inside its kernel for a peer's candidates before it gives up (default 5000 ms). */
int mlv_exchange_set_timeout_ms(mlv_exchange_t x, uint32_t ms);
int mlv_exchange_destroy(mlv_exchange_t x);
/* row_bases: world entries, the global row of every rank's local row 0.  x == NULL detaches. */
int mlv_index_attach_exchange(mlv_index_t h, mlv_exchange_t x, const uint64_t *row_bases);
int mlv_index_exchange_supported(mlv_index_t h, uint32_t k);
int mlv_index_search_exchange_device(mlv_index_t h, const float *queries_dev, uint32_t nq, uint32_t k,
                                     const uint32_t *filter_bitmap_dev, float *out_dists_dev, int64_t *out_rows_dev,
                                     int32_t *out_counts_dev, void *stream);
/* Same with host buffers (pinned staging inside, blocks until the results are back), like mlv_index_search. */
int mlv_index_search_exchange(mlv_index_t h, const float *queries, uint32_t nq, uint32_t k, const uint32_t *filter_bitmap,
                              float *out_dists, int64_t *out_rows, int32_t *out_counts);

/*
 * Sharded RANGE search (SURVEY.md section 8e: concatenation of the shards' hit lists) with the same fused
 * peer-memory exchange: one kernel per query and rank -- local range scan, the last CTA sorts the rank's hits,
 * stores them into every peer's exchange buffer, waits for the peers' lists and merges them ordered by
 * (distance, global row).  Every rank receives the complete list.  A rank's list may hold up to
 * MLV_RANGE_EXCHANGE_SLOTS / world hits; each query owns MLV_RANGE_EXCHANGE_SLOTS entries of out_dists / out_rows in
 * the device variant (max_hits entries in the host variant, which blocks until the lists are in the host buffers).
 * out_counts[q] = number of hits, or -- with bit 63 set -- a marker: MLV_RANGE_OVERFLOW | total when some rank found
 * more hits than its share (nothing was written; use mlv_index_range_search per rank and exchange the lists
 * yourself, as the Python host does through NCCL), all ones when a peer timed out.  Collective, like the kNN exchange.
 */
#define MLV_RANGE_EXCHANGE_SLOTS 8192u
#define MLV_RANGE_OVERFLOW (1ull << 63)
int mlv_index_range_exchange_supported(mlv_index_t h);
int mlv_index_range_search_exchange_device(mlv_index_t h, const float *queries_dev, uint32_t nq, float radius,
                                           const uint32_t *filter_bitmap_dev, float *out_dists_dev, int64_t *out_rows_dev,
                                           uint64_t *out_counts_dev, void *stream);
int mlv_index_range_search_exchange(mlv_index_t h, const float *queries, uint32_t nq, float radius,
                                    const uint32_t *filter_bitmap, uint64_t max_hits, float *out_dists, int64_t *out_rows,
                                    uint64_t *out_counts);

/*
 * Tracing: with MLV_NVTX=1 in the environment every entry point that touches the device (add, mark_deleted, compact,
 * search*, submit / collect, range_search*, filter_create_where) and every tensor-core tier opens an NVTX range of its
 * own name, so a profiler's timeline shows the host call around the kernels it launched.  Off by default.
 */

/*
 * Measurement hooks (bench.py / profiles): when enabled, every search records CUDA events
 * around its scan kernel on the launching stream; mlv_index_scan_time_ms returns the sum
 * of the completed scan-kernel durations since the last call and how many launches that
 * covers, and resets both.
 */
int mlv_index_set_timing(mlv_index_t h, int enabled);
int mlv_index_scan_time_ms(mlv_index_t h, double *total_ms, uint64_t *launches);
/*
 * Experimental scan tuning (profiling sweeps): key in {"cw" consumer warps per CTA, "pw" producer warps of a gathered
 * scan (0 = auto), "stage_kb"
 * ring-stage target size, "max_stages", "r" rows per warp step (0 = auto), "evict_first"
 * (-1 auto / 0 / 1), "ctas" grid size (0 = one per SM), "dynamic" (1 = work-stealing tile scheduler,
 * 0 = static round-robin), "tile_batch" tiles claimed per atomic, "fused" (1 = the last CTA does the
 * final select, 0 = separate select kernel), "gather" (-1 auto, 0 = filters stream every row and mask,
 * 1 = filters always gather; the tensor-core path compacts the passing rows accordingly), "staged_upload"
 * (1 = bulk mlv_index_add through two pinned chunks filled by worker threads, 0 = plain copy), "fast_host" (1 = single-query
 * mlv_index_search takes the one-launch latency path, 0 = always staged), "scan_half" / "scan_half_mma" / "scan_q8" (below), and the
 * tensor-core keys listed at mlv_index_gemm_stats}.  Results never depend on these.
 *
 * Shadow scan ("scan_half": -1 auto = matrices of 256 MB and more, 0 never, 1 whenever the shape allows).  A SINGLE
 * query with k <= 16 reads an fp16 shadow of the rows -- half the bytes of the HBM-bound pass; the
 * shadow (rows * 2^s, 2 bytes per element, built on first use and kept up to date like the row norms: + 50 % device
 * memory; without room for it the search is the fp32 one) is the one the tensor-core tier uses -- keeps 32 candidates by
 * approximate distance, and the last CTA re-scores them from the fp32 matrix in the scan's own arithmetic and certifies
 * the answer (rows outside the candidates are at least the 32nd approximate distance minus the fp16 error bound away).
 * An fp32 scan launch is queued right behind it and returns at once unless the certificate failed, so the fallback is
 * decided on the device and the call stays asynchronous; the results are the fp32 scan's bit for bit either way.
 * "scan_half_mma" (1 default): rows of whole 128-byte chunks are scored by tensor-core consumers (mma.sync), 0 = FMA
 * consumers.  "scan_half_gather" (1 default): a gathered (selectively filtered) single query reads the shadow's rows too
 * when they are at least 256 bytes and the row list is worth 1 GB of fp32 rows; 0 = gathered scans read the fp32 rows.  A shadow that certifies less than half of its searches sits out 64, 128, ... searches.  In an exchange
 * search every rank issues the same two launches whether or not it has a shadow to read (the ranks agree on the
 * certificate through the exchange itself), so "scan_half" must be 0 on all ranks or on none.
 * Int8 shadow ("scan_q8": -1 auto, 0 never, 1 whatever the matrix size).  With "scan_half" auto (-1), a shadow scan of a
 * full (not gathered) matrix of 256 MB and more reads an int8 shadow instead: one int8 digit per element and one scale per
 * row (+ 25 % device memory, built and kept up to date like the fp16 one), a quarter of the fp32 bytes.  It keeps 64
 * candidates and certifies them against its own error bound (q8_delta in scan_kernel.cuh); the fp32 launch behind it
 * works as above, so the results are again the fp32 scan's bit for bit.  An int8 shadow that certifies less than half of
 * its searches sits out 64, 128, ... searches while the fp16 shadow answers.  "scan_half" = 1 always reads the fp16 shadow.
 * Each rank of an exchange search picks its own shadow.
 * mlv_index_gemm_stats reports half_scan_queries / half_scan_uncertified (both shadows) and q8_scan_queries /
 * q8_scan_uncertified (the int8 one alone).
 */
int mlv_index_set_tuning(mlv_index_t h, const char *key, int value);
/*
 * Debug: after set_tuning("timeline", 1) every top-k scan records sixteen %globaltimer stamp slots (ns)
 * per CTA: 0 start, 1 first tile landed, 2 last tile consumed, 3 lists folded, 4 ticket taken, and -- for the last CTA
 * only, 0 elsewhere -- 5 final select done, 6 outputs written, 7 completion flag raised; finer ones: 8 own lists sorted,
 * 9 every warp's lists sorted, last CTA 10 past the fence, 11 threshold known, 12 survivors gathered.  Copies 16 * n_ctas
 * values of the most recent scan into `out` (synchronises the device).
 */
int mlv_index_debug_timeline(mlv_index_t h, uint64_t *out, uint32_t max_ctas, uint32_t *n_ctas);
/*
 * Tensor-core batch path (csrc/gemm_kernel.cuh): searches with nq >= 5 queries on a matrix of >= 1 GB (nq >= 9 on >= 16384 rows otherwise)
 * run as a tcgen05 GEMM that selects k + slack candidates per query, re-scores them in the
 * reference's arithmetic and certifies the result.  Tiers: a one-pass GEMM on an fp16 SHADOW of the rows
 * (kind::f16: the same 10 explicit mantissa bits as TF32 at twice the tensor rate; the shadow costs half
 * the matrix again in HBM and is built lazily -- without room for it the one-pass TF32 GEMM on the fp32 rows
 * takes its place), then the 3xTF32 GEMM for the queries the first tier could not certify; what neither
 * certifies is re-run by the exact scan, so results do not depend on the path.  set_tuning keys: "gemm"
 * (-1 auto, 0 never, 1 whenever the shape allows), "gemm_min_nq", "gemm_bn" (queries per tensor-core tile: 0 auto, 64 / 128 / 256), "gemm_passes" (0 auto, 1 one-pass TF32 tier
 * then scan, 2 fp16 tier then scan, 3 3xTF32 tier only), "gemm_wide" (which kernel runs the one-pass tiers of
 * batches wider than 128 queries: non-zero = CTA pairs, tcgen05 cta_group::2 (default); 0 = the single-tile kernel),
 * "gemm_debug" (profiling only: bit 0 = the epilogue compares nothing -- results are wrong), "gemm_predict" (1 default: the one-pass tiers' per-query thresholds are PREDICTED from the rows
 * seen so far -- a round that has seen S of N rows thresholds at its max(32, 4 k' S / N)-th best instead of its k'-th,
 * so later rounds append a fraction of the candidates; the last round verifies the prediction (k' candidates at or
 * below the tightest threshold used) and a query that fails goes to the next tier, whose thresholds are the plain
 * rule; predictions sit out 8, 16, ... batches after failing for more than an eighth of a batch; 0 = plain rule
 * everywhere).  Results never depend on "gemm_wide" / "gemm_passes" / "gemm_predict".  This call returns cumulative counters
 * and, when timing is enabled, the summed device time of the GEMM launches since the last call.
 */
typedef struct mlv_gemm_stats {
    double gemm_ms;               /* CUDA-event time of the GEMM launches since the last call */
    uint64_t gemm_launches_timed; /* how many launches gemm_ms covers */
    uint64_t searches;            /* batches that took the GEMM path (cumulative) */
    uint64_t queries;             /* queries in those batches */
    uint64_t fallback_queries;    /* of those, re-run by the scan (certificate failed / buffer overflow) */
    uint64_t rounds;              /* GEMM launches (one per round) */
    uint64_t fast_queries;        /* of `queries`, certified by the one-pass TF32 tier (no 3xTF32 work spent on them) */
    uint64_t gathered_searches;   /* of `searches`, filtered batches that multiplied a compacted copy of the passing rows */
    uint64_t half_queries;        /* of `fast_queries`, certified by the fp16-shadow tier (kind::f16 on halves of the rows) */
    uint64_t mispredicted_queries; /* queries whose predicted thresholds failed the final check ("gemm_predict"); answered by the next tier */
    uint64_t half_scan_queries;    /* single queries answered through the shadow scan ("scan_half"; not a tensor-core path, counted here for one stats call) */
    uint64_t half_scan_uncertified; /* of those, re-run by the fp32 scan launch queued behind (certificate failed / shadow overflowed) */
    uint64_t q8_scan_queries;      /* of half_scan_queries, those whose shadow scan read the int8 shadow ("scan_q8") */
    uint64_t q8_scan_uncertified;  /* of those, re-run by the fp32 scan launch queued behind */
} mlv_gemm_stats_t;
int mlv_index_gemm_stats(mlv_index_t h, mlv_gemm_stats_t *out);
/*
 * Debug / parity tests: the APPROXIMATE distances the tensor-core kernel computes (3xTF32 GEMM form, the
 * one-pass TF32 form after set_tuning("gemm_passes", 1), the fp16-shadow form after set_tuning("gemm_passes", 2); before the exact re-rank) for nq host queries against every stored row: out_approx[nq, rows],
 * NaN for tombstoned rows.  1 <= rows <= 8192, dim >= 32.
 */
int mlv_index_debug_gemm(mlv_index_t h, const float *queries, uint32_t nq, float *out_approx);
/*
 * Debug / selection tests: GEMM rounds over every stored row as a batch search runs them -- the production kernels
 * (gemm_topk_kernel or the CTA-pair kernel, each round optionally followed by refine_kernel) -- with the tier, kernel,
 * grid, initial thresholds, candidate capacity and round schedule chosen by the caller.  Returns the raw buffers:
 * out_keys[nq, cap] (slot j of query i is meaningful for j < min(out_counts[i], cap); keys are (distance, row) packed
 * as in gemm_kernel.cuh: f32_orderable(distance) << 32 | row), out_counts[nq] (uncapped: hits beyond `cap` are
 * counted, not stored), out_thr[nq] and out_flags[nq] (refine_kernel: bit 0 overflow, bit 2 starved / failed
 * prediction), and *out_pad_count, what the padding queries of the last query tile appended (0 when correct).
 * thresholds[nq] = the initial per-query thresholds (NULL = +inf; padding queries keep -inf); filter_bitmap =
 * ceil(rows / 32) words or NULL.  Any output pointer may be NULL.  rows >= 1, dim >= 32.
 */
typedef struct mlv_gemm_rounds_cfg {
    uint32_t passes;                /* 1 = one-pass TF32, 2 = fp16 shadow, 3 = 3xTF32 */
    uint32_t bn;                    /* single-tile kernel with 64 / 128 / 256 queries per tile; 0 = CTA-pair kernel (passes 1, 2) */
    uint32_t max_ctas;              /* grid limit, 0 = the grid a search launches (pairs: rounded down to an even count, >= 2) */
    uint32_t cap;                   /* candidate slots per query (>= 1; a power of two <= 8192 when kprime > 0) */
    uint32_t kprime;                /* refine_kernel keeps this many after every round; 0 = no refine (raw emission) */
    uint32_t n_rounds;              /* >= 1 */
    const uint32_t *round_end;      /* [n_rounds] row tile (128 rows) each round ends before, ascending, the last <= ceil(rows / 128) */
    const uint32_t *round_jrank;    /* [n_rounds] rank refine_kernel sets the threshold from, 1..kprime (unused when kprime is 0) */
} mlv_gemm_rounds_cfg_t;
int mlv_index_debug_gemm_rounds(mlv_index_t h, const float *queries, uint32_t nq, const float *thresholds,
                                const uint32_t *filter_bitmap, const mlv_gemm_rounds_cfg_t *cfg, uint64_t *out_keys,
                                uint32_t *out_counts, float *out_thr, uint32_t *out_flags, uint64_t *out_pad_count);
/*
 * Debug / bound tests: the APPROXIMATE distances the shadow scan's consumers compute for ONE host query against every
 * stored row (the same consumer code: FMA or tensor-core consumers, whichever "scan_half_mma" and the row length select
 * for a search), before any re-scoring: out_approx[rows], +inf for tombstoned rows.  *out_info receives what the
 * certificate and the range margin are computed from.  1 <= rows <= 8192.
 */
typedef struct mlv_half_scan_debug {
    float delta_rel;    /* bound on |approx - exact| / scale (gemm_kernel.cuh, gemm_delta_rel_f16) */
    float scale;        /* as the kernel computed it: (sqrt(max_norm2) + |q|)^2 for l2, sqrt(max_norm2) |q| for ip, 1 for cosine */
    float q_norm2;      /* |q|^2 of the prepared query, as the kernel computed it */
    float max_norm2;    /* largest |x|^2 of the rows (0 for cosine: unit rows) */
    float x_unscale;    /* 2^-s: the shadow holds halves of row * 2^s, s frozen when the shadow was built */
    float q_unscale;    /* 2^-t: the tensor-core consumers multiply halves of q * 2^t (1 for the FMA consumers) */
    uint32_t overflow;  /* rows appended after the scale froze overflowed fp16: searches do not trust the shadow */
    uint32_t consumers; /* 1 = FMA consumers, 2 = tensor-core consumers (mma.sync) */
} mlv_half_scan_debug_t;
int mlv_index_debug_half_scan(mlv_index_t h, const float *query, float *out_approx, mlv_half_scan_debug_t *out_info);
/*
 * Debug / bound tests: the same for the int8 shadow's consumers (scan_kernel_q8): out_approx[rows] (+inf for tombstoned
 * rows) and what its certificate uses.  1 <= rows <= 8192.
 */
typedef struct mlv_q8_scan_debug {
    float delta;        /* bound on |approx - exact| for every row (scan_kernel.cuh, q8_delta), as the kernel computed it */
    float q_norm2;      /* |q|^2 of the prepared query, as the kernel computed it */
    float q_scale;      /* t: the query is t (h + l / 254) + r with int8 digits h, l */
    float max_norm2;    /* largest |x|^2 of the rows (0 for cosine: unit rows) */
    float e_max;        /* E: largest bound on |x - s_x x^| over the rows */
    uint32_t ld8;       /* bytes per row of the int8 shadow */
} mlv_q8_scan_debug_t;
int mlv_index_debug_q8_scan(mlv_index_t h, const float *query, float *out_approx, mlv_q8_scan_debug_t *out_info);
/* Kernels launched by this handle since creation (scan + select + maintenance). */
int mlv_index_kernel_launches(mlv_index_t h, uint64_t *launches);

#ifdef __cplusplus
}
#endif
#endif /* MLV_INDEX_H */
