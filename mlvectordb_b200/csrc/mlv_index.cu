// mlv_index.cu -- C ABI (include/mlv_index.h) and host-side orchestration of the B200 exact-search
// index.  Everything the reference does through hnswlib inside
// src/mlvectordb/implementations/index.py (add_items :65, mark_deleted :80, knn_query :111) lands
// here.  No CPU fallback: without a CUDA device mlv_index_create fails with MLV_E_NO_DEVICE.
#include "../../include/mlv_index.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <charconv>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include "column_kernels.cuh"
#include "common.cuh"
#include "gemm_kernel.cuh"
#include "maint_kernels.cuh"
#include "scan_kernel.cuh"
#include "select_kernel.cuh"

using namespace mlv;

// ---- NVTX ranges (SURVEY.md section 5: tracing).  nvtx3 is header-only and binds to a profiler's injection library at
// run time; with MLV_NVTX unset (default) a range is one branch on a cached flag.
#include <nvtx3/nvToolsExt.h>
namespace {
struct NvtxRange {
    bool on;
    explicit NvtxRange(const char* name) : on(enabled()) {
        if (on) nvtxRangePushA(name);
    }
    ~NvtxRange() {
        if (on) nvtxRangePop();
    }
    static bool enabled() {
        static const bool v = [] {
            const char* s = getenv("MLV_NVTX");
            return s && *s && *s != '0';
        }();
        return v;
    }
};
}  // namespace

#include "host_state.inl"
#include "host_scan.inl"
#include "host_gemm.inl"
#include "host_columns.inl"


// =================================================================================== C ABI
extern "C" {

int mlv_abi_version(void) { return MLV_ABI_VERSION; }

int mlv_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

const char* mlv_status_string(int s) {
    switch (s) {
        case MLV_OK: return "ok";
        case MLV_E_INVALID: return "invalid argument";
        case MLV_E_CUDA: return "CUDA error";
        case MLV_E_NOMEM: return "out of memory";
        case MLV_E_UNSUPPORTED: return "unsupported by this build";
        case MLV_E_NO_DEVICE: return "no CUDA device (there is no CPU fallback)";
        default: return "unknown status";
    }
}

const char* mlv_last_error(mlv_index_t h) { return h ? h->err.c_str() : "null handle"; }

int mlv_index_create(uint32_t dim, int metric, uint64_t capacity_hint, int device, mlv_index_t* out) {
    if (!out) return MLV_E_INVALID;
    *out = nullptr;
    if (dim == 0 || metric < MLV_L2 || metric > MLV_COSINE) return MLV_E_INVALID;
    int ndev = mlv_device_count();
    if (ndev <= 0) return MLV_E_NO_DEVICE;
    if (device < 0 || device >= ndev) return MLV_E_INVALID;
    mlv_index* h = new (std::nothrow) mlv_index();
    if (!h) return MLV_E_NOMEM;
    h->device = device;
    h->dim = dim;
    h->ld = (dim + 3u) & ~3u;
    h->metric = metric;
    h->tune_cw = env_int("MLV_SCAN_CW", h->tune_cw);
    h->tune_stage_kb = env_int("MLV_SCAN_STAGE_KB", h->tune_stage_kb);
    h->tune_evict_first = env_int("MLV_SCAN_EVICT_FIRST", h->tune_evict_first);
    h->tune_r = env_int("MLV_SCAN_R", h->tune_r);
    h->tune_max_stages = env_int("MLV_SCAN_MAX_STAGES", h->tune_max_stages);
    h->tune_ctas = env_int("MLV_SCAN_CTAS", h->tune_ctas);
    h->tune_pw = env_int("MLV_SCAN_PW", h->tune_pw);
    h->tune_dynamic = env_int("MLV_SCAN_DYNAMIC", h->tune_dynamic);
    h->tune_tile_batch = env_int("MLV_SCAN_TILE_BATCH", h->tune_tile_batch);
    h->tune_fused = env_int("MLV_SCAN_FUSED", h->tune_fused);
    h->tune_gemm = env_int("MLV_GEMM", h->tune_gemm);
    h->tune_gemm_min_nq = env_int("MLV_GEMM_MIN_NQ", h->tune_gemm_min_nq);
    h->tune_gemm_bn = env_int("MLV_GEMM_BN", h->tune_gemm_bn);
    h->tune_gemm_passes = env_int("MLV_GEMM_PASSES", h->tune_gemm_passes);
    h->tune_gemm_wide = env_int("MLV_GEMM_WIDE", h->tune_gemm_wide);
    h->tune_gemm_debug = env_int("MLV_GEMM_DEBUG", h->tune_gemm_debug);
    h->tune_gemm_predict = env_int("MLV_GEMM_PREDICT", h->tune_gemm_predict);
    h->tune_scan_half = env_int("MLV_SCAN_HALF", h->tune_scan_half);
    h->tune_scan_half_mma = env_int("MLV_SCAN_HALF_MMA", h->tune_scan_half_mma);
    h->tune_scan_half_gather = env_int("MLV_SCAN_HALF_GATHER", h->tune_scan_half_gather);
    h->tune_scan_q8 = env_int("MLV_SCAN_Q8", h->tune_scan_q8);
    DeviceGuard g(device);
    cudaDeviceProp prop;
    cudaError_t e = g.ok ? cudaGetDeviceProperties(&prop, device) : cudaErrorInvalidDevice;
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        cudaGetLastError();
        delete h;
        return MLV_E_CUDA;
    }
    h->sm_count = prop.multiProcessorCount;
    h->smem_optin = prop.sharedMemPerBlockOptin;
    if (prop.major != 10) {
        // sm_100a cubin only: fail loudly instead of at the first launch
        cudaStreamDestroy(h->stream);
        delete h;
        return MLV_E_NO_DEVICE;
    }
    if (capacity_hint) {
        int rc = reserve_rows(h, capacity_hint);
        if (rc != MLV_OK) {
            cudaStreamDestroy(h->stream);
            delete h;
            return rc;
        }
    }
    *out = h;
    return MLV_OK;
}

int mlv_index_destroy(mlv_index_t h) {
    if (!h) return MLV_E_INVALID;
    DeviceGuard g(h->device);
    cudaStreamSynchronize(h->stream);
    if (h->d_rows) cudaFree(h->d_rows);
    if (h->d_live) cudaFree(h->d_live);
    for (DevBuf* b : {&h->d_qraw, &h->d_filter, &h->d_outd, &h->d_outr, &h->d_outc, &h->d_misc, &h->d_range, &h->d_timeline,
                      &h->d_norms, &h->d_gq, &h->d_cand, &h->d_maxn2, &h->d_sub, &h->d_gx, &h->d_rows16, &h->d_f16st, &h->d_gx16, &h->d_half_stats,
                      &h->d_rows8, &h->d_q8sx, &h->d_q8e})
        free_dev(*b);
    for (Lane& l : h->lanes)
        for (DevBuf* b : {&l.d_q, &l.d_keys0, &l.d_keys1, &l.d_sched, &l.d_flist, &l.d_fscratch, &l.d_cert}) free_dev(*b);
    drop_columns(h);
    drop_filter_pool(h);
    if (h->h_stage.p) cudaFreeHost(h->h_stage.p);
    if (h->h_range.p) cudaFreeHost(h->h_range.p);
    if (h->h_half_stats.p) cudaFreeHost(h->h_half_stats.p);
    if (h->maint_event) cudaEventDestroy(h->maint_event);
    if (h->h_upload.p) cudaFreeHost(h->h_upload.p);
    for (AsyncSlot& sl : h->slots) {
        if (sl.stream) cudaStreamSynchronize(sl.stream);
        if (sl.stage.p) cudaFreeHost(sl.stage.p);
        free_dev(sl.d_q);
        free_dev(sl.d_out);
        if (sl.done) cudaEventDestroy(sl.done);
        if (sl.stream) cudaStreamDestroy(sl.stream);
    }
    for (auto* vec : {&h->pending, &h->gemm_pending})
        for (auto& pr : *vec) {
            cudaEventDestroy(pr.first);
            cudaEventDestroy(pr.second);
        }
    for (auto ev : h->event_pool) cudaEventDestroy(ev);
    cudaStreamDestroy(h->stream);
    delete h;
    return MLV_OK;
}

int mlv_index_set_row_base(mlv_index_t h, uint64_t row_base) {
    if (!h) return MLV_E_INVALID;
    h->row_base = row_base;
    return MLV_OK;
}

int mlv_index_set_tuning(mlv_index_t h, const char* key, int value) {
    if (!h || !key) return MLV_E_INVALID;
    std::string k(key);
    if (k == "cw") h->tune_cw = value;
    else if (k == "stage_kb") h->tune_stage_kb = value;
    else if (k == "evict_first") h->tune_evict_first = value;
    else if (k == "r") h->tune_r = value;
    else if (k == "max_stages") h->tune_max_stages = value;
    else if (k == "ctas") h->tune_ctas = value;
    else if (k == "pw") h->tune_pw = value;
    else if (k == "timeline") h->tune_timeline = value;
    else if (k == "dynamic") h->tune_dynamic = value;
    else if (k == "tile_batch") h->tune_tile_batch = value;
    else if (k == "fused") h->tune_fused = value;
    else if (k == "gather") h->tune_gather = value;
    else if (k == "gemm") h->tune_gemm = value;
    else if (k == "gemm_min_nq") h->tune_gemm_min_nq = value;
    else if (k == "gemm_bn") h->tune_gemm_bn = value;
    else if (k == "staged_upload") h->tune_staged_upload = value;
    else if (k == "gemm_passes") h->tune_gemm_passes = value;
    else if (k == "fast_host") h->tune_fast_host = value;
    else if (k == "gemm_wide") h->tune_gemm_wide = value;
    else if (k == "gemm_debug") h->tune_gemm_debug = value;
    else if (k == "scan_half_mma") h->tune_scan_half_mma = value;
    else if (k == "scan_half_gather") h->tune_scan_half_gather = value;
    else if (k == "scan_half") {
        h->tune_scan_half = value;
        h->half_skip = h->half_backoff = 0;
        h->q8_skip = h->q8_backoff = 0;
    } else if (k == "scan_q8") {
        h->tune_scan_q8 = value;
        h->q8_skip = h->q8_backoff = 0;
    } else if (k == "gemm_predict") {
        h->tune_gemm_predict = value;
        h->gemm_predict_skip = h->gemm_predict_backoff = 0;
    }
    else return fail(h, MLV_E_INVALID, "unknown tuning key " + k);
    return MLV_OK;
}

// Host rows -> device matrix through two pinned staging buffers: worker threads copy chunk i+1 out of the
// caller's pageable memory while the DMA engine moves chunk i.  (A cudaMemcpy from pageable memory stages through
// the driver's own small pinned buffer on one thread: ~9 GB/s measured; PCIe 5 x16 carries ~55 GB/s.)
static int upload_rows_staged(mlv_index_t h, float* dst, const float* rows, uint64_t n) {
    const size_t row_bytes = (size_t)h->dim * 4;
    const size_t chunk_bytes = (size_t)48 << 20;
    const uint64_t chunk_rows = std::max<uint64_t>(1, chunk_bytes / row_bytes);
    int rc = ensure_host(h, h->h_upload, 2 * chunk_rows * row_bytes);
    if (rc != MLV_OK) return rc;
    cudaEvent_t done[2] = {nullptr, nullptr};
    for (auto& ev : done) {
        cudaError_t ce = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
        if (ce != cudaSuccess) {
            for (auto& made : done)
                if (made) cudaEventDestroy(made);
            return fail_cuda(h, ce, "row upload events");
        }
    }
    const unsigned n_threads = std::max(1u, std::min(8u, std::thread::hardware_concurrency() / 2));
    cudaError_t e = cudaSuccess;
    int slot = 0;
    for (uint64_t r0 = 0; r0 < n && e == cudaSuccess; r0 += chunk_rows, slot ^= 1) {
        const uint64_t nr = std::min(chunk_rows, n - r0);
        char* stage = (char*)h->h_upload.p + (size_t)slot * chunk_rows * row_bytes;
        if (r0 >= 2 * chunk_rows) e = cudaEventSynchronize(done[slot]);   // the DMA out of this buffer has finished
        if (e != cudaSuccess) break;
        const char* src = (const char*)(rows + r0 * h->dim);
        const size_t bytes = nr * row_bytes;
        if (bytes < ((size_t)4 << 20) || n_threads == 1) {
            memcpy(stage, src, bytes);
        } else {
            std::vector<std::thread> pool;
            const size_t per = (bytes / n_threads + 4095) & ~(size_t)4095;
            for (unsigned t = 0; t < n_threads; t++) {
                const size_t lo = std::min(bytes, (size_t)t * per), hi = std::min(bytes, lo + per);
                if (hi > lo) pool.emplace_back([=] { memcpy(stage + lo, src + lo, hi - lo); });
            }
            for (auto& th : pool) th.join();
        }
        e = cudaMemcpy2DAsync(dst + r0 * h->ld, (size_t)h->ld * 4, stage, row_bytes, row_bytes, nr, cudaMemcpyHostToDevice, h->stream);
        if (e == cudaSuccess) e = cudaEventRecord(done[slot], h->stream);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    for (auto& ev : done) cudaEventDestroy(ev);
    if (e != cudaSuccess) return fail_cuda(h, e, "row upload");
    return MLV_OK;
}

static int add_common(mlv_index_t h, const float* rows, uint64_t n, uint64_t* first_row, cudaMemcpyKind kind, bool normalize = true) {
    NvtxRange nvtx_range("mlv_index_add");
    if (!h || (!rows && n)) return MLV_E_INVALID;
    if (n == 0) {
        if (first_row) *first_row = h->rows;
        return MLV_OK;
    }
    DeviceGuard g(h->device);
    int rc = reserve_rows(h, h->rows + n);
    if (rc != MLV_OK) return rc;
    float* dst = h->d_rows + h->rows * h->ld;
    // pitched copy straight into the matrix; padding columns were zeroed at allocation
    if (kind == cudaMemcpyHostToDevice && n * (uint64_t)h->dim * 4 >= ((uint64_t)8 << 20) && h->tune_staged_upload) {
        if ((rc = upload_rows_staged(h, dst, rows, n)) != MLV_OK) return rc;
        return finish_append(h, n, first_row, normalize);
    }
    const uint64_t max_rows_per_copy = 1u << 20;  // cudaMemcpy2D height limits
    for (uint64_t r0 = 0; r0 < n; r0 += max_rows_per_copy) {
        const uint64_t nr = std::min(max_rows_per_copy, n - r0);
        CK(h, cudaMemcpy2DAsync(dst + r0 * h->ld, (size_t)h->ld * 4, rows + r0 * h->dim, (size_t)h->dim * 4,
                                (size_t)h->dim * 4, nr, kind, h->stream));
    }
    return finish_append(h, n, first_row, normalize);
}

int mlv_index_add(mlv_index_t h, const float* rows, uint64_t n, uint64_t* first_row) {
    return add_common(h, rows, n, first_row, cudaMemcpyHostToDevice);
}
int mlv_index_add_device(mlv_index_t h, const float* rows_dev, uint64_t n, uint64_t* first_row) {
    return add_common(h, rows_dev, n, first_row, cudaMemcpyDeviceToDevice);
}

int mlv_index_add_synthetic(mlv_index_t h, uint64_t seed, uint64_t first_gen_row, uint64_t n, int scaled,
                            uint64_t* first_row) {
    NvtxRange nvtx_range("mlv_index_add_synthetic");
    if (!h) return MLV_E_INVALID;
    if (n == 0) {
        if (first_row) *first_row = h->rows;
        return MLV_OK;
    }
    DeviceGuard g(h->device);
    int rc = reserve_rows(h, h->rows + n);
    if (rc != MLV_OK) return rc;
    const uint64_t key = splitmix64(seed), key2 = splitmix64(seed ^ 0xA5A5A5A5A5A5A5A5ull);
    const uint64_t total = n * h->ld;
    const unsigned blocks = (unsigned)std::min<uint64_t>((total + 255) / 256, (uint64_t)h->sm_count * 32);
    fill_synthetic_kernel<<<blocks, 256, 0, h->stream>>>(h->d_rows, h->rows, n, h->dim, h->ld, key, key2, first_gen_row,
                                                         scaled);
    h->launches++;
    CK(h, cudaGetLastError());
    return finish_append(h, n, first_row);
}

int mlv_index_mark_deleted(mlv_index_t h, const uint64_t* rows, uint64_t n, uint64_t* newly_deleted) {
    NvtxRange nvtx_range("mlv_index_mark_deleted");
    if (!h || (!rows && n)) return MLV_E_INVALID;
    if (newly_deleted) *newly_deleted = 0;
    if (n == 0 || h->rows == 0) return MLV_OK;
    DeviceGuard g(h->device);
    int rc = ensure_dev(h, h->d_misc, n * 8 + 8);
    if (rc != MLV_OK) return rc;
    unsigned long long* d_changed = (unsigned long long*)h->d_misc.p;
    uint64_t* d_ids = (uint64_t*)h->d_misc.p + 1;
    CK(h, cudaMemsetAsync(d_changed, 0, 8, h->stream));
    CK(h, cudaMemcpyAsync(d_ids, rows, n * 8, cudaMemcpyHostToDevice, h->stream));
    mark_deleted_kernel<<<(unsigned)std::min<uint64_t>((n + 255) / 256, 1024), 256, 0, h->stream>>>(h->d_live, d_ids, n,
                                                                                                h->rows, d_changed);
    h->launches++;
    CK(h, cudaGetLastError());
    unsigned long long changed = 0;
    CK(h, cudaMemcpyAsync(&changed, d_changed, 8, cudaMemcpyDeviceToHost, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    h->n_deleted += changed;
    if (changed) h->epoch++;
    if (newly_deleted) *newly_deleted = changed;
    return MLV_OK;
}

int mlv_index_compact(mlv_index_t h, int64_t* old_to_new, uint64_t* new_rows) {
    NvtxRange nvtx_range("mlv_index_compact");
    if (!h) return MLV_E_INVALID;
    DeviceGuard g(h->device);
    const uint64_t n = h->rows;
    if (n == 0 || h->n_deleted == 0) {
        if (old_to_new)
            for (uint64_t i = 0; i < n; i++) old_to_new[i] = (int64_t)i;
        if (new_rows) *new_rows = n;
        return MLV_OK;
    }
    const uint64_t n_words = (n + 31) / 32;
    const size_t row_bytes = (size_t)h->ld * 4;
    int rc = ensure_dev(h, h->d_misc, n_words * 8 + 8 + (old_to_new ? n * 8 : 0));
    if (rc != MLV_OK) return rc;
    uint64_t* d_total = (uint64_t*)h->d_misc.p;
    uint64_t* d_wbase = d_total + 1;
    int64_t* d_map = old_to_new ? (int64_t*)(d_wbase + n_words) : nullptr;
    float* nrows = nullptr;
    CK(h, cudaMalloc(&nrows, h->capacity * row_bytes));
    cudaError_t e = cudaMemsetAsync(nrows, 0, h->capacity * row_bytes, h->stream);
    if (e == cudaSuccess) {
        live_prefix_kernel<<<1, 1024, 0, h->stream>>>(h->d_live, n, d_wbase, d_total);
        const int wpb = 8;
        compact_rows_kernel<<<(unsigned)((n + wpb - 1) / wpb), wpb * 32, 0, h->stream>>>(
            reinterpret_cast<const float4*>(h->d_rows), reinterpret_cast<float4*>(nrows), h->d_live, d_wbase, n, h->ld / 4,
            d_map);
        h->launches += 2;
        e = cudaGetLastError();
    }
    int32_t* fresh_cols[MLV_MAX_COLUMNS] = {nullptr};
    if (e == cudaSuccess && (rc = compact_columns(h, d_wbase, n, fresh_cols)) != MLV_OK) {
        cudaStreamSynchronize(h->stream);
        cudaFree(nrows);
        return rc;
    }
    uint64_t total = 0;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&total, d_total, 8, cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess && old_to_new) e = cudaMemcpyAsync(old_to_new, d_map, n * 8, cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    if (e != cudaSuccess) {
        cudaFree(nrows);
        for (int32_t* c : fresh_cols)
            if (c) cudaFree(c);
        return fail_cuda(h, e, "compact");
    }
    cudaFree(h->d_rows);
    h->d_rows = nrows;
    adopt_compacted_columns(h, fresh_cols);
    h->rows = total;
    h->n_deleted = 0;
    h->norms_valid = 0;
    h->f16_valid = 0;
    h->q8_valid = 0;
    h->epoch++;
    h->compact_gen++;
    CK(h, cudaMemsetAsync(h->d_live, 0, h->live_words * 4, h->stream));
    if (total) {
        const uint64_t words = (total + 31) / 32;
        set_live_range_kernel<<<(unsigned)std::min<uint64_t>((words + 255) / 256, 4096), 256, 0, h->stream>>>(h->d_live, 0, total);
        h->launches++;
        CK(h, cudaGetLastError());
    }
    CK(h, cudaStreamSynchronize(h->stream));
    if (new_rows) *new_rows = total;
    return MLV_OK;
}

int mlv_index_clear(mlv_index_t h) {
    if (!h) return MLV_E_INVALID;
    DeviceGuard g(h->device);
    if (h->d_live) {
        CK(h, cudaMemsetAsync(h->d_live, 0, h->live_words * 4, h->stream));
        CK(h, cudaStreamSynchronize(h->stream));
    }
    h->rows = 0;
    h->n_deleted = 0;
    h->norms_valid = 0;
    h->f16_valid = 0;
    h->q8_valid = 0;
    h->epoch++;
    h->compact_gen++;
    drop_columns(h);
    return MLV_OK;
}

int mlv_index_search_device(mlv_index_t h, const float* queries_dev, uint32_t nq, uint32_t k,
                            const uint32_t* filter_bitmap_dev, float* out_dists_dev, int64_t* out_rows_dev,
                            int32_t* out_counts_dev, void* stream) {
    NvtxRange nvtx_range("mlv_index_search_device");
    if (!h || !queries_dev || !out_dists_dev || !out_rows_dev || !out_counts_dev || nq == 0 || k == 0) return fail(h, MLV_E_INVALID, "bad argument");
    if (k > MLV_MAX_K) return fail(h, MLV_E_UNSUPPORTED, "k exceeds MLV_MAX_K");
    DeviceGuard g(h->device);
    cudaStream_t st = (cudaStream_t)stream;  // NULL = the legacy default stream, as everywhere in CUDA
    if (h->rows == h->n_deleted) {  // nothing live (reference index.py:99-104 returns [])
        fill_empty_kernel<<<32, 256, 0, st>>>(out_dists_dev, out_rows_dev, out_counts_dev, nq, k);
        h->launches++;
        CK(h, cudaGetLastError());
        return MLV_OK;
    }
    int rc = prep_queries(h, queries_dev, nq, st);
    if (rc != MLV_OK) return rc;
    if (gemm_eligible(h, nq, k))
        return search_gemm(h, (const float*)lane_for(h, st)->d_q.p, nq, k, filter_bitmap_dev, out_dists_dev, out_rows_dev, out_counts_dev, st);
    return search_prepared(h, (const float*)lane_for(h, st)->d_q.p, nq, k, filter_bitmap_dev, out_dists_dev, out_rows_dev, out_counts_dev, st);
}

int mlv_filter_create(mlv_index_t h, const uint32_t* bitmap, uint64_t n_words, mlv_filter_t* out) {
    if (!h || !out || (!bitmap && n_words)) return MLV_E_INVALID;
    *out = nullptr;
    DeviceGuard g(h->device);
    mlv_filter* f = new_filter(h, n_words);
    if (!f) return MLV_E_NOMEM;
    int rc = ensure_dev(h, f->d_bitmap, std::max<uint64_t>(n_words, 1) * 4);
    if (rc == MLV_OK && n_words) {
        cudaError_t e = cudaMemcpyAsync(f->d_bitmap.p, bitmap, n_words * 4, cudaMemcpyHostToDevice, h->stream);
        if (e != cudaSuccess) rc = fail_cuda(h, e, "filter upload");
    }
    if (rc != MLV_OK) {
        retire_filter(h, f);
        return rc;
    }
    return finish_filter(h, f, out);
}

int mlv_filter_create_where(mlv_index_t h, const mlv_predicate_t* preds, uint32_t n_preds, mlv_filter_t* out) {
    NvtxRange nvtx_range("mlv_filter_create_where");
    if (!h || !out || (!preds && n_preds)) return MLV_E_INVALID;
    *out = nullptr;
    if (n_preds > MLV_MAX_PREDICATES) return fail(h, MLV_E_UNSUPPORTED, "more than MLV_MAX_PREDICATES predicates");
    WhereArgs args{};
    args.n = n_preds;
    for (uint32_t i = 0; i < n_preds; i++) {
        if (preds[i].column >= MLV_MAX_COLUMNS) return fail(h, MLV_E_UNSUPPORTED, "column index exceeds MLV_MAX_COLUMNS");
        if (preds[i].op < MLV_OP_EQ || preds[i].op > MLV_OP_BETWEEN) return fail(h, MLV_E_INVALID, "unknown predicate operator");
        const uint32_t c = preds[i].column;
        args.p[i].col = (const int32_t*)h->d_cols[c].p;     // never written: every row is missing
        args.p[i].col_rows = h->d_cols[c].p ? h->col_rows[c] : 0;
        where_range(preds[i].op, preds[i].a, preds[i].b, &args.p[i]);
    }
    DeviceGuard g(h->device);
    const uint64_t n_words = (h->rows + 31) / 32;
    mlv_filter* f = new_filter(h, n_words);
    if (!f) return MLV_E_NOMEM;
    int rc = ensure_dev(h, f->d_bitmap, std::max<uint64_t>(n_words, 1) * 4);
    if (rc == MLV_OK && n_words) {
        constexpr int GROUPS = 4;   // 4 x 128 rows per warp step
        const uint64_t warps = ((h->rows + 127) / 128 + GROUPS - 1) / GROUPS;
        where_kernel<GROUPS><<<grid_for(h, warps, 8), 256, 0, h->stream>>>(args, h->rows, (uint32_t*)f->d_bitmap.p);
        h->launches++;
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) rc = fail_cuda(h, e, "where_kernel");
    }
    if (rc != MLV_OK) {
        retire_filter(h, f);
        return rc;
    }
    return finish_filter(h, f, out);
}

int mlv_filter_get_bitmap(mlv_filter_t f, uint32_t* out_words, uint64_t n_words) {
    if (!f || (!out_words && n_words)) return MLV_E_INVALID;
    mlv_index* h = f->owner;
    DeviceGuard g(h->device);
    const uint64_t have = std::min(n_words, f->bitmap_words);
    if (have) CK(h, cudaMemcpyAsync(out_words, f->d_bitmap.p, have * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    for (uint64_t i = have; i < n_words; i++) out_words[i] = 0;
    return MLV_OK;
}

int mlv_index_set_column(mlv_index_t h, uint32_t column, uint64_t first_row, const int32_t* values, uint64_t n) {
    return set_column_common(h, column, first_row, values, n, cudaMemcpyHostToDevice);
}
int mlv_index_set_column_device(mlv_index_t h, uint32_t column, uint64_t first_row, const int32_t* values_dev, uint64_t n) {
    return set_column_common(h, column, first_row, values_dev, n, cudaMemcpyDeviceToDevice);
}

int mlv_index_get_column(mlv_index_t h, uint32_t column, uint64_t first_row, uint64_t n, int32_t* out) {
    if (!h || (!out && n)) return MLV_E_INVALID;
    if (column >= MLV_MAX_COLUMNS) return fail(h, MLV_E_UNSUPPORTED, "column index exceeds MLV_MAX_COLUMNS");
    if (first_row + n > h->rows || first_row + n < first_row) return fail(h, MLV_E_INVALID, "column read beyond the stored rows");
    if (n == 0) return MLV_OK;
    DeviceGuard g(h->device);
    const uint64_t have = h->d_cols[column].p ? h->col_rows[column] : 0;
    const uint64_t from_dev = first_row < have ? std::min(n, have - first_row) : 0;
    if (from_dev) {
        CK(h, cudaMemcpyAsync(out, (const int32_t*)h->d_cols[column].p + first_row, from_dev * 4, cudaMemcpyDeviceToHost, h->stream));
        CK(h, cudaStreamSynchronize(h->stream));
    }
    for (uint64_t i = from_dev; i < n; i++) out[i] = MLV_COLUMN_MISSING;
    return MLV_OK;
}

int mlv_format_f32_json(const float* values, uint64_t n, char* out, uint64_t cap, uint64_t* len) {
    if ((!values && n) || !out || !len) return MLV_E_INVALID;
    if (cap < 16 * n + 2) return MLV_E_INVALID;
    char* p = out;
    char* const end = out + cap;
    *p++ = '[';
    for (uint64_t i = 0; i < n; i++) {
        if (i) *p++ = ',';
        const float v = values[i];
        if (v == 0.0f) {   // "-0" would parse as the integer 0 and lose the sign
            const char* t = std::signbit(v) ? "-0.0" : "0.0";
            const size_t tl = strlen(t);
            memcpy(p, t, tl);
            p += tl;
        } else if (std::isfinite(v)) {
            auto r = std::to_chars(p, end, v);   // shortest text that round-trips the float32
            if (r.ec != std::errc()) return MLV_E_INVALID;
            p = r.ptr;
        } else {
            const char* t = std::isnan(v) ? "NaN" : (v > 0 ? "Infinity" : "-Infinity");
            const size_t tl = strlen(t);
            memcpy(p, t, tl);
            p += tl;
        }
    }
    *p++ = ']';
    *len = (uint64_t)(p - out);
    return MLV_OK;
}

int mlv_index_export_rows(mlv_index_t h, uint64_t first_row, uint64_t n, float* out) {
    if (!h || (!out && n)) return MLV_E_INVALID;
    if (first_row + n > h->rows || first_row + n < first_row) return fail(h, MLV_E_INVALID, "export beyond the stored rows");
    if (n == 0) return MLV_OK;
    DeviceGuard g(h->device);
    const uint64_t max_rows_per_copy = 1u << 20;
    for (uint64_t r0 = 0; r0 < n; r0 += max_rows_per_copy) {
        const uint64_t nr = std::min(max_rows_per_copy, n - r0);
        CK(h, cudaMemcpy2DAsync(out + r0 * h->dim, (size_t)h->dim * 4, h->d_rows + (first_row + r0) * h->ld, (size_t)h->ld * 4,
                                (size_t)h->dim * 4, nr, cudaMemcpyDeviceToHost, h->stream));
    }
    CK(h, cudaStreamSynchronize(h->stream));
    return MLV_OK;
}

int mlv_index_export_live(mlv_index_t h, uint32_t* out_words, uint64_t n_words) {
    if (!h || (!out_words && n_words)) return MLV_E_INVALID;
    DeviceGuard g(h->device);
    const uint64_t have = std::min(n_words, (h->rows + 31) / 32);
    if (have) CK(h, cudaMemcpyAsync(out_words, h->d_live, have * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    for (uint64_t i = have; i < n_words; i++) out_words[i] = 0;
    return MLV_OK;
}

int mlv_index_import_rows(mlv_index_t h, const float* rows, uint64_t n, const uint32_t* live_words, uint64_t* first_row) {
    if (!h || (!rows && n)) return MLV_E_INVALID;
    if (n == 0) {
        if (first_row) *first_row = h->rows;
        return MLV_OK;
    }
    uint64_t first = 0;
    int rc = add_common(h, rows, n, &first, cudaMemcpyHostToDevice, /*normalize=*/false);   // stored form: already normalised
    if (rc != MLV_OK) return rc;
    if (first_row) *first_row = first;
    if (live_words) {
        std::vector<uint64_t> gone;
        for (uint64_t i = 0; i < n; i++)
            if (!((live_words[i >> 5] >> (i & 31)) & 1u)) gone.push_back(first + i);
        if (!gone.empty()) return mlv_index_mark_deleted(h, gone.data(), gone.size(), nullptr);
    }
    return MLV_OK;
}

int mlv_filter_passing(mlv_filter_t f, uint64_t* passing) {
    if (!f || !passing) return MLV_E_INVALID;
    mlv_index* h = f->owner;
    DeviceGuard g(h->device);
    if (f->epoch != h->epoch && h->rows) {
        int rc = build_gather_list(h, f->d_list, f->d_scratch, (const uint32_t*)f->d_bitmap.p, f->bitmap_words, h->stream);
        if (rc != MLV_OK) return rc;
        f->epoch = h->epoch;
        f->counted = false;
    }
    if (!f->counted && h->rows) {
        uint64_t total = 0;
        CK(h, cudaMemcpyAsync(&total, f->d_scratch.p, 8, cudaMemcpyDeviceToHost, h->stream));
        CK(h, cudaStreamSynchronize(h->stream));
        f->passing = total;
        f->counted = true;
    }
    *passing = h->rows ? f->passing : 0;
    return MLV_OK;
}

int mlv_filter_destroy(mlv_filter_t f) {
    if (!f) return MLV_E_INVALID;
    mlv_index* h = f->owner;
    DeviceGuard g(h->device);
    if (h->bound_filter == f) h->bound_filter = nullptr;
    cudaDeviceSynchronize();   // searches in flight on other streams may still read the list
    retire_filter(h, f);
    return MLV_OK;
}

int mlv_index_set_filter(mlv_index_t h, mlv_filter_t f) {
    if (!h || (f && f->owner != h)) return MLV_E_INVALID;
    h->bound_filter = f;
    return MLV_OK;
}

int mlv_exchange_create(int device, uint32_t world, uint32_t rank, mlv_exchange_t* out, unsigned char* handle_out) {
    if (!out || !handle_out || world == 0 || world > XCHG_MAX_WORLD || rank >= world) return MLV_E_INVALID;
    *out = nullptr;
    int ndev = mlv_device_count();
    if (ndev <= 0) return MLV_E_NO_DEVICE;
    if (device < 0 || device >= ndev) return MLV_E_INVALID;
    DeviceGuard g(device);
    mlv_exchange* x = new (std::nothrow) mlv_exchange();
    if (!x) return MLV_E_NOMEM;
    x->device = device;
    x->world = world;
    x->rank = rank;
    static_assert(sizeof(cudaIpcMemHandle_t) == MLV_EXCHANGE_HANDLE_BYTES, "IPC handle size");
    cudaIpcMemHandle_t hd;
    void* buf = nullptr;
    cudaError_t e = cudaMalloc(&buf, (size_t)XCHG_WORDS * 8 + 64);
    if (e == cudaSuccess) e = cudaMemset(buf, 0, (size_t)XCHG_WORDS * 8 + 64);
    if (e == cudaSuccess) e = cudaIpcGetMemHandle(&hd, buf);
    if (e != cudaSuccess) {
        cudaGetLastError();
        if (buf) cudaFree(buf);
        delete x;
        return MLV_E_CUDA;
    }
    x->bufs[rank] = (uint64_t*)buf;
    x->d_error = (int*)((uint64_t*)buf + XCHG_WORDS);  // behind the slots, in the same allocation
    memcpy(handle_out, &hd, sizeof(hd));
    x->connected = world == 1;
    const int ms = env_int("MLV_EXCHANGE_TIMEOUT_MS", 0);
    if (ms > 0) x->timeout_ns = (unsigned long long)ms * 1000000ull;
    *out = x;
    return MLV_OK;
}

int mlv_exchange_set_timeout_ms(mlv_exchange_t x, uint32_t ms) {
    if (!x || ms == 0) return MLV_E_INVALID;
    x->timeout_ns = (unsigned long long)ms * 1000000ull;
    return MLV_OK;
}

int mlv_exchange_connect(mlv_exchange_t x, const unsigned char* all_handles) {
    if (!x || !all_handles) return MLV_E_INVALID;
    DeviceGuard g(x->device);
    for (uint32_t r = 0; r < x->world; r++) {
        if (r == x->rank || x->bufs[r]) continue;
        cudaIpcMemHandle_t hd;
        memcpy(&hd, all_handles + (size_t)r * sizeof(hd), sizeof(hd));
        void* ptr = nullptr;
        if (cudaIpcOpenMemHandle(&ptr, hd, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
            cudaGetLastError();
            return MLV_E_CUDA;
        }
        x->bufs[r] = (uint64_t*)ptr;
    }
    x->connected = true;
    return MLV_OK;
}

int mlv_exchange_check(mlv_exchange_t x) {
    if (!x) return MLV_E_INVALID;
    DeviceGuard g(x->device);
    int err = 0;
    if (cudaMemcpy(&err, x->d_error, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess) {
        cudaGetLastError();
        return MLV_E_CUDA;
    }
    if (err) cudaMemset(x->d_error, 0, sizeof(int));   // reported once; the ranks' sequence numbers are out of step now:
    return err ? MLV_E_CUDA : MLV_OK;                   // the caller re-creates the exchange (collective) before searching on
}

int mlv_exchange_destroy(mlv_exchange_t x) {
    if (!x) return MLV_E_INVALID;
    DeviceGuard g(x->device);
    cudaDeviceSynchronize();
    for (uint32_t r = 0; r < x->world; r++) {
        if (!x->bufs[r]) continue;
        if (r == x->rank)
            cudaFree(x->bufs[r]);
        else
            cudaIpcCloseMemHandle(x->bufs[r]);
    }
    cudaGetLastError();
    delete x;
    return MLV_OK;
}

int mlv_index_attach_exchange(mlv_index_t h, mlv_exchange_t x, const uint64_t* row_bases) {
    if (!h) return MLV_E_INVALID;
    if (!x) {
        h->xchg = nullptr;
        return MLV_OK;
    }
    if (!row_bases || x->device != h->device) return fail(h, MLV_E_INVALID, "exchange lives on another device");
    h->xchg = x;
    for (uint32_t i = 0; i < x->world; i++) h->xchg_row_bases[i] = row_bases[i];
    return MLV_OK;
}

int mlv_index_exchange_supported(mlv_index_t h, uint32_t k) {
    if (!h) return 0;
    return exchange_ok(h, k) ? 1 : 0;
}

int mlv_index_search_exchange_device(mlv_index_t h, const float* queries_dev, uint32_t nq, uint32_t k,
                                     const uint32_t* filter_bitmap_dev, float* out_dists_dev, int64_t* out_rows_dev,
                                     int32_t* out_counts_dev, void* stream) {
    NvtxRange nvtx_range("mlv_index_search_exchange_device");
    if (!h || !queries_dev || !out_dists_dev || !out_rows_dev || !out_counts_dev || nq == 0 || k == 0) return fail(h, MLV_E_INVALID, "bad argument");
    if (!exchange_ok(h, k)) return fail(h, MLV_E_UNSUPPORTED, "no connected exchange, or k too large for the fused exchange");
    DeviceGuard g(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (h->rows == h->n_deleted) {
        // nothing to scan here, but the peers wait for this rank's (empty) lists: same launch grouping
        // as a scanning rank (groups of up to XCHG_MAX_NQ queries, one sequence number each)
        ExchangeView x{};
        fill_exchange(h, x);
        ScanCfg c;
        int rc0 = choose_cfg(h, nq, k, false, &c);  // same query grouping as a scanning rank
        if (rc0 != MLV_OK) return rc0;
        const bool pair = half_scan_proto(h, nq, k);   // the peers' searches take two launches: so does this rank's part
        Lane* ln = lane_for(h, st);
        if (pair && (rc0 = ensure_dev(h, ln->d_cert, 4)) != MLV_OK) return rc0;
        for (uint32_t g0 = 0; g0 < nq; g0 += c.NQ) {
            const uint32_t n = std::min<uint32_t>(c.NQ, nq - g0);
            x.seq = ++h->xseq;
            exchange_only_kernel<<<1, 256, 0, st>>>(x, n, k, out_dists_dev + (size_t)g0 * k, out_rows_dev + (size_t)g0 * k,
                                                   out_counts_dev + g0, pair ? (uint32_t*)ln->d_cert.p : nullptr, nullptr);
            h->launches++;
            if (pair) {
                x.seq = ++h->xseq;
                exchange_only_kernel<<<1, 256, 0, st>>>(x, n, k, out_dists_dev + (size_t)g0 * k, out_rows_dev + (size_t)g0 * k,
                                                       out_counts_dev + g0, nullptr, (const uint32_t*)ln->d_cert.p);
                h->launches++;
            }
        }
        CK(h, cudaGetLastError());
        return MLV_OK;
    }
    int rc = prep_queries(h, queries_dev, nq, st);
    if (rc != MLV_OK) return rc;
    return search_prepared(h, (const float*)lane_for(h, st)->d_q.p, nq, k, filter_bitmap_dev, out_dists_dev, out_rows_dev, out_counts_dev, st, true);
}

static int search_host_common(mlv_index_t h, const float* queries, uint32_t nq, uint32_t k, const uint32_t* filter_bitmap,
                              float* out_dists, int64_t* out_rows, int32_t* out_counts, bool exchange) {
    NvtxRange nvtx_range("mlv_index_search");
    if (!h || !queries || !out_dists || !out_rows || !out_counts || nq == 0 || k == 0) return fail(h, MLV_E_INVALID, "bad argument");
    if (k > MLV_MAX_K) return fail(h, MLV_E_UNSUPPORTED, "k exceeds MLV_MAX_K");
    DeviceGuard g(h->device);
    const size_t qbytes = (size_t)nq * h->dim * 4;
    const size_t nk = (size_t)nq * k;
    const size_t out_bytes = nk * 4 + nk * 8 + (size_t)nq * 4;
    int rc;
    if ((rc = ensure_host(h, h->h_stage, std::max(qbytes, out_bytes) + 192)) != MLV_OK) return rc;
    if (nq == 1 && !filter_bitmap && h->rows != h->n_deleted && h->dim <= SCAN_INLINE_MAX_DIM && h->tune_fast_host &&
        (!exchange || exchange_ok(h, k))) {
        // Batch-1 latency path (BASELINE configs[0]): ONE launch and nothing else.  The raw query travels in the kernel
        // parameters (padded / normalised inside the kernel), the fused tail writes the final top-k straight into this
        // pinned, device-mapped staging block and raises a flag there; the host polls the flag (a short spin, then a
        // stream synchronise for long scans) -- no H2D copy, no preparation launch, no D2H copy.
        char* hs = (char*)h->h_stage.p;
        unsigned int* flag = (unsigned int*)(hs + ((out_bytes + 63) & ~(size_t)63));
        // single GPU: the results come as tagged 16-byte records at the start of the block (k records + a count record);
        // an exchange search writes the three arrays and raises the flag behind a system fence
        uint4* recs = (uint4*)hs;
        const bool tagged = !exchange && (size_t)(k + 1) * 16 <= h->h_stage.bytes - 128;
        bool took = false;
        FastArgs fa;
        fa.inline_q = queries;
        fa.done_flag = flag;
        fa.done_value = ++h->flag_seq ? h->flag_seq : ++h->flag_seq;
        fa.took_fast = &took;
        fa.tagged_out = tagged ? recs : nullptr;
        *(volatile unsigned int*)flag = 0;   // nothing of this handle is in flight on the block: every call waits for its own results
        if (tagged) ((volatile unsigned int*)&recs[k])[1] = 0;
        rc = search_prepared(h, nullptr, 1, k, nullptr, (float*)(hs + nk * 8), (int64_t*)hs, (int32_t*)(hs + nk * 12), h->stream, exchange, &fa);
        if (rc != MLV_OK) return rc;
        if (took && tagged) {
            volatile unsigned int* vr = (volatile unsigned int*)recs;
            const unsigned int tag = fa.done_value;
            bool seen = false;
            for (int spin = 0; spin < 200000 && !seen; spin++) seen = vr[4 * k + 1] == tag;   // ~100-200 us of polling
            if (!seen) CK(h, cudaStreamSynchronize(h->stream));
            std::atomic_thread_fence(std::memory_order_acquire);
            const uint32_t count = std::min<uint32_t>((uint32_t)vr[4 * k], k);
            for (uint32_t i = 0; i < k; i++) {
                if (i < count) {
                    // a record is complete once it carries the tag (one 16-byte store); after the stream synchronise all are
                    for (int spin = 0; vr[4 * i + 1] != tag && spin < 100000000; spin++) {
                    }
                    std::atomic_thread_fence(std::memory_order_acquire);
                    uint32_t bits = vr[4 * i];
                    memcpy(&out_dists[i], &bits, 4);
                    out_rows[i] = (int64_t)(((uint64_t)vr[4 * i + 3] << 32) | vr[4 * i + 2]);
                } else {
                    out_dists[i] = std::numeric_limits<float>::infinity();
                    out_rows[i] = -1;
                }
            }
            out_counts[0] = (int32_t)count;
            return MLV_OK;
        }
        if (took) {
            volatile unsigned int* vf = flag;
            bool seen = false;
            for (int spin = 0; spin < 200000 && !seen; spin++) seen = *vf == fa.done_value;   // ~100-200 us of polling
            if (!seen) CK(h, cudaStreamSynchronize(h->stream));
            std::atomic_thread_fence(std::memory_order_acquire);
            memcpy(out_rows, hs, nk * 8);
            memcpy(out_dists, hs + nk * 8, nk * 4);
            memcpy(out_counts, hs + nk * 12, (size_t)nq * 4);
            return MLV_OK;
        }
    }
    if ((rc = ensure_dev(h, h->d_qraw, qbytes)) != MLV_OK) return rc;
    // one device block for the results (rows | dists | counts): a single copy brings them back
    if ((rc = ensure_dev(h, h->d_outr, out_bytes)) != MLV_OK) return rc;
    int64_t* d_rows_out = (int64_t*)h->d_outr.p;
    float* d_dists_out = (float*)((char*)h->d_outr.p + nk * 8);
    int32_t* d_counts_out = (int32_t*)((char*)h->d_outr.p + nk * 12);
    const uint32_t* filter_dev;
    if ((rc = upload_filter_bitmap(h, filter_bitmap, &filter_dev)) != MLV_OK) return rc;
    memcpy(h->h_stage.p, queries, qbytes);
    CK(h, cudaMemcpyAsync(h->d_qraw.p, h->h_stage.p, qbytes, cudaMemcpyHostToDevice, h->stream));
    if (exchange)
        rc = mlv_index_search_exchange_device(h, (const float*)h->d_qraw.p, nq, k, filter_dev, d_dists_out, d_rows_out,
                                              d_counts_out, h->stream);
    else
        rc = mlv_index_search_device(h, (const float*)h->d_qraw.p, nq, k, filter_dev, d_dists_out, d_rows_out, d_counts_out,
                                     h->stream);
    if (rc != MLV_OK) return rc;
    char* hs = (char*)h->h_stage.p;
    CK(h, cudaMemcpyAsync(hs, h->d_outr.p, out_bytes, cudaMemcpyDeviceToHost, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    memcpy(out_rows, hs, nk * 8);
    memcpy(out_dists, hs + nk * 8, nk * 4);
    memcpy(out_counts, hs + nk * 12, (size_t)nq * 4);
    return MLV_OK;
}

int mlv_index_search(mlv_index_t h, const float* queries, uint32_t nq, uint32_t k, const uint32_t* filter_bitmap,
                     float* out_dists, int64_t* out_rows, int32_t* out_counts) {
    return search_host_common(h, queries, nq, k, filter_bitmap, out_dists, out_rows, out_counts, false);
}

int mlv_index_search_exchange(mlv_index_t h, const float* queries, uint32_t nq, uint32_t k, const uint32_t* filter_bitmap,
                              float* out_dists, int64_t* out_rows, int32_t* out_counts) {
    return search_host_common(h, queries, nq, k, filter_bitmap, out_dists, out_rows, out_counts, true);
}

// argument checks both grouped entries share (pointers and nq aside)
static int grouped_args(mlv_index_t h, uint32_t k, uint32_t column) {
    if (k == 0 || column >= MLV_MAX_COLUMNS) return fail(h, MLV_E_INVALID, "bad argument");
    if (k > MLV_MAX_GROUP_K) return fail(h, MLV_E_UNSUPPORTED, "k exceeds MLV_MAX_GROUP_K");
    if (!h->tune_dynamic || !h->tune_fused)
        return fail(h, MLV_E_UNSUPPORTED, "grouped search finishes in the fused last-CTA tail: set_tuning \"dynamic\" and \"fused\" must be 1");
    return MLV_OK;
}

int mlv_index_search_grouped_device(mlv_index_t h, const float* queries_dev, uint32_t nq, uint32_t k, uint32_t column,
                                    const uint32_t* filter_bitmap_dev, float* out_dists_dev, int64_t* out_rows_dev,
                                    int32_t* out_groups_dev, int32_t* out_counts_dev, void* stream) {
    NvtxRange nvtx_range("mlv_index_search_grouped_device");
    if (!h || !queries_dev || !out_dists_dev || !out_rows_dev || !out_groups_dev || !out_counts_dev || nq == 0) return fail(h, MLV_E_INVALID, "bad argument");
    int rc = grouped_args(h, k, column);
    if (rc != MLV_OK) return rc;
    DeviceGuard g(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (h->rows == h->n_deleted || !h->d_cols[column].p) {   // nothing live, or a column never written: no groups
        fill_empty_kernel<<<32, 256, 0, st>>>(out_dists_dev, out_rows_dev, out_counts_dev, nq, k);
        fill_i32_kernel<<<32, 256, 0, st>>>(out_groups_dev, (uint64_t)nq * k, COLUMN_MISSING);
        h->launches += 2;
        CK(h, cudaGetLastError());
        return MLV_OK;
    }
    if ((rc = prep_queries(h, queries_dev, nq, st)) != MLV_OK) return rc;
    return search_grouped(h, (const float*)lane_for(h, st)->d_q.p, nq, k, (const int32_t*)h->d_cols[column].p, h->col_rows[column],
                          filter_bitmap_dev, out_dists_dev, out_rows_dev, out_groups_dev, out_counts_dev, st);
}

int mlv_index_search_grouped(mlv_index_t h, const float* queries, uint32_t nq, uint32_t k, uint32_t column, const uint32_t* filter_bitmap,
                             float* out_dists, int64_t* out_rows, int32_t* out_groups, int32_t* out_counts) {
    NvtxRange nvtx_range("mlv_index_search_grouped");
    if (!h || !queries || !out_dists || !out_rows || !out_groups || !out_counts || nq == 0) return fail(h, MLV_E_INVALID, "bad argument");
    int rc = grouped_args(h, k, column);
    if (rc != MLV_OK) return rc;
    DeviceGuard g(h->device);
    const size_t qbytes = (size_t)nq * h->dim * 4;
    const size_t nk = (size_t)nq * k;
    const size_t out_bytes = nk * 16 + (size_t)nq * 4;   // rows | dists | groups | counts: one copy brings them back
    if ((rc = ensure_host(h, h->h_stage, std::max(qbytes, out_bytes))) != MLV_OK) return rc;
    if ((rc = ensure_dev(h, h->d_qraw, qbytes)) != MLV_OK) return rc;
    if ((rc = ensure_dev(h, h->d_outr, out_bytes)) != MLV_OK) return rc;
    char* d = (char*)h->d_outr.p;
    const uint32_t* filter_dev;
    if ((rc = upload_filter_bitmap(h, filter_bitmap, &filter_dev)) != MLV_OK) return rc;
    memcpy(h->h_stage.p, queries, qbytes);
    CK(h, cudaMemcpyAsync(h->d_qraw.p, h->h_stage.p, qbytes, cudaMemcpyHostToDevice, h->stream));
    rc = mlv_index_search_grouped_device(h, (const float*)h->d_qraw.p, nq, k, column, filter_dev, (float*)(d + nk * 8), (int64_t*)d,
                                         (int32_t*)(d + nk * 12), (int32_t*)(d + nk * 16), h->stream);
    if (rc != MLV_OK) return rc;
    char* hs = (char*)h->h_stage.p;
    CK(h, cudaMemcpyAsync(hs, d, out_bytes, cudaMemcpyDeviceToHost, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    memcpy(out_rows, hs, nk * 8);
    memcpy(out_dists, hs + nk * 8, nk * 4);
    memcpy(out_groups, hs + nk * 12, nk * 4);
    memcpy(out_counts, hs + nk * 16, (size_t)nq * 4);
    return MLV_OK;
}

int mlv_index_submit(mlv_index_t h, const float* queries, uint32_t nq, uint32_t k, int exchange, uint32_t* ticket) {
    NvtxRange nvtx_range("mlv_index_submit");
    if (!h || !queries || !ticket || nq == 0 || k == 0) return fail(h, MLV_E_INVALID, "bad argument");
    if (k > MLV_MAX_K) return fail(h, MLV_E_UNSUPPORTED, "k exceeds MLV_MAX_K");
    DeviceGuard g(h->device);
    int idx = -1;
    for (int i = 0; i < MLV_ASYNC_SLOTS; i++) {
        const int c = (int)((h->next_slot + i) % MLV_ASYNC_SLOTS);
        if (!h->slots[c].busy) {
            idx = c;
            break;
        }
    }
    if (idx < 0) return fail(h, MLV_E_UNSUPPORTED, "all asynchronous search slots are in flight: collect one first");
    if (exchange) {
        int flying = 0;
        for (const AsyncSlot& s2 : h->slots) flying += s2.busy && s2.exchange;
        if (flying >= XCHG_MAX_IN_FLIGHT) return fail(h, MLV_E_UNSUPPORTED, "four exchange searches are in flight already: collect one first");
    }
    h->next_slot = (uint32_t)(idx + 1) % MLV_ASYNC_SLOTS;
    AsyncSlot& sl = h->slots[idx];
    if (!sl.stream) {
        CK(h, cudaStreamCreateWithFlags(&sl.stream, cudaStreamNonBlocking));
        CK(h, cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming));
    }
    const size_t qbytes = (size_t)nq * h->dim * 4;
    const size_t nk = (size_t)nq * k;
    const size_t out_bytes = nk * 12 + (size_t)nq * 4;
    int rc;
    if ((rc = ensure_host(h, sl.stage, std::max(qbytes, out_bytes))) != MLV_OK) return rc;
    if ((rc = ensure_dev(h, sl.d_q, qbytes)) != MLV_OK) return rc;
    if ((rc = ensure_dev(h, sl.d_out, out_bytes)) != MLV_OK) return rc;
    memcpy(sl.stage.p, queries, qbytes);
    CK(h, cudaMemcpyAsync(sl.d_q.p, sl.stage.p, qbytes, cudaMemcpyHostToDevice, sl.stream));
    int64_t* d_rows_out = (int64_t*)sl.d_out.p;
    float* d_dists_out = (float*)((char*)sl.d_out.p + nk * 8);
    int32_t* d_counts_out = (int32_t*)((char*)sl.d_out.p + nk * 12);
    if (exchange)
        rc = mlv_index_search_exchange_device(h, (const float*)sl.d_q.p, nq, k, nullptr, d_dists_out, d_rows_out, d_counts_out, sl.stream);
    else
        rc = mlv_index_search_device(h, (const float*)sl.d_q.p, nq, k, nullptr, d_dists_out, d_rows_out, d_counts_out, sl.stream);
    if (rc != MLV_OK) return rc;
    // the queries have left the staging buffer (stream order), so the results may land in it
    CK(h, cudaMemcpyAsync(sl.stage.p, sl.d_out.p, out_bytes, cudaMemcpyDeviceToHost, sl.stream));
    CK(h, cudaEventRecord(sl.done, sl.stream));
    sl.nq = nq;
    sl.k = k;
    sl.busy = true;
    sl.exchange = exchange != 0;
    *ticket = (uint32_t)idx;
    return MLV_OK;
}

int mlv_index_collect(mlv_index_t h, uint32_t ticket, float* out_dists, int64_t* out_rows, int32_t* out_counts) {
    NvtxRange nvtx_range("mlv_index_collect");
    if (!h || ticket >= (uint32_t)MLV_ASYNC_SLOTS || !out_dists || !out_rows || !out_counts) return fail(h, MLV_E_INVALID, "bad argument");
    AsyncSlot& sl = h->slots[ticket];
    if (!sl.busy) return fail(h, MLV_E_INVALID, "no search in flight under this ticket");
    DeviceGuard g(h->device);
    sl.busy = false;
    CK(h, cudaEventSynchronize(sl.done));
    const size_t nk = (size_t)sl.nq * sl.k;
    const char* hs = (const char*)sl.stage.p;
    memcpy(out_rows, hs, nk * 8);
    memcpy(out_dists, hs + nk * 8, nk * 4);
    memcpy(out_counts, hs + nk * 12, (size_t)sl.nq * 4);
    return MLV_OK;
}

int mlv_index_range_search_device(mlv_index_t h, const float* queries_dev, uint32_t nq, float radius,
                                  const uint32_t* filter_bitmap_dev, uint64_t max_hits, float* out_dists_dev,
                                  int64_t* out_rows_dev, uint64_t* out_counts_dev, void* stream) {
    NvtxRange nvtx_range("mlv_index_range_search_device");
    if (!h || !queries_dev || !out_counts_dev || nq == 0 || (max_hits && (!out_dists_dev || !out_rows_dev))) return fail(h, MLV_E_INVALID, "bad argument");
    DeviceGuard g(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (h->rows == h->n_deleted) {
        CK(h, cudaMemsetAsync(out_counts_dev, 0, (size_t)nq * 8, st));
        return MLV_OK;
    }
    RangeScan r;
    int rc;
    if ((rc = range_setup(h, queries_dev, nq, filter_bitmap_dev, std::max<uint64_t>(max_hits, 1), st, &r)) != MLV_OK) return rc;
    r.p.radius = radius;
    r.p.max_hits = max_hits;
    for (uint32_t q = 0; q < nq; q++) CK(h, launch_range(h, r, q, st));
    CK(h, raise_smem_once<range_finish_kernel>(SELECT_MAX_P * 8));
    range_finish_kernel<<<nq, SELECT_THREADS, (size_t)SELECT_MAX_P * 8, st>>>(r.d_keys, r.d_counts, r.slots, max_hits, h->row_base,
                                                                            out_dists_dev, out_rows_dev, (unsigned long long*)out_counts_dev);
    h->launches++;
    CK(h, cudaGetLastError());
    return MLV_OK;
}

int mlv_index_range_search(mlv_index_t h, const float* queries, uint32_t nq, float radius, const uint32_t* filter_bitmap,
                           uint64_t max_hits, float* out_dists, int64_t* out_rows, uint64_t* out_counts) {
    NvtxRange nvtx_range("mlv_index_range_search");
    if (!h || !queries || !out_counts || nq == 0 || (max_hits && (!out_dists || !out_rows))) return fail(h, MLV_E_INVALID, "bad argument");
    DeviceGuard g(h->device);
    for (uint32_t q = 0; q < nq; q++) out_counts[q] = 0;
    if (h->rows == h->n_deleted) return MLV_OK;
    const size_t qbytes = (size_t)nq * h->dim * 4;
    const size_t nh = (size_t)nq * max_hits;
    int rc;
    if ((rc = ensure_dev(h, h->d_qraw, qbytes)) != MLV_OK) return rc;
    if ((rc = ensure_dev(h, h->d_outd, std::max<size_t>(nh, 1) * 4)) != MLV_OK) return rc;
    if ((rc = ensure_dev(h, h->d_outr, std::max<size_t>(nh, 1) * 8)) != MLV_OK) return rc;
    if ((rc = ensure_dev(h, h->d_outc, (size_t)nq * 8)) != MLV_OK) return rc;
    const uint32_t* filter_dev;
    if ((rc = upload_filter_bitmap(h, filter_bitmap, &filter_dev)) != MLV_OK) return rc;
    CK(h, cudaMemcpyAsync(h->d_qraw.p, queries, qbytes, cudaMemcpyHostToDevice, h->stream));
    rc = mlv_index_range_search_device(h, (const float*)h->d_qraw.p, nq, radius, filter_dev, max_hits, (float*)h->d_outd.p,
                                       (int64_t*)h->d_outr.p, (uint64_t*)h->d_outc.p, h->stream);
    if (rc != MLV_OK) return rc;
    CK(h, cudaMemcpyAsync(out_counts, h->d_outc.p, (size_t)nq * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
    h->range_hits_hint = 0;   // how wide this caller's radii are (range_setup: the shadow range scan re-scores every hit)
    for (uint32_t q = 0; q < nq; q++) h->range_hits_hint = std::max<uint64_t>(h->range_hits_hint, out_counts[q]);
    const uint64_t slots = std::max<uint64_t>(max_hits, 1);
    for (uint32_t q = 0; q < nq; q++) {
        const uint64_t got = std::min<uint64_t>(out_counts[q], max_hits);
        if (!got) continue;
        float* dd = (float*)h->d_outd.p + (size_t)q * max_hits;
        int64_t* dr = (int64_t*)h->d_outr.p + (size_t)q * max_hits;
        if (got > SELECT_MAX_P) {  // more hits than one CTA sorts: global bitonic network over the query's keys
            uint64_t* keys = (uint64_t*)h->d_range.p + nq + (size_t)q * slots;
            if ((rc = sort_big_device(h, keys, got, dd, dr, h->stream)) != MLV_OK) return rc;
        }
        CK(h, cudaMemcpyAsync(out_dists + (size_t)q * max_hits, dd, got * 4, cudaMemcpyDeviceToHost, h->stream));
        CK(h, cudaMemcpyAsync(out_rows + (size_t)q * max_hits, dr, got * 8, cudaMemcpyDeviceToHost, h->stream));
    }
    CK(h, cudaStreamSynchronize(h->stream));
    return MLV_OK;
}

static_assert(MLV_RANGE_EXCHANGE_SLOTS == XCHG_SLOT_KEYS, "header and exchange.cuh disagree on the range slot size");
static_assert(MLV_RANGE_OVERFLOW == RANGE_OVERFLOW, "header and exchange.cuh disagree on the overflow marker");

int mlv_index_range_exchange_supported(mlv_index_t h) {
    if (!h) return 0;
    return (h->xchg && h->xchg->connected && h->tune_dynamic && h->tune_fused) ? 1 : 0;
}

int mlv_index_range_search_exchange_device(mlv_index_t h, const float* queries_dev, uint32_t nq, float radius,
                                           const uint32_t* filter_bitmap_dev, float* out_dists_dev, int64_t* out_rows_dev,
                                           uint64_t* out_counts_dev, void* stream) {
    NvtxRange nvtx_range("mlv_index_range_search_exchange_device");
    if (!h || !queries_dev || !out_dists_dev || !out_rows_dev || !out_counts_dev || nq == 0) return fail(h, MLV_E_INVALID, "bad argument");
    if (!mlv_index_range_exchange_supported(h)) return fail(h, MLV_E_UNSUPPORTED, "no connected exchange");
    DeviceGuard g(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    ExchangeView x{};
    fill_exchange(h, x);
    const uint64_t share = XCHG_SLOT_KEYS / x.world;
    int rc;
    if (h->rows == h->n_deleted) {   // nothing to scan here, but the peers wait for this rank's (empty) list
        CK(h, raise_smem_once<range_exchange_only_kernel>(XCHG_SLOT_KEYS * 8));
        for (uint32_t q = 0; q < nq; q++) {
            x.seq = ++h->xseq;
            range_exchange_only_kernel<<<1, 256, (size_t)XCHG_SLOT_KEYS * 8, st>>>(x, out_dists_dev + (size_t)q * XCHG_SLOT_KEYS,
                                                                               out_rows_dev + (size_t)q * XCHG_SLOT_KEYS,
                                                                               (unsigned long long*)out_counts_dev + q);
            h->launches++;
        }
        CK(h, cudaGetLastError());
        return MLV_OK;
    }
    RangeScan r;
    if ((rc = range_setup(h, queries_dev, nq, filter_bitmap_dev, share, st, &r)) != MLV_OK) return rc;
    r.c.smem = std::max(r.c.smem, (size_t)XCHG_SLOT_KEYS * 8);   // the last CTA sorts / merges up to a slot's worth of keys
    r.p.radius = radius;
    r.p.max_hits = share;
    r.p.fused = 1;
    r.p.xchg = x;
    for (uint32_t q = 0; q < nq; q++) {
        r.p.out_dists = out_dists_dev + (size_t)q * XCHG_SLOT_KEYS;
        r.p.out_rows = out_rows_dev + (size_t)q * XCHG_SLOT_KEYS;
        r.p.range_out_count = (unsigned long long*)out_counts_dev + q;
        r.p.xchg.seq = ++h->xseq;
        CK(h, launch_range(h, r, q, st));
    }
    return MLV_OK;
}

int mlv_index_range_search_exchange(mlv_index_t h, const float* queries, uint32_t nq, float radius, const uint32_t* filter_bitmap,
                                    uint64_t max_hits, float* out_dists, int64_t* out_rows, uint64_t* out_counts) {
    if (!h || !queries || !out_counts || nq == 0 || (max_hits && (!out_dists || !out_rows))) return fail(h, MLV_E_INVALID, "bad argument");
    if (!mlv_index_range_exchange_supported(h)) return fail(h, MLV_E_UNSUPPORTED, "no connected exchange");
    DeviceGuard g(h->device);
    const size_t qbytes = (size_t)nq * h->dim * 4;
    // results land in pinned, device-mapped host memory straight from the kernel (a hit list is ~1 KB; the slot-sized
    // device buffers would cost a 100 KB copy per query): counts | dists | rows
    const size_t per_q = (size_t)XCHG_SLOT_KEYS * 12;
    int rc;
    if ((rc = ensure_host(h, h->h_range, (size_t)nq * (8 + per_q) + qbytes)) != MLV_OK) return rc;
    if ((rc = ensure_dev(h, h->d_qraw, qbytes)) != MLV_OK) return rc;
    uint64_t* hc = (uint64_t*)h->h_range.p;
    float* hd = (float*)(hc + nq);
    int64_t* hr = (int64_t*)((char*)hd + (size_t)nq * XCHG_SLOT_KEYS * 4);
    char* hq = (char*)hr + (size_t)nq * XCHG_SLOT_KEYS * 8;
    const uint32_t* filter_dev;
    if ((rc = upload_filter_bitmap(h, filter_bitmap, &filter_dev)) != MLV_OK) return rc;
    memcpy(hq, queries, qbytes);
    CK(h, cudaMemcpyAsync(h->d_qraw.p, hq, qbytes, cudaMemcpyHostToDevice, h->stream));
    rc = mlv_index_range_search_exchange_device(h, (const float*)h->d_qraw.p, nq, radius, filter_dev, hd, hr, hc, h->stream);
    if (rc != MLV_OK) return rc;
    CK(h, cudaStreamSynchronize(h->stream));
    for (uint32_t q = 0; q < nq; q++) {
        out_counts[q] = hc[q];
        if (hc[q] & (1ull << 63)) continue;   // overflow / timeout marker: no hits were written
        const uint64_t got = std::min<uint64_t>(hc[q], max_hits);
        memcpy(out_dists + (size_t)q * max_hits, hd + (size_t)q * XCHG_SLOT_KEYS, got * 4);
        memcpy(out_rows + (size_t)q * max_hits, hr + (size_t)q * XCHG_SLOT_KEYS, got * 8);
    }
    return MLV_OK;
}

int mlv_index_order_pairs_device(mlv_index_t h, const float* dists_dev, const int64_t* rows_dev, uint64_t n, float* out_dists_dev,
                                 int64_t* out_rows_dev, void* stream) {
    if (!h || (n && (!dists_dev || !rows_dev || !out_dists_dev || !out_rows_dev))) return fail(h, MLV_E_INVALID, "bad argument");
    if (n == 0) return MLV_OK;
    DeviceGuard g(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    uint64_t P = SELECT_MAX_P;
    while (P < n) P <<= 1;
    if (P > (1ull << 31)) return fail(h, MLV_E_UNSUPPORTED, "too many pairs to order");
    int rc = ensure_dev(h, h->d_misc, P * 8);
    if (rc != MLV_OK) return rc;
    uint64_t* a = (uint64_t*)h->d_misc.p;
    encode_pairs_kernel<<<(unsigned)std::min<uint64_t>((P + 255) / 256, 2048), 256, 0, st>>>(dists_dev, rows_dev, n, P, a);
    if ((rc = sort_keys_device(h, a, P, st)) != MLV_OK) return rc;
    decode_keys_kernel<<<(unsigned)std::min<uint64_t>((n + 255) / 256, 1024), 256, 0, st>>>(a, n, 0, out_dists_dev, out_rows_dev);
    h->launches += 2;
    CK(h, cudaGetLastError());
    return MLV_OK;
}

int mlv_index_get_rows(mlv_index_t h, const uint64_t* rows, uint64_t n, float* out) {
    if (!h || (n && (!rows || !out))) return MLV_E_INVALID;
    DeviceGuard g(h->device);
    for (uint64_t i = 0; i < n; i++) {
        if (rows[i] >= h->rows) return fail(h, MLV_E_INVALID, "row out of range");
        CK(h, cudaMemcpyAsync(out + i * h->dim, h->d_rows + rows[i] * h->ld, (size_t)h->dim * 4, cudaMemcpyDeviceToHost, h->stream));
    }
    CK(h, cudaStreamSynchronize(h->stream));
    return MLV_OK;
}

int mlv_index_info(mlv_index_t h, mlv_index_info_t* info) {
    if (!h || !info) return MLV_E_INVALID;
    info->rows = h->rows;
    info->live = h->rows - h->n_deleted;
    info->capacity = h->capacity;
    info->row_base = h->row_base;
    size_t b = (size_t)h->capacity * h->ld * 4 + (size_t)h->live_words * 4;
    for (const DevBuf* d : {&h->d_qraw, &h->d_filter, &h->d_outd, &h->d_outr, &h->d_outc, &h->d_misc, &h->d_range, &h->d_norms,
                            &h->d_gq, &h->d_cand, &h->d_maxn2, &h->d_rows16, &h->d_gx, &h->d_gx16,
                            &h->d_rows8, &h->d_q8sx})
        b += d->bytes;
    for (const Lane& l : h->lanes)
        for (const DevBuf* d : {&l.d_q, &l.d_keys0, &l.d_keys1, &l.d_sched, &l.d_flist, &l.d_fscratch}) b += d->bytes;
    for (const DevBuf& c : h->d_cols) b += c.bytes;
    for (const FilterBufs& fb : h->filter_pool) b += fb.bitmap.bytes + fb.list.bytes + fb.scratch.bytes;
    info->device_bytes = b;
    info->dim = h->dim;
    info->ld = h->ld;
    info->metric = h->metric;
    info->device = h->device;
    return MLV_OK;
}

int mlv_merge_topk(int device, const float* dists_dev, const int64_t* rows_dev, uint32_t n_lists, uint32_t nq, uint32_t k,
                   float* out_dists_dev, int64_t* out_rows_dev, int32_t* out_counts_dev, void* stream) {
    if (!dists_dev || !rows_dev || !out_dists_dev || !out_rows_dev || !out_counts_dev || !n_lists || !nq || !k) return MLV_E_INVALID;
    if ((uint64_t)n_lists * k > SELECT_MAX_P) return MLV_E_UNSUPPORTED;
    DeviceGuard g(device);
    if (!g.ok) return MLV_E_CUDA;
    if (raise_smem_once<merge_pairs_kernel>(SELECT_MAX_P * 8) != cudaSuccess) return MLV_E_CUDA;
    MergePairsParams p{};
    p.dists = dists_dev;
    p.rows = rows_dev;
    p.n_lists = n_lists;
    p.nq = nq;
    p.k = k;
    p.P = pow2_ceil(std::max<uint32_t>(n_lists * k, 2));
    p.out_dists = out_dists_dev;
    p.out_rows = out_rows_dev;
    p.out_counts = out_counts_dev;
    const int threads = (int)std::min<uint32_t>(SELECT_THREADS, std::max<uint32_t>(p.P / 2, 32));
    merge_pairs_kernel<<<nq, threads, (size_t)p.P * 8, (cudaStream_t)stream>>>(p);
    return cudaGetLastError() == cudaSuccess ? MLV_OK : MLV_E_CUDA;
}

int mlv_index_set_timing(mlv_index_t h, int enabled) {
    if (!h) return MLV_E_INVALID;
    h->timing = enabled != 0;
    return MLV_OK;
}

int mlv_index_scan_time_ms(mlv_index_t h, double* total_ms, uint64_t* launches) {
    if (!h) return MLV_E_INVALID;
    DeviceGuard g(h->device);
    double total = 0;
    uint64_t n = 0;
    for (auto& pr : h->pending) {
        CK(h, cudaEventSynchronize(pr.second));
        float ms = 0;
        CK(h, cudaEventElapsedTime(&ms, pr.first, pr.second));
        total += ms;
        n++;
        h->event_pool.push_back(pr.first);
        h->event_pool.push_back(pr.second);
    }
    h->pending.clear();
    if (total_ms) *total_ms = total;
    if (launches) *launches = n;
    return MLV_OK;
}

int mlv_index_gemm_stats(mlv_index_t h, mlv_gemm_stats_t* out) {
    if (!h || !out) return MLV_E_INVALID;
    DeviceGuard g(h->device);
    double total = 0;
    uint64_t n = 0;
    for (auto& pr : h->gemm_pending) {
        CK(h, cudaEventSynchronize(pr.second));
        float ms = 0;
        CK(h, cudaEventElapsedTime(&ms, pr.first, pr.second));
        total += ms;
        n++;
        h->event_pool.push_back(pr.first);
        h->event_pool.push_back(pr.second);
    }
    h->gemm_pending.clear();
    out->gemm_ms = total;
    out->gemm_launches_timed = n;
    out->searches = h->gemm_searches;
    out->queries = h->gemm_queries;
    out->fallback_queries = h->gemm_fallback_queries;
    out->fast_queries = h->gemm_fast_queries;
    out->half_queries = h->gemm_half_queries;
    out->mispredicted_queries = h->gemm_mispredicted_queries;
    out->half_scan_queries = out->half_scan_uncertified = 0;
    out->q8_scan_queries = out->q8_scan_uncertified = 0;
    if (h->d_half_stats.p) {   // counters the shadow-scan kernels keep on the device: {fp16 q, uncertified, int8 q, uncertified}
        uint32_t hs[4] = {0, 0, 0, 0};
        CK(h, cudaDeviceSynchronize());
        CK(h, cudaMemcpy(hs, h->d_half_stats.p, 16, cudaMemcpyDeviceToHost));
        out->half_scan_queries = (uint64_t)hs[0] + hs[2];
        out->half_scan_uncertified = (uint64_t)hs[1] + hs[3];
        out->q8_scan_queries = hs[2];
        out->q8_scan_uncertified = hs[3];
    }
    out->gathered_searches = h->gemm_gathered_searches;
    out->rounds = h->gemm_rounds;
    return MLV_OK;
}

int mlv_index_debug_gemm(mlv_index_t h, const float* queries, uint32_t nq, float* out_approx) {
    if (!h || !queries || !out_approx || nq == 0) return fail(h, MLV_E_INVALID, "bad argument");
    if (h->rows == 0 || h->rows > SELECT_MAX_P || h->ld < (uint32_t)GEMM_BK) return fail(h, MLV_E_UNSUPPORTED, "debug_gemm needs 1..8192 rows and dim >= 32");
    DeviceGuard g(h->device);
    // one round over every row tile at threshold +inf: each live row is a candidate of every query
    const uint32_t tiles = (uint32_t)((h->rows + GEMM_BM - 1) / GEMM_BM);
    mlv_gemm_rounds_cfg_t c{};
    const GemmTierRule tiers = gemm_tier_rule(h, 1);   // the distances of the last tier a batch runs before the scan
    c.passes = tiers.one_pass && !tiers.second ? (tiers.half ? (uint32_t)GEMM_TIER_F16 : 1u) : 3u;
    c.bn = gemm_tile_width(h, nq);
    c.cap = pow2_ceil((uint32_t)h->rows);
    c.n_rounds = 1;
    c.round_end = &tiles;
    std::vector<uint64_t> keys((size_t)nq * c.cap);
    std::vector<uint32_t> counts(nq);
    int rc;
    if ((rc = gemm_rounds_debug(h, queries, nq, nullptr, nullptr, c, keys.data(), counts.data(), nullptr, nullptr, nullptr)) != MLV_OK) return rc;
    for (size_t i = 0; i < (size_t)nq * h->rows; i++) out_approx[i] = std::numeric_limits<float>::quiet_NaN();
    for (uint32_t q = 0; q < nq; q++)
        for (uint32_t i = 0; i < std::min(counts[q], c.cap); i++) {
            const uint64_t key = keys[(size_t)q * c.cap + i];
            if (key_row(key) < h->rows) out_approx[(size_t)q * h->rows + key_row(key)] = key_dist(key);
        }
    return MLV_OK;
}

int mlv_index_debug_gemm_rounds(mlv_index_t h, const float* queries, uint32_t nq, const float* thresholds, const uint32_t* filter_bitmap,
                                const mlv_gemm_rounds_cfg_t* cfg, uint64_t* out_keys, uint32_t* out_counts, float* out_thr,
                                uint32_t* out_flags, uint64_t* out_pad_count) {
    if (!h) return MLV_E_INVALID;
    if (!cfg) return fail(h, MLV_E_INVALID, "bad argument");
    DeviceGuard g(h->device);
    return gemm_rounds_debug(h, queries, nq, thresholds, filter_bitmap, *cfg, out_keys, out_counts, out_thr, out_flags, out_pad_count);
}

int mlv_index_debug_half_scan(mlv_index_t h, const float* query, float* out_approx, mlv_half_scan_debug_t* out_info) {
    if (!h) return MLV_E_INVALID;
    if (!query || !out_approx || !out_info) return fail(h, MLV_E_INVALID, "bad argument");
    if (h->rows == 0 || h->rows > SELECT_MAX_P || h->ld < 8) return fail(h, MLV_E_UNSUPPORTED, "debug_half_scan needs 1..8192 rows and dim >= 8");
    DeviceGuard g(h->device);
    cudaStream_t st = h->stream;
    Lane* ln = lane_for(h, st);
    int rc;
    if ((rc = ensure_dev(h, h->d_qraw, (size_t)h->dim * 4)) != MLV_OK) return rc;
    CK(h, cudaMemcpyAsync(h->d_qraw.p, query, (size_t)h->dim * 4, cudaMemcpyHostToDevice, st));
    if ((rc = prep_queries(h, (const float*)h->d_qraw.p, 1, st)) != MLV_OK) return rc;
    bool usable = false;
    if ((rc = ensure_shadow(h, st, &usable)) != MLV_OK) return rc;
    if (!usable) return fail(h, MLV_E_NOMEM, "no room for the fp16 shadow");
    ScanCfg c;
    if ((rc = choose_cfg(h, 1, 1, true, &c, false, shadow_consumers(h))) != MLV_OK) return rc;
    ScanParams p = shadow_params(h, c, FilterPlan{}, ln, 1);
    p.sched = nullptr;
    p.queries = reinterpret_cast<const float4*>(ln->d_q.p);
    p.nq_valid = 1;
    // [rows] approximate distances (+inf where the kernel stores nothing) | |q|^2, 2^-s 2^-t, scale
    const size_t n_out = (size_t)h->rows + 3;
    if ((rc = ensure_dev(h, h->d_outd, n_out * 4)) != MLV_OK) return rc;
    std::vector<float> out(n_out, std::numeric_limits<float>::infinity());
    CK(h, cudaMemcpyAsync(h->d_outd.p, out.data(), n_out * 4, cudaMemcpyHostToDevice, st));
    p.out_dists = (float*)h->d_outd.p;
    CK(h, h->metric == MLV_L2 ? launch_scan_half_debug_m<METRIC_L2>(p, c, st) : launch_scan_half_debug_m<METRIC_IP>(p, c, st));
    h->launches++;
    uint32_t f16st[3] = {0, 0, 0}, maxn2 = 0;
    CK(h, cudaMemcpyAsync(out.data(), h->d_outd.p, n_out * 4, cudaMemcpyDeviceToHost, st));
    CK(h, cudaMemcpyAsync(f16st, h->d_f16st.p, 12, cudaMemcpyDeviceToHost, st));
    if (h->metric != MLV_COSINE) CK(h, cudaMemcpyAsync(&maxn2, h->d_maxn2.p, 4, cudaMemcpyDeviceToHost, st));
    CK(h, cudaStreamSynchronize(st));
    memcpy(out_approx, out.data(), (size_t)h->rows * 4);
    float x_unscale;
    memcpy(&x_unscale, &f16st[0], 4);
    memcpy(&out_info->max_norm2, &maxn2, 4);
    out_info->delta_rel = p.delta_rel;
    out_info->q_norm2 = out[h->rows];
    out_info->x_unscale = x_unscale;
    out_info->q_unscale = out[h->rows + 1] / x_unscale;   // powers of two: exact
    out_info->scale = out[h->rows + 2];
    out_info->overflow = f16st[2];
    out_info->consumers = c.R == 16 ? 2u : 1u;   // rows too long for two 16-row stages take the FMA consumers
    return MLV_OK;
}

int mlv_index_debug_q8_scan(mlv_index_t h, const float* query, float* out_approx, mlv_q8_scan_debug_t* out_info) {
    if (!h) return MLV_E_INVALID;
    if (!query || !out_approx || !out_info) return fail(h, MLV_E_INVALID, "bad argument");
    if (h->rows == 0 || h->rows > SELECT_MAX_P) return fail(h, MLV_E_UNSUPPORTED, "debug_q8_scan needs 1..8192 rows");
    DeviceGuard g(h->device);
    cudaStream_t st = h->stream;
    Lane* ln = lane_for(h, st);
    int rc;
    if ((rc = ensure_dev(h, h->d_qraw, (size_t)h->dim * 4)) != MLV_OK) return rc;
    CK(h, cudaMemcpyAsync(h->d_qraw.p, query, (size_t)h->dim * 4, cudaMemcpyHostToDevice, st));
    if ((rc = prep_queries(h, (const float*)h->d_qraw.p, 1, st)) != MLV_OK) return rc;
    bool usable = false;
    if ((rc = ensure_shadow(h, st, &usable, true)) != MLV_OK) return rc;
    if (!usable) return fail(h, MLV_E_NOMEM, "no room for the int8 shadow");
    ScanCfg c;
    if ((rc = choose_cfg(h, 1, 1, true, &c, false, SHADOW_Q8)) != MLV_OK) return rc;
    ScanParams p = q8_params(h, c, FilterPlan{}, ln, 1);
    p.sched = nullptr;
    p.queries = reinterpret_cast<const float4*>(ln->d_q.p);
    p.nq_valid = 1;
    // [rows] approximate distances (+inf where the kernel stores nothing) | |q|^2, t, delta
    const size_t n_out = (size_t)h->rows + 3;
    if ((rc = ensure_dev(h, h->d_outd, n_out * 4)) != MLV_OK) return rc;
    std::vector<float> out(n_out, std::numeric_limits<float>::infinity());
    CK(h, cudaMemcpyAsync(h->d_outd.p, out.data(), n_out * 4, cudaMemcpyHostToDevice, st));
    p.out_dists = (float*)h->d_outd.p;
    CK(h, h->metric == MLV_L2 ? launch_smem<scan_kernel_q8_debug<METRIC_L2>>(c, st, p) : launch_smem<scan_kernel_q8_debug<METRIC_IP>>(c, st, p));
    h->launches++;
    uint32_t e_bits = 0, maxn2 = 0;
    CK(h, cudaMemcpyAsync(out.data(), h->d_outd.p, n_out * 4, cudaMemcpyDeviceToHost, st));
    CK(h, cudaMemcpyAsync(&e_bits, h->d_q8e.p, 4, cudaMemcpyDeviceToHost, st));
    if (h->metric != MLV_COSINE) CK(h, cudaMemcpyAsync(&maxn2, h->d_maxn2.p, 4, cudaMemcpyDeviceToHost, st));
    CK(h, cudaStreamSynchronize(st));
    memcpy(out_approx, out.data(), (size_t)h->rows * 4);
    out_info->q_norm2 = out[h->rows];
    out_info->q_scale = out[h->rows + 1];
    out_info->delta = out[h->rows + 2];
    memcpy(&out_info->max_norm2, &maxn2, 4);
    memcpy(&out_info->e_max, &e_bits, 4);
    out_info->ld8 = q8_ld(h);
    return MLV_OK;
}

int mlv_index_debug_timeline(mlv_index_t h, uint64_t* out, uint32_t max_ctas, uint32_t* n_ctas) {
    if (!h || !out || !n_ctas) return MLV_E_INVALID;
    DeviceGuard g(h->device);
    const uint32_t n = std::min<uint32_t>(max_ctas, (uint32_t)h->last_grid);
    *n_ctas = n;
    if (n == 0 || !h->d_timeline.p) return MLV_OK;
    CK(h, cudaDeviceSynchronize());
    CK(h, cudaMemcpy(out, h->d_timeline.p, (size_t)n * 16 * 8, cudaMemcpyDeviceToHost));
    return MLV_OK;
}

int mlv_index_kernel_launches(mlv_index_t h, uint64_t* launches) {
    if (!h || !launches) return MLV_E_INVALID;
    *launches = h->launches;
    return MLV_OK;
}

}  // extern "C"
