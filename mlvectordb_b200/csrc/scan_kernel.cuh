// scan_kernel.cuh -- the hot path: one streaming pass over a namespace's row matrix with the
// metric transform, tombstone/filter mask and top-k (or radius) selection fused in.
//
// Replaces hnswlib's knn_query (reference src/mlvectordb/implementations/index.py:111) by an
// exact scan.  HBM-bound: every stored row is read once; distances never touch HBM.
//
// Structure (sm_100a):
//   * persistent grid, one CTA per SM; CTA = CW consumer warps + 1 producer warp
//   * the producer lane streams tiles of T consecutive rows into an S-stage shared-memory ring
//     with 1-D bulk async copies (cp.async.bulk -> SASS UBLKCP) completing on mbarriers;
//     consumers never issue a global load for row data
//   * a consumer warp scores R rows x NQ queries per step: lane l accumulates the float4
//     columns l, l+32, ... of each row against the queries held in shared memory, then a
//     transposing butterfly leaves each (row, query) sum in one lane class
//   * per-warp, per-query candidate lists in shared memory (k <= 32: k unsorted entries with replace-
//     the-maximum insertion; larger k: an append buffer compacted by a warp-local bitonic sort) guarded by a
//     register threshold: a row costs one compare unless it beats the current k-th best
//   * at the end the block folds its warps' lists into one list per query and writes
//     k keys per (query, block); select_kernel.cuh merges the blocks' lists.
#pragma once
#include "common.cuh"
#include "exchange.cuh"

namespace mlv {

constexpr int METRIC_L2 = 0;
constexpr int METRIC_IP = 1;  // cosine == ip over rows/queries normalised at add/query time
constexpr int SCAN_MAX_CW = 16;                          // consumer warps per CTA (runtime, <= this)
constexpr int SCAN_MAX_PW = 4;                           // producer warps (1 unless gathering short rows)
constexpr int SCAN_MAX_THREADS = (SCAN_MAX_CW + SCAN_MAX_PW) * 32;  // 640 -> ptxas may use up to 102 registers
// 4 and 8 queries per pass hold R * NQ accumulators + NQ query float4s per lane: 102 registers spilled (r01: 44 - 116
// bytes per thread).  Those instantiations run at most 8 consumer warps (each does 4 - 8x the math per row byte, so
// half the warps still cover the shared-memory latency) and may use 170 registers.
constexpr int SCAN_WIDE_CW = 8;
template <int NQ>
constexpr int scan_max_threads() {
    return NQ >= 2 ? (SCAN_WIDE_CW + SCAN_MAX_PW) * 32 : SCAN_MAX_THREADS;   // (NQ = 2, R = 4 spilled 16 bytes at 96 registers)
}

// scale exponent for a largest magnitude `m`: 2^s with m * 2^s in [2^13, 2^14) (fp16 overflows at 2^16: two bits of
// headroom for rows appended after the scale was frozen); m == 0 or not finite -> 0
__host__ __device__ inline int f16_scale_exp(float m) {
    if (!(m > 0.f) || m > 3.0e38f) return 0;
    int ex;
    frexpf(m, &ex);   // m = f * 2^ex, f in [0.5, 1)
    int s = 14 - ex;
    return s < -100 ? -100 : (s > 100 ? 100 : s);
}

// Int8 shadow (scan_kernel_q8): a row is x = s_x x^ + e with int8 digits x^, one scale per row and |e|_2 <= e_x <= E (every
// e_x rounded up, E their maximum); the query is q = t (h + l / 254) + r with int8 digits h, l.  The consumers compute
// a = s_x t (D_h + D_l / 254) from the exact int32 sums D_h = x^.h and D_l = x^.l, and
//   x.q - s_x t (D_h + D_l / 254) = e.q + s_x x^.r,   |e.q| <= E |q|,   |s_x x^.r| <= (|x|max + E) |r|   (Cauchy-Schwarz).
// fp32 rounding: converting the sums, the product with fl(1/254), their sum and the two scale products are <= 12 roundings
// of terms each at most A tq (A = |x|max + E, tq = t (|h| + |l| / 254)): <= 2^-20 A tq.  The exact side is the fp32 scan's
// own sum, off by <= d 2^-23 |x||q|, and 1 - dot on either side adds <= 2^-24 (1 + |dot|); all of it is below
// (d + 64) 2^-22 A (|q| + tq) + 2^-22.  l2: a = |x|^2 + |q|^2 - 2 dot with fp32 norms (each off by <= d 2^-23 of itself)
// against the fp32 sum of (x - q)^2 (off by <= (d + 2) 2^-23 (|x| + |q|)^2): twice the dot terms plus
// (d + 64) 2^-21 (A + |q| + tq)^2.  Returns the bound on |a - exact| for every row (absolute, not relative to a scale).
__host__ __device__ inline float q8_delta(bool l2, uint32_t d, float xmax, float E, float qn, float rn, float tq) {
    const float A = xmax + E;
    const float dot = E * qn + A * rn;
    const float eps = (float)(d + 64) * 2.384185791015625e-7f;
    if (!l2) return dot + eps * A * (qn + tq) + 2.384185791015625e-7f;
    const float w = A + qn + tq;
    return 2.0f * dot + 2.0f * eps * w * w;
}

constexpr uint32_t SCAN_FUSED_MAX_KEYS = 8192;  // keys the last CTA folds (gridDim.x * k): k <= 55 on 148 SMs
// ... the int8 shadow scan's k' = 64 on 148 SMs (9472 keys): 128 KB of candidate slots in its idle ring
constexpr uint32_t SCAN_FUSED_MAX_KEYS_Q8 = 16384;

struct ScanParams {
    const float4* rows;     // [n_rows, ld4]
    uint32_t n_rows;
    uint32_t ld4;           // float4 per row
    uint32_t tile_rows;     // T (multiple of R)
    uint32_t n_tiles;
    uint32_t stages;        // S (a multiple of producer_warps)
    uint32_t producer_warps;  // PW: producer warp w owns the stages s with s % PW == w
    uint32_t stage_f4;      // float4 per ring stage (= T * ld4)
    const float4* queries;  // [nq_valid, ld4] device, zero padded, normalised for cosine
    uint32_t nq_valid;      // <= NQ
    uint32_t k;
    // slots of one (warp, query) candidate list.  == k: unsorted list, replace-the-maximum insertion
    // (k <= 32, one shared-memory pass per insertion).  > k (a power of two >= 2k): append buffer --
    // rows that beat the threshold are appended, and when fewer than 32 free slots remain the warp
    // sorts the buffer, keeps the k best and tightens the threshold (amortised O(log^2) per insertion
    // instead of two passes over k entries).
    uint32_t list_cap;
    const uint32_t* live;    // tombstone bitmap (bit set = live) or nullptr when nothing is deleted
    const uint32_t* filter;  // caller's filter bitmap or nullptr
    // gather mode (selective filters): `gather` lists the passing-and-live rows ascending; n_rows is
    // the length of the list, tiles are runs of list positions and the producer copies row by row,
    // so only passing rows are read from HBM.  live / filter are already folded into the list.
    const uint32_t* gather;
    const uint32_t* n_rows_dev;  // gather mode: length of the list, produced on the device just before (no host sync)
    uint64_t* out_keys;      // top-k mode: [nq_valid][gridDim.x][k]
    float radius;            // range mode
    unsigned long long* range_counts;  // [nq_valid]
    uint64_t* range_keys;              // [nq_valid][max_hits]
    unsigned long long max_hits;
    int evict_first;
    unsigned long long* timeline;  // debug: 4 globaltimer stamps per CTA (nullptr = off)
    // dynamic tile scheduler: sched[0] = next batch of `tile_batch` tiles, sched[1] = CTAs finished.
    // Both are zero between launches (the last CTA to finish resets them).  nullptr = static round-robin.
    uint32_t* sched;
    uint32_t tile_batch;
    // fused final select (top-k mode, needs sched, gridDim.x * k <= SCAN_FUSED_MAX_KEYS): the last
    // CTA to finish folds the grid's lists into the final ascending top-k instead of select_kernel
    int fused;
    uint32_t fused_cap;   // slots of the last CTA's candidate array: power of two >= max(gridDim.x * k, 1024)
    float* out_dists;     // [nq_valid][k]
    int64_t* out_rows;    // [nq_valid][k]
    int32_t* out_counts;  // [nq_valid]
    uint64_t row_base;
    // fused multi-GPU exchange (world > 1): the last CTA also writes its k best into every peer's
    // exchange buffer over NVLink, waits for the peers' lists and merges -- no NCCL call, no extra launch
    ExchangeView xchg;
    // range mode with `fused`: the last CTA sorts this rank's hits and runs the range exchange (exchange.cuh);
    // out_dists / out_rows then hold XCHG_SLOT_KEYS slots and range_out_count the merged count
    unsigned long long* range_out_count;
    // inline-query launches (scan_kernel_iq): the raw query rides in the kernel parameters; the CTA pads it and, for
    // cosine, normalises it exactly like prep_queries_kernel -- no H2D copy, no preparation launch
    uint32_t dim;
    int normalize;
    // completion flag in mapped pinned host memory (nullptr = none): written with done_value after the final outputs,
    // so the host can poll instead of synchronising the stream
    unsigned int* done_flag;
    unsigned int done_value;
    // Tagged result records in mapped pinned host memory (nullptr = off; single GPU, one query): record i < k is
    // {distance bits, tag, row low, row high}, record k is {count, tag, 0, 0}, each ONE 16-byte store.  A record is
    // valid for the host as soon as it carries this launch's tag, so no system fence and no flag are needed (the
    // fence + flag cost 4 us of a 27 us launch on a 10k-row namespace).
    uint4* tagged_out;
    unsigned int tag;
    // ---- shadow scan (HALF instantiations: one query, k' = k <= 64 candidates, fused tail) -------------------------
    // rows / ld4 / stage_f4 describe the fp16 SHADOW of the matrix (halves of row * 2^s, ld4 = 16-byte units per row):
    // the pass reads half the bytes and selects k' candidates by approximate distance; the last CTA re-scores them from
    // the fp32 matrix in the scan's own arithmetic, keeps the best k_out and certifies the answer exactly like the
    // tensor-core tiers (gemm_kernel.cuh): rows outside the candidates have a >= a_k', hence exact distance >= a_k' - delta.
    const float4* rows_exact;        // the fp32 matrix [n_rows, ld4_exact]
    uint32_t ld4_exact;              // float4 per fp32 row == float4 per prepared query
    uint32_t k_out;                  // neighbours returned (<= k)
    const uint32_t* half_state;      // {2^-s as float bits, s, overflow flag} (f16_freeze_scale_kernel)
    const float* row_norms;          // |x|^2 per row (l2)
    const uint32_t* max_norm2_bits;  // max |x|^2 (nullptr: unit rows)
    float delta_rel;                 // bound on |a - exact| / scale
    int cosine;                      // unit rows and queries: scale 1
    // *cert (device word) = 1 when some query of this launch is not certified (on any rank of an exchange search), else
    // 0: the fp32 launch queued right behind this one carries run_if = cert and returns at once when it reads 0 -- the
    // fallback is decided on the device, no host synchronisation
    uint32_t* cert;
    const uint32_t* run_if;
    // device counters {fp16 queries, not certified, int8 queries, not certified}
    uint32_t* half_stats;
    // mapped pinned mirror {fp16 queries, not certified, overflow flag, -, int8 queries, not certified} (plain stores)
    volatile uint32_t* half_stats_host;
    // ---- int8 shadow (HALF = 3, scan_kernel_q8): rows / ld4 / stage_f4 describe int8 digits (ld4 = 16-byte units per row),
    // k' = k <= 64 candidates; the error bound is q8_delta (above), computed per query in the kernel
    const float* q8_scale;           // s_x per row
    const uint32_t* q8_e_bits;       // E = max e_x (float bits)
};

constexpr uint32_t SCAN_INLINE_MAX_DIM = 2048;   // floats of a query carried in the kernel parameters (8 KB)
struct InlineQuery {
    float v[SCAN_INLINE_MAX_DIM];
};

struct StageMeta {
    uint32_t row0;
    int32_t n_rows;  // < 0: no more tiles
};

template <int METRIC>
__device__ __forceinline__ float accum4(float acc, const float4& x, const float4& q) {
    if (METRIC == METRIC_L2) {
        float t0 = x.x - q.x, t1 = x.y - q.y, t2 = x.z - q.z, t3 = x.w - q.w;
        acc = fmaf(t0, t0, acc);
        acc = fmaf(t1, t1, acc);
        acc = fmaf(t2, t2, acc);
        acc = fmaf(t3, t3, acc);
    } else {
        acc = fmaf(x.x, q.x, acc);
        acc = fmaf(x.y, q.y, acc);
        acc = fmaf(x.z, q.z, acc);
        acc = fmaf(x.w, q.w, acc);
    }
    return acc;
}

// Sum v[i] over the 32 lanes for every i in [0, V).  Afterwards the lane holds the total of
// index lane_slot<V>(lane); V - 1 + (5 - log2 V) shuffles instead of 5 V.
template <int V>
__device__ __forceinline__ float transpose_reduce(float (&v)[V], int lane) {
    int off = 16;
#pragma unroll
    for (int h = V / 2; h >= 1; h >>= 1) {
        const bool upper = (lane & off) != 0;
#pragma unroll
        for (int i = 0; i < h; i++) {
            float send = upper ? v[i] : v[i + h];
            float keep = upper ? v[i + h] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
        }
        off >>= 1;
    }
    float s = v[0];
    for (; off >= 1; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
    return s;
}
template <int V>
__device__ __forceinline__ int lane_slot(int lane) {
    int idx = 0, off = 16;
#pragma unroll
    for (int h = V / 2; h >= 1; h >>= 1) {
        if (lane & off) idx += h;
        off >>= 1;
    }
    return idx;
}

// Replace the maximum (== oldthr) of list[0..k) by ckey; returns the new maximum.  Whole warp.
__device__ __forceinline__ uint64_t list_replace_max(uint64_t* list, uint32_t k, uint64_t ckey, uint64_t oldthr,
                                                     int lane) {
    int match = -1;
    for (uint32_t j = lane; j < k; j += 32)
        if (match < 0 && list[j] == oldthr) match = (int)j;
    unsigned b = __ballot_sync(0xffffffffu, match >= 0);
    if (lane == __ffs(b) - 1) list[match] = ckey;
    __syncwarp();
    uint64_t m = 0;
    for (uint32_t j = lane; j < k; j += 32) {
        uint64_t v = list[j];
        m = v > m ? v : m;
    }
    return warp_max_u64(m);
}

// Whole warp: order list[0..n) ascending inside its `cap` (power of two) slots, pad with sentinels.
__device__ __forceinline__ void warp_sort_list(uint64_t* list, uint32_t n, uint32_t cap, int lane) {
    uint32_t P = 32;
    while (P < n) P <<= 1;  // n <= cap, cap is a power of two >= 64
    for (uint32_t i = n + lane; i < cap; i += 32) list[i] = KEY_SENTINEL;
    for (uint32_t size = 2; size <= P; size <<= 1) {
        for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
            __syncwarp();
            for (uint32_t t = lane; t < (P >> 1); t += 32) {
                const uint32_t i = 2 * t - (t & (stride - 1));
                const uint32_t j = i + stride;
                const bool up = (i & size) == 0;
                const uint64_t a = list[i], b = list[j];
                if ((a > b) == up) {
                    list[i] = b;
                    list[j] = a;
                }
            }
        }
    }
    __syncwarp();
}

// 32 keys, one per lane -> ascending across the lanes (bitonic network over shuffles)
__device__ __forceinline__ uint64_t warp_bitonic_sort_u64(uint64_t v, int lane) {
#pragma unroll
    for (int size = 2; size <= 32; size <<= 1) {
#pragma unroll
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            const uint64_t o = shfl_u64(v, lane ^ stride);
            const bool keep_min = ((lane & size) == 0) == ((lane & stride) == 0);
            v = (keep_min == (o < v)) ? o : v;
        }
    }
    return v;
}

// number of keys of the ascending list[0..k) that are < key (strict) or <= key (!strict)
__device__ __forceinline__ uint32_t sorted_count_below(const uint64_t* list, uint32_t k, uint64_t key, bool strict) {
    uint32_t lo = 0, hi = k;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        const uint64_t v = list[mid];
        if (strict ? (v < key) : (v <= key))
            lo = mid + 1;
        else
            hi = mid;
    }
    return lo;
}

// D += A B: A 16 x 32 int8 (row-major fragment a0..a3), B 32 x 8 int8 (b0, b1), int32 accumulators (exact)
__device__ __forceinline__ void mma_m16n8k32_s8(int (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k32.row.col.s32.s8.s8.s32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                 : "+r"(c[0]), "+r"(c[1]), "+r"(c[2]), "+r"(c[3])
                 : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

// D += A B: A 16 x 16 halves (row-major fragment a0..a3), B 16 x 8 halves (b0, b1), fp32 accumulators
__device__ __forceinline__ void mma_m16n8k16_f16(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                                 uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

template <int METRIC, int NQ, int R, bool RANGE, bool INLINE, int HALF = 0, bool DEBUG = false>
__device__ __forceinline__ void scan_body(const ScanParams& p, const float* iq) {
    constexpr int V = R * NQ;
    static_assert(V <= 32 && (V & (V - 1)) == 0, "R*NQ must be a power of two <= 32");
    // HALF: 0 = the fp32 rows; 1 = the fp16 shadow, FMA consumers; 2 = the fp16 shadow, tensor-core consumers
    // (mma.sync m16n8k16 on 16 rows x 64 halves per step, the query as halves too; rows of a multiple of 64 halves);
    // 3 = the int8 shadow, tensor-core consumers (mma.sync m16n8k32 s8 on 16 rows x 128 bytes per step, the query as two
    // int8 digits; rows of a multiple of 128 bytes)
    static_assert(!HALF || (NQ == 1 && !INLINE), "the shadow scan takes one prepared query");
    // DEBUG (scan_kernel_half_debug): the shadow range instantiation's set-up and consumers, but every live row's
    // approximate distance is stored to out_dists[row] instead of being tested, then {|q|^2, 2^-s 2^-t, scale} to
    // out_dists[n_rows ..]; static tile schedule (sched == nullptr), no tail
    static_assert(!DEBUG || (HALF && RANGE), "the debug view is of the shadow range scan");
    static_assert(HALF < 2 || R == 16, "the tensor-core consumers score 16 rows per step");
    constexpr bool Q8 = HALF == 3;
    static_assert(!Q8 || !RANGE || DEBUG, "the int8 shadow takes single kNN queries");
    constexpr bool HMMA = HALF >= 2;   // tensor-core consumers: fp16 or int8
    extern __shared__ __align__(128) unsigned char smem[];
    // fallback launch behind a shadow scan: nothing to do when that one certified its answer
    if (NQ == 1 && p.run_if && *reinterpret_cast<const volatile uint32_t*>(p.run_if) == 0) return;   // (single queries only)

    const int tid = threadIdx.x;
    const int warp = tid >> 5;
    const int lane = tid & 31;
    const int PW = (int)p.producer_warps;
    const int CW = (blockDim.x >> 5) - PW;  // consumer warps 0..CW-1; warps CW..CW+PW-1 produce
    const uint32_t n_rows = p.n_rows_dev ? __ldg(p.n_rows_dev) : p.n_rows;
    const uint32_t n_tiles = p.n_rows_dev ? (n_rows + p.tile_rows - 1) / p.tile_rows : p.n_tiles;
    const uint32_t S = p.stages;
    const uint32_t ld4 = p.ld4;
    const uint32_t k = p.k;

    float4* ring = reinterpret_cast<float4*>(smem);
    float4* qs = ring + (size_t)S * p.stage_f4;                                   // [NQ][ld4]
    const uint32_t lcap = p.list_cap;             // slots per (warp, query) list
    const bool buffered = lcap > k;               // append buffer + compaction instead of replace-max
    // float4 per query in shared memory (HALF: ld4 counts 8-half units, Q8: 16-byte units)
    const uint32_t ldq4 = Q8 ? 4 * ld4 : (HALF ? 2 * ld4 : ld4);
    // HMMA: the query once more as halves of q * 2^t ([ld4] 16-byte units), behind the fp32 copy the re-rank reads;
    // Q8: its int8 digits h | l ([ld4] 16-byte units each)
    const unsigned char* q16 = reinterpret_cast<const unsigned char*>(qs + (size_t)NQ * ldq4);
    uint64_t* lists = reinterpret_cast<uint64_t*>(qs + (size_t)NQ * ldq4 + (Q8 ? 2 * ld4 : (HMMA ? ld4 : 0)));   // [CW][NQ][lcap]
    uint64_t* full = lists + (RANGE ? 0 : (size_t)CW * NQ * lcap);                // [S]
    uint64_t* empty = full + S;                                                   // [S]
    StageMeta* meta = reinterpret_cast<StageMeta*>(empty + S);                    // [S]

    float half_qn = 0.f;                                                           // HALF: |q|^2
    float half_margin = 0.f;                                                       // HALF range mode: candidate margin
    float half_us = (HALF && !Q8) ? __uint_as_float(__ldg(p.half_state)) : 1.0f;   // HALF: 2^-s of the shadow (x 2^-t of the query); Q8: t
    float q8_del = 0.f;                                                            // Q8: the query's q8_delta
    if (tid == 0) {
        for (uint32_t s = 0; s < S; s++) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], CW);
        }
        mbar_fence_init();
    }
    if (!RANGE)
        for (uint32_t i = tid; i < (uint32_t)CW * NQ * lcap; i += blockDim.x) lists[i] = KEY_SENTINEL;
    if (INLINE) {
        // the raw query comes with the launch: pad it to ld and, for cosine, normalise it with prep_queries_kernel's
        // exact arithmetic (lane l sums elements l, l+32, ... with fmaf, butterfly over the lanes, v * inv)
        __shared__ float s_inv;
        float* qf = reinterpret_cast<float*>(qs);
        for (uint32_t j = tid; j < ld4 * 4; j += blockDim.x) qf[j] = j < p.dim ? iq[j] : 0.f;
        __syncthreads();
        if (p.normalize) {
            if (warp == 0) {
                float acc = 0.f;
                for (uint32_t j = lane; j < p.dim; j += 32) acc = fmaf(qf[j], qf[j], acc);
#pragma unroll
                for (int off = 16; off >= 1; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
                if (lane == 0) s_inv = 1.0f / (sqrtf(acc) + 1e-30f);
            }
            __syncthreads();
            const float inv = s_inv;
            for (uint32_t j = tid; j < p.dim; j += blockDim.x) qf[j] = qf[j] * inv;
        }
    } else if (HALF) {
        // the fp32 prepared query, zero padded to the shadow's row length; |q|^2 for the l2 form and the certificate
        __shared__ float s_qn_init, s_q_unscale, s_q8[3];
        for (uint32_t i = tid; i < ldq4; i += blockDim.x)
            qs[i] = i < p.ld4_exact ? p.queries[i] : make_float4(0.f, 0.f, 0.f, 0.f);
        __syncthreads();
        if (warp == 0) {
            float acc = 0.f;
            for (uint32_t j = lane; j < p.ld4_exact; j += 32) {
                const float4 v = qs[j];
                acc = fmaf(v.x, v.x, acc);
                acc = fmaf(v.y, v.y, acc);
                acc = fmaf(v.z, v.z, acc);
                acc = fmaf(v.w, v.w, acc);
            }
#pragma unroll
            for (int off = 16; off >= 1; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
            if (lane == 0) s_qn_init = acc;
            if (Q8) {
                // q = t (h + l / 254) + r: two int8 digits per element, t = max |q| / 127; zero padding stays zero
                float m = 0.f;
                for (uint32_t j = lane; j < ldq4; j += 32) {
                    const float4 v = qs[j];
                    m = fmaxf(m, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
                }
#pragma unroll
                for (int off = 16; off >= 1; off >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, off));
                const float t = m / 127.0f, inv = m > 0.f ? 127.0f / m : 0.f, tl = t * (1.0f / 254.0f);
                uint32_t* dh = reinterpret_cast<uint32_t*>(const_cast<unsigned char*>(q16));
                uint32_t* dl = dh + ld4 * 4;
                float rr = 0.f, hh = 0.f, ll = 0.f;
                for (uint32_t j = lane; j < ldq4; j += 32) {
                    const float4 v4 = qs[j];
                    const float v[4] = {v4.x, v4.y, v4.z, v4.w};
                    uint32_t ph = 0, pl = 0;
#pragma unroll
                    for (int i = 0; i < 4; i++) {
                        const float h = fminf(fmaxf(rintf(v[i] * inv), -127.f), 127.f);
                        const float r1 = fmaf(-t, h, v[i]);
                        const float l = fminf(fmaxf(rintf(r1 * inv * 254.0f), -127.f), 127.f);
                        const float r = fmaf(-tl, l, r1);
                        rr = fmaf(r, r, rr);
                        hh = fmaf(h, h, hh);
                        ll = fmaf(l, l, ll);
                        ph |= ((uint32_t)(int32_t)h & 0xffu) << (8 * i);
                        pl |= ((uint32_t)(int32_t)l & 0xffu) << (8 * i);
                    }
                    dh[j] = ph;
                    dl[j] = pl;
                }
#pragma unroll
                for (int off = 16; off >= 1; off >>= 1) {
                    rr += __shfl_xor_sync(0xffffffffu, rr, off);
                    hh += __shfl_xor_sync(0xffffffffu, hh, off);
                    ll += __shfl_xor_sync(0xffffffffu, ll, off);
                }
                if (lane == 0) {
                    // |r| rounded up: the two fmas per element and fl(t / 254) leave <= 2^-22 t each, the sum of squares
                    // is off by <= d 2^-23 of itself
                    const float d = (float)(ldq4 * 4);
                    s_q8[0] = t;
                    s_q8[1] = sqrtf(rr) * (1.0f + d * 1.1920928955078125e-7f) + t * sqrtf(d) * 2.384185791015625e-7f;
                    s_q8[2] = t * (sqrtf(hh) + sqrtf(ll) * (1.0f / 254.0f)) * 1.0001f;
                }
            }
            if (HMMA && !Q8) {
                // halves of q * 2^t, t from the largest component (split_queries_f16_kernel's rule); zero padding stays zero
                float m = 0.f;
                for (uint32_t j = lane; j < p.ld4_exact; j += 32) {
                    const float4 v = qs[j];
                    m = fmaxf(m, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
                }
#pragma unroll
                for (int off = 16; off >= 1; off >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, off));
                const int sq = f16_scale_exp(m);
                const float scale = ldexpf(1.0f, sq);
                if (lane == 0) s_q_unscale = ldexpf(1.0f, -sq);
                __half2* dst = reinterpret_cast<__half2*>(const_cast<unsigned char*>(q16));
                for (uint32_t j = lane; j < ldq4; j += 32) {   // ldq4 float4 = ld16 floats -> ld16 halves
                    const float4 v = qs[j];
                    dst[2 * j] = __floats2half2_rn(v.x * scale, v.y * scale);
                    dst[2 * j + 1] = __floats2half2_rn(v.z * scale, v.w * scale);
                }
            }
        }
        __syncthreads();
        half_qn = s_qn_init;
        if (HMMA && !Q8) half_us *= s_q_unscale;
        if (Q8) {
            half_us = s_q8[0];
            const float xmax = p.cosine ? 1.0f : sqrtf(__uint_as_float(*p.max_norm2_bits));
            q8_del = q8_delta(METRIC == METRIC_L2, p.ld4_exact * 4, xmax, __uint_as_float(*p.q8_e_bits), sqrtf(half_qn), s_q8[1], s_q8[2]);
            if (DEBUG && blockIdx.x == 0 && tid == 0) {
                p.out_dists[p.n_rows] = half_qn;
                p.out_dists[p.n_rows + 1] = half_us;
                p.out_dists[p.n_rows + 2] = q8_del;
            }
        } else if (RANGE) {
            // shadow range scan: a row is a CANDIDATE when its approximate distance is within the fp16 error bound of the
            // radius; candidates are re-scored from the fp32 matrix on the spot and tested exactly, so the hit list is the
            // fp32 scan's by construction -- no certificate, no second launch.  An overflowed shadow makes every row a
            // candidate (slow once, still exact; the host rebuilds the shadow when it sees the flag in the mirror).
            float scale = 1.0f;
            if (!p.cosine) {
                const float xmax = sqrtf(__uint_as_float(*p.max_norm2_bits)), qsn = sqrtf(half_qn);
                scale = (METRIC == METRIC_L2) ? (xmax + qsn) * (xmax + qsn) : xmax * qsn;
            }
            const bool over = __ldg(p.half_state + 2) != 0;
            half_margin = over ? __int_as_float(0x7f800000) : p.delta_rel * scale;
            if (over && p.half_stats_host && blockIdx.x == 0 && tid == 0) p.half_stats_host[2] = 1;
            if (DEBUG && blockIdx.x == 0 && tid == 0) {
                p.out_dists[p.n_rows] = half_qn;
                p.out_dists[p.n_rows + 1] = half_us;
                p.out_dists[p.n_rows + 2] = scale;
            }
        }
    } else {
        // queries -> shared (missing queries of a short group repeat the last one; masked later)
        for (uint32_t i = tid; i < NQ * ld4; i += blockDim.x) {
            uint32_t qi = i / ld4, j = i - qi * ld4;
            uint32_t src = qi < p.nq_valid ? qi : p.nq_valid - 1;
            qs[i] = p.queries[(size_t)src * ld4 + j];
        }
    }
    __syncthreads();
    if (p.timeline && tid == 0) p.timeline[blockIdx.x * 16 + 0] = global_timer_ns();

    if (warp >= CW) {
        // ------------------------------------------------------------------ producer(s)
        // Each producer warp fills its own residue class of ring stages and claims tiles on its own, so
        // which tile lands in which stage is arbitrary; consumers walk the stages in order.
        uint32_t stage = (uint32_t)(warp - CW), phase = 0;
        const uint64_t pol = policy_evict_first();
        // whole warp (converged); lane 0 owns the barriers, in gather mode every lane issues copies
        auto issue = [&](uint32_t tile) {
            const uint32_t row0 = tile * p.tile_rows;
            const uint32_t n = min(p.tile_rows, n_rows - row0);
            // gather mode: fetch this tile's row numbers before waiting for a free stage, so the
            // lookup latency hides behind the wait (up to 128 rows per tile are prefetched)
            uint32_t ridx[4] = {0, 0, 0, 0};
            if (p.gather) {
#pragma unroll
                for (int c = 0; c < 4; c++) {
                    const uint32_t i = lane + 32u * c;
                    if (i < n) ridx[c] = __ldg(p.gather + row0 + i);
                }
            }
            if (lane == 0) mbar_wait(&empty[stage], phase ^ 1);
            __syncwarp();
            float4* dst = ring + (size_t)stage * p.stage_f4;
            if (lane == 0) {
                meta[stage].row0 = row0;
                meta[stage].n_rows = (int32_t)n;
                mbar_arrive_expect_tx(&full[stage], n * ld4 * 16u);
            }
            if (p.gather) {
                __syncwarp();
#pragma unroll
                for (int c = 0; c < 4; c++) {
                    const uint32_t i = lane + 32u * c;
                    if (i < n) bulk_g2s_hint(dst + (size_t)i * ld4, p.rows + (size_t)ridx[c] * ld4, ld4 * 16u, &full[stage], pol);
                }
                for (uint32_t i = lane + 128u; i < n; i += 32) {
                    const uint32_t r = __ldg(p.gather + row0 + i);
                    bulk_g2s_hint(dst + (size_t)i * ld4, p.rows + (size_t)r * ld4, ld4 * 16u, &full[stage], pol);
                }
            } else if (lane == 0) {
                const float4* src = p.rows + (size_t)row0 * ld4;
                if (p.evict_first)
                    bulk_g2s_hint(dst, src, n * ld4 * 16u, &full[stage], pol);
                else
                    bulk_g2s(dst, src, n * ld4 * 16u, &full[stage]);
            }
            stage += (uint32_t)PW;
            if (stage >= S) {
                stage -= S;
                phase ^= 1;
            }
        };
        if (p.sched) {
            // work stealing: claim `tile_batch` consecutive tiles per atomic; the next claim is
            // in flight while this batch's copies are issued
            uint32_t next = 0;
            if (lane == 0) next = atomicAdd(p.sched, 1u);
            next = __shfl_sync(0xffffffffu, next, 0);
            for (;;) {
                const uint32_t t0 = next * p.tile_batch;
                if (t0 >= n_tiles) break;
                if (lane == 0) next = atomicAdd(p.sched, 1u);
                const uint32_t t1 = min(t0 + p.tile_batch, n_tiles);
                for (uint32_t tile = t0; tile < t1; tile++) issue(tile);
                next = __shfl_sync(0xffffffffu, next, 0);
            }
        } else {
            for (uint32_t tile = blockIdx.x * (uint32_t)PW + (uint32_t)(warp - CW); tile < n_tiles; tile += gridDim.x * (uint32_t)PW)
                issue(tile);
        }
        if (lane == 0) {
            mbar_wait(&empty[stage], phase ^ 1);
            meta[stage].n_rows = -1;
            mbar_arrive(&full[stage]);
        }
        return;
    }

    // ---------------------------------------------------------------------- consumers
    const int slot = lane_slot<V>(lane);     // which (row-in-group, query) total this lane ends up with
    // HMMA: lane (g, t) = (lane / 4, lane % 4) of the accumulator fragment holds rows g and g + 8; t == 0 speaks for
    // row g, t == 1 for row g + 8
    const int my_r = HMMA ? ((lane >> 2) + ((lane & 3) == 1 ? 8 : 0)) : slot / NQ;
    const int my_q = HMMA ? 0 : slot - my_r * NQ;
    const bool rep = HMMA ? (lane & 3) < 2 : (lane & (32 / V - 1)) == 0;  // one representative lane per slot
    const bool q_ok = (uint32_t)my_q < p.nq_valid;
    uint64_t thr = KEY_SENTINEL;                  // current k-th best of list (warp, my_q)
    uint64_t* my_lists = lists + (size_t)warp * NQ * lcap;
    uint32_t cnt = 0;                             // buffered mode: entries in list (warp, my_q), same in every lane of a slot class

    uint32_t stage = 0, phase = 0, seq = 0;
    uint32_t rot = 0;       // == seq % CW without the division
    uint32_t finished = 0;  // producers (= stage residue classes) that have posted their end mark
    const uint32_t all_finished = (1u << PW) - 1u;
    auto advance = [&]() {
        if (++stage == S) {
            stage = 0;
            phase ^= 1;
        }
    };
    for (;;) {
        const uint32_t owner = stage & (uint32_t)(PW - 1);  // PW is 1, 2 or 4 and divides S
        if ((finished >> owner) & 1u) {  // nothing will ever land here again
            advance();
            continue;
        }
        mbar_wait(&full[stage], phase);
        if (p.timeline && tid == 0 && seq == 0) p.timeline[blockIdx.x * 16 + 1] = global_timer_ns();
        const int n = meta[stage].n_rows;
        if (n < 0) {
            finished |= 1u << owner;
            if (finished == all_finished) break;
            advance();
            continue;
        }
        const uint32_t row0 = meta[stage].row0;
        const float4* tile = ring + (size_t)stage * p.stage_f4;
        const uint32_t n_groups = ((uint32_t)n + R - 1) / R;
        // rotate the group -> warp assignment per tile so short tiles do not always hit warp 0
        uint32_t g = (uint32_t)(warp >= (int)rot ? warp - (int)rot : warp + CW - (int)rot);
        for (; g < n_groups; g += CW) {
            const uint32_t base = g * R;
            const uint32_t my_local = base + my_r;
            const uint32_t pos = min(row0 + my_local, n_rows - 1);
            // gather mode: the tile holds list positions; the list has the row numbers and is pre-masked
            const uint32_t row = p.gather ? __ldg(p.gather + pos) : row0 + my_local;
            const uint32_t rowc = p.gather ? 0u : pos;
            uint32_t wl = 0xffffffffu, wf = 0xffffffffu;
            if (!p.gather) {
                if (p.live) wl = __ldg(p.live + (rowc >> 5));
                if (p.filter) wf = __ldg(p.filter + (rowc >> 5));
            }

            float acc[V];
#pragma unroll
            for (int i = 0; i < V; i++) acc[i] = 0.f;
            const float4* trow = tile + (size_t)base * ld4;
            float xn = 0.f;
            if (HALF && METRIC == METRIC_L2) xn = __ldg(p.row_norms + (p.gather ? row : pos));   // own slot's row; in flight during the dot products
            float s_mma = 0.f;
            if constexpr (Q8) {
                // Int8 consumers: the fp16 consumers' access pattern below, with 32 bytes of k per instruction.  B columns
                // n with bit 1 clear take the query's high digit h, the others its low digit l, so one MMA yields both sums
                // for a row: D_h in column (row parity), D_l in column (row parity) + 2 -- lanes t = 0 and t = 1 of the row
                // group, which trade one value so that t == 0 holds both sums of row g and t == 1 both of row g + 8.
                const float xs = __ldg(p.q8_scale + pos);
                const int g = lane >> 2, t = lane & 3;
                const uint32_t rowbytes = ld4 * 16;
                const unsigned char* r0 = reinterpret_cast<const unsigned char*>(tile) + (size_t)(base + g) * rowbytes;
                const unsigned char* r1 = r0 + 8 * (size_t)rowbytes;
                const unsigned char* qd = q16 + ((g & 2) ? rowbytes : 0u);
                int c[4] = {0, 0, 0, 0}, d[4] = {0, 0, 0, 0};
                const uint32_t o0 = (uint32_t)(t + 4 * (g & 1)) * 16, o1 = (uint32_t)(t + 4 * ((g & 1) ^ 1)) * 16;
                for (uint32_t ch = 0; ch < rowbytes; ch += 128) {
                    {
                        const uint4 xa = *reinterpret_cast<const uint4*>(r0 + ch + o0);
                        const uint4 xb = *reinterpret_cast<const uint4*>(r1 + ch + o0);
                        const uint4 qv = *reinterpret_cast<const uint4*>(qd + ch + o0);
                        mma_m16n8k32_s8(c, xa.x, xb.x, xa.y, xb.y, qv.x, qv.y);
                        mma_m16n8k32_s8(d, xa.z, xb.z, xa.w, xb.w, qv.z, qv.w);
                    }
                    {
                        const uint4 xa = *reinterpret_cast<const uint4*>(r0 + ch + o1);
                        const uint4 xb = *reinterpret_cast<const uint4*>(r1 + ch + o1);
                        const uint4 qv = *reinterpret_cast<const uint4*>(qd + ch + o1);
                        mma_m16n8k32_s8(c, xa.x, xb.x, xa.y, xb.y, qv.x, qv.y);
                        mma_m16n8k32_s8(d, xa.z, xb.z, xa.w, xb.w, qv.z, qv.w);
                    }
                }
                // lane (g, t) holds C[g][2t + j] (j = 0, 1) and C[g + 8][2t + j]; the row parity picks j
                const int par = g & 1;
                const int lo_g = par ? c[1] + d[1] : c[0] + d[0], lo_g8 = par ? c[3] + d[3] : c[2] + d[2];
                const int got = __shfl_xor_sync(0xffffffffu, t == 0 ? lo_g8 : lo_g, 1);
                const int dh = t == 0 ? lo_g : got, dl = t == 0 ? got : lo_g8;
                s_mma = xs * ((float)dh + (float)dl * (1.0f / 254.0f));
            } else if constexpr (HMMA) {
                // Tensor-core consumers.  The dot product does not care in which order k is walked, as long as rows and
                // query agree: lane (g, t) feeds the fragment slots (row g / g + 8, k 2t.. and 2t + 8..) with the 16 bytes
                // at offset 16 (t + 4 ((g & 1) ^ step)) of the rows' current 128-byte chunk, and the B fragment (column n
                // = g) with the query's 16 bytes at the SAME offset -- so every quarter-warp reads 128 contiguous bytes
                // of two rows (no bank conflicts on rows a multiple of 128 bytes apart), and column n of the result is
                // right for the rows of n's parity.  Two steps cover the chunk; two accumulator sets halve the MMA chain.
                const int g = lane >> 2, t = lane & 3;
                const uint32_t rowbytes = ld4 * 16;
                const unsigned char* r0 = reinterpret_cast<const unsigned char*>(tile) + (size_t)(base + g) * rowbytes;
                const unsigned char* r1 = r0 + 8 * (size_t)rowbytes;
                float c[4] = {0.f, 0.f, 0.f, 0.f}, d[4] = {0.f, 0.f, 0.f, 0.f};
                const uint32_t o0 = (uint32_t)(t + 4 * (g & 1)) * 16, o1 = (uint32_t)(t + 4 * ((g & 1) ^ 1)) * 16;
                for (uint32_t ch = 0; ch < rowbytes; ch += 128) {
                    {
                        const uint4 xa = *reinterpret_cast<const uint4*>(r0 + ch + o0);
                        const uint4 xb = *reinterpret_cast<const uint4*>(r1 + ch + o0);
                        const uint4 qv = *reinterpret_cast<const uint4*>(q16 + ch + o0);
                        mma_m16n8k16_f16(c, xa.x, xb.x, xa.y, xb.y, qv.x, qv.y);
                        mma_m16n8k16_f16(d, xa.z, xb.z, xa.w, xb.w, qv.z, qv.w);
                    }
                    {
                        const uint4 xa = *reinterpret_cast<const uint4*>(r0 + ch + o1);
                        const uint4 xb = *reinterpret_cast<const uint4*>(r1 + ch + o1);
                        const uint4 qv = *reinterpret_cast<const uint4*>(q16 + ch + o1);
                        mma_m16n8k16_f16(c, xa.x, xb.x, xa.y, xb.y, qv.x, qv.y);
                        mma_m16n8k16_f16(d, xa.z, xb.z, xa.w, xb.w, qv.z, qv.w);
                    }
                }
                // lane (g, t) holds C[g][2t], C[g][2t+1], C[g+8][2t], C[g+8][2t+1]: the column of the row's parity
                const float lo = (g & 1) ? c[1] + d[1] : c[0] + d[0], hi = (g & 1) ? c[3] + d[3] : c[2] + d[2];
                s_mma = t == 0 ? lo : hi;
            } else if (HALF) {
                // 8 halves of the row against 8 floats of the query per step; the sum is a plain dot product (the
                // distance form is applied below): only candidates are chosen with it
                float acc2[V];
#pragma unroll
                for (int i = 0; i < V; i++) acc2[i] = 0.f;
#pragma unroll 2
                for (uint32_t j = lane; j < ld4; j += 32) {
                    const float4 qa = qs[2 * j], qb = qs[2 * j + 1];
#pragma unroll
                    for (int r = 0; r < R; r++) {
                        const float4 xr = trow[r * ld4 + j];
                        const float2 f0 = __half22float2(*reinterpret_cast<const __half2*>(&xr.x));
                        const float2 f1 = __half22float2(*reinterpret_cast<const __half2*>(&xr.y));
                        const float2 f2 = __half22float2(*reinterpret_cast<const __half2*>(&xr.z));
                        const float2 f3 = __half22float2(*reinterpret_cast<const __half2*>(&xr.w));
                        // two chains per row: at the power-capped clock the consumers are bound by FMA latency, not issue
                        float a = acc[r], b = acc2[r];
                        a = fmaf(f0.x, qa.x, a);
                        b = fmaf(f2.x, qb.x, b);
                        a = fmaf(f0.y, qa.y, a);
                        b = fmaf(f2.y, qb.y, b);
                        a = fmaf(f1.x, qa.z, a);
                        b = fmaf(f3.x, qb.z, b);
                        a = fmaf(f1.y, qa.w, a);
                        b = fmaf(f3.y, qb.w, b);
                        acc[r] = a;
                        acc2[r] = b;
                    }
                }
#pragma unroll
                for (int r = 0; r < R; r++) acc[r] += acc2[r];
            } else {
#pragma unroll 2
                for (uint32_t j = lane; j < ld4; j += 32) {
                    float4 q[NQ];
#pragma unroll
                    for (int qi = 0; qi < NQ; qi++) q[qi] = qs[qi * ld4 + j];
#pragma unroll
                    for (int r = 0; r < R; r++) {
                        const float4 x = trow[r * ld4 + j];
#pragma unroll
                        for (int qi = 0; qi < NQ; qi++) acc[r * NQ + qi] = accum4<METRIC>(acc[r * NQ + qi], x, q[qi]);
                    }
                }
            }
            const float s = HMMA ? s_mma : transpose_reduce<V>(acc, lane);
            float dist;
            if (HALF)   // approximate: the GEMM form on the shadow's dot product
                dist = (METRIC == METRIC_IP) ? 1.0f - half_us * s : fmaf(-2.0f * half_us, s, xn + half_qn);
            else
                dist = (METRIC == METRIC_IP) ? 1.0f - s : s;
            const uint64_t key = make_key(dist, row);
            const bool ok = rep && q_ok && my_local < (uint32_t)n && ((wl & wf) >> (rowc & 31) & 1u);
            if constexpr (DEBUG) {
                if (ok) p.out_dists[row] = dist;
            } else if (RANGE && HALF) {
                // candidates (NaN included) -> exact distance by the whole warp, the scan's own arithmetic
                unsigned cm = __ballot_sync(0xffffffffu, ok && !(dist > p.radius + half_margin));
                while (cm) {
                    const int src = __ffs(cm) - 1;
                    cm &= cm - 1;
                    const uint32_t crow = __shfl_sync(0xffffffffu, row, src);
                    const float4* xrow = p.rows_exact + (size_t)crow * p.ld4_exact;
                    float acc = 0.f;
                    for (uint32_t j = lane; j < p.ld4_exact; j += 32) acc = accum4<METRIC>(acc, __ldg(xrow + j), qs[j]);
#pragma unroll
                    for (int off = 16; off >= 1; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
                    const float exact = (METRIC == METRIC_IP) ? 1.0f - acc : acc;
                    if (lane == 0 && exact <= p.radius) {
                        unsigned long long pos = atomicAdd(p.range_counts, 1ull);
                        if (pos < p.max_hits) p.range_keys[pos] = make_key(exact, crow);
                    }
                }
            } else if (RANGE) {
                if (ok && dist <= p.radius) {
                    unsigned long long pos = atomicAdd(p.range_counts + my_q, 1ull);
                    if (pos < p.max_hits) p.range_keys[(size_t)my_q * p.max_hits + pos] = key;
                }
            } else {
                unsigned m = __ballot_sync(0xffffffffu, ok && key < thr);
                if (!buffered) {
                    while (m) {
                        const int src = __ffs(m) - 1;
                        m &= m - 1;
                        const uint64_t ckey = shfl_u64(key, src);
                        const uint64_t cthr = shfl_u64(thr, src);
                        const int cq = __shfl_sync(0xffffffffu, my_q, src);
                        if (ckey < cthr) {
                            const uint64_t nthr = list_replace_max(my_lists + (size_t)cq * k, k, ckey, cthr, lane);
                            if (my_q == cq) thr = nthr;
                        }
                    }
                } else {
                    while (m) {
                        // all candidates of one query in this step are appended together
                        const int src = __ffs(m) - 1;
                        const int cq = __shfl_sync(0xffffffffu, my_q, src);
                        const unsigned mq = __ballot_sync(0xffffffffu, ((m >> lane) & 1u) && my_q == cq);
                        m &= ~mq;
                        const uint32_t base = __shfl_sync(0xffffffffu, cnt, src);
                        uint64_t* list = my_lists + (size_t)cq * lcap;
                        if ((mq >> lane) & 1u) list[base + __popc(mq & ((1u << lane) - 1u))] = key;
                        uint32_t ncnt = base + __popc(mq);
                        uint64_t nthr = shfl_u64(thr, src);
                        if (ncnt + 32 > lcap) {  // fewer than a step's worth of free slots: keep the k best
                            __syncwarp();
                            warp_sort_list(list, ncnt, lcap, lane);
                            ncnt = min(ncnt, k);
                            nthr = list[k - 1];  // sentinel while fewer than k rows were seen
                        }
                        if (my_q == cq) {
                            cnt = ncnt;
                            thr = nthr;
                        }
                    }
                }
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[stage]);
        seq++;
        if (++rot == (uint32_t)CW) rot = 0;
        advance();
    }
    if (p.timeline && tid == 0) p.timeline[blockIdx.x * 16 + 2] = global_timer_ns();
    const uint32_t nthr = (uint32_t)CW * 32u;  // consumer threads (the producer warps have left)
    if (!RANGE) {
        // --------------------------------------------- fold the CW warp lists into one per query
        if (buffered) {
            // last compaction: every list of this warp ascending, k slots valid-or-sentinel
            for (uint32_t qi = 0; qi < (uint32_t)NQ && qi < p.nq_valid; qi++) {
                const unsigned owners = __ballot_sync(0xffffffffu, my_q == (int)qi);
                const uint32_t n = __shfl_sync(0xffffffffu, cnt, __ffs(owners) - 1);
                warp_sort_list(my_lists + (size_t)qi * lcap, n, lcap, lane);
            }
        } else {
            // k <= 32 unsorted keys per list: one key per lane, sorted in registers (a rank-by-counting fold over
            // CW * k unsorted keys cost 7 us of a 12 us launch on a 10k-row namespace; the merge below costs < 1 us)
            __syncwarp();
            for (uint32_t qi = 0; qi < (uint32_t)NQ && qi < p.nq_valid; qi++) {
                uint64_t* l = my_lists + (size_t)qi * lcap;
                uint64_t v = (uint32_t)lane < k ? l[lane] : KEY_SENTINEL;
                v = warp_bitonic_sort_u64(v, lane);
                if ((uint32_t)lane < k) l[lane] = v;
            }
        }
        if (p.timeline && tid == 0) p.timeline[blockIdx.x * 16 + 8] = global_timer_ns();    // own lists sorted
        named_bar_sync(1, CW * 32);
        if (p.timeline && tid == 0) p.timeline[blockIdx.x * 16 + 9] = global_timer_ns();    // every warp's lists sorted
        const uint32_t n_in = (uint32_t)CW * k;
        __shared__ uint32_t s_fm;
        __shared__ unsigned long long s_fT;
        for (uint32_t qi = 0; qi < p.nq_valid; qi++) {
            uint64_t* out = p.out_keys + ((size_t)qi * gridDim.x + blockIdx.x) * k;
            if (buffered) {
                for (uint32_t e = tid; e < n_in; e += nthr) {
                    const uint32_t w = e / k, j = e - w * k;
                    const uint64_t key = lists[((size_t)w * NQ + qi) * lcap + j];
                    // CW ascending lists: rank = own position + keys below it in the other lists (binary
                    // search); equal keys (sentinels only) are ordered by list, then position
                    uint32_t rank = j;
                    for (uint32_t w2 = 0; w2 < (uint32_t)CW; w2++)
                        if (w2 != w) rank += sorted_count_below(lists + ((size_t)w2 * NQ + qi) * lcap, k, key, w2 > w);
                    if (rank < k) out[rank] = key;  // the block's k best, ascending
                }
                continue;
            }
            // k <= 32, every warp list ascending.  The first ceil(k / CW) keys of each list are >= k keys, so the k-th
            // smallest of that small pool bounds the block's k-th best: only keys <= it survive (about k of CW * k), and
            // ranking the survivors is O(k^2) instead of O((CW k)^2).  Scratch: the ring, idle since the barrier above.
            uint64_t* pool = reinterpret_cast<uint64_t*>(ring);   // [<= 64] pool, then [CW * k] survivors
            uint64_t* surv = pool + 64;
            const uint32_t take = (k + (uint32_t)CW - 1) / (uint32_t)CW;
            const uint32_t P = min((uint32_t)CW * take, 64u);
            if (tid < P) {
                const uint32_t w = tid / take, j = tid - w * take;
                pool[tid] = lists[((size_t)w * NQ + qi) * lcap + j];
            }
            if (tid == 0) s_fm = 0;
            named_bar_sync(1, CW * 32);
            if (tid < P) {
                const uint64_t key = pool[tid];
                uint32_t rank = 0;
#pragma unroll 8
                for (uint32_t i = 0; i < P; i++) {
                    const uint64_t o = pool[i];
                    rank += (o < key) || (o == key && i < tid);
                }
                if (rank == min(k, P) - 1) s_fT = key;
            }
            named_bar_sync(1, CW * 32);
            if (p.timeline && tid == 0) p.timeline[blockIdx.x * 16 + 13] = global_timer_ns();   // fold: pool threshold known
            const uint64_t T = s_fT;
            for (uint32_t e = tid; e < n_in; e += nthr) {
                const uint32_t w = e / k, j = e - w * k;
                const uint64_t key = lists[((size_t)w * NQ + qi) * lcap + j];
                if (key <= T && key != KEY_SENTINEL) surv[atomicAdd(&s_fm, 1u)] = key;
            }
            named_bar_sync(1, CW * 32);
            if (p.timeline && tid == 0) p.timeline[blockIdx.x * 16 + 14] = global_timer_ns();   // fold: survivors gathered
            const uint32_t m = s_fm;
            if (p.timeline && tid == 0) p.timeline[blockIdx.x * 16 + 15] = m;                   // (a count, not a time)
            for (uint32_t e = tid; e < m; e += nthr) {
                const uint64_t key = surv[e];
                uint32_t rank = 0;
#pragma unroll 8
                for (uint32_t i = 0; i < m; i++) {
                    const uint64_t o = surv[i];
                    rank += (o < key) || (o == key && i < e);
                }
                if (rank < k) out[rank] = key;  // the block's k best, ascending
            }
            for (uint32_t r = m + tid; r < k; r += nthr) out[r] = KEY_SENTINEL;   // fewer than k rows seen
            named_bar_sync(1, CW * 32);   // pool / surv are reused by the next query
        }
    }
    if (p.timeline && tid == 0) p.timeline[blockIdx.x * 16 + 3] = global_timer_ns();
    if (!p.sched) return;

    // ------------------------------------------------- last CTA: scheduler reset, fused final select
    __shared__ uint32_t s_ticket, s_m, s_valid;
    __shared__ unsigned long long s_T;
    __shared__ unsigned long long s_rcnt[XCHG_MAX_WORLD + 3];
    named_bar_sync(1, CW * 32);  // every out_keys store of this CTA has been issued
    if (tid == 0) {
        __threadfence();
        s_valid = 0;
        s_ticket = atomicAdd(p.sched + 1, 1u);
    }
    named_bar_sync(1, CW * 32);
    if (p.timeline && tid == 0) p.timeline[blockIdx.x * 16 + 4] = global_timer_ns();   // ticket taken
    if (s_ticket != gridDim.x - 1) return;
    __threadfence();
    if (p.timeline && tid == 0) p.timeline[blockIdx.x * 16 + 10] = global_timer_ns();       // last CTA: past the fence
    if (!RANGE && p.fused) {
        // The ring is idle now: reuse it.  cand[fused_cap] | top[nq_valid][k]
        uint64_t* cand = reinterpret_cast<uint64_t*>(ring);
        uint64_t* top = cand + p.fused_cap;
        const uint32_t n_lists = gridDim.x, n = n_lists * k;
        for (uint32_t qi = 0; qi < p.nq_valid; qi++) {
            const uint64_t* keys = p.out_keys + (size_t)qi * n_lists * k;
            if (tid == 0) {
                s_T = KEY_SENTINEL;
                s_m = 0;
            }
            named_bar_sync(1, CW * 32);
            // every block list is sorted, so its last key is its maximum; the global k-th best is at
            // most the smallest of those maxima: only keys <= T can be in the final top-k
            // (148 threads doing a 64-bit atomicMin on one shared word is a CAS loop that cost ~5 us: reduce in the warp first)
            {
                uint64_t mine = KEY_SENTINEL;
                for (uint32_t l = tid; l < n_lists; l += nthr) {
                    const uint64_t v = __ldcg(keys + (size_t)l * k + k - 1);
                    mine = v < mine ? v : mine;
                }
                mine = ~warp_max_u64(~mine);
                if (lane == 0 && mine != KEY_SENTINEL) atomicMin(&s_T, (unsigned long long)mine);
            }
            // A much tighter bound when a warp's worth of lists holds at least k valid FIRST keys: sorted across the lanes,
            // the k-th of them has k keys <= it, so the global k-th best is too.  On 148 lists of 10 it leaves ~40
            // survivors instead of ~250 (whose O(m^2) ranking cost 7 us), for one register sort per warp.
            if (HALF && k > 16 && k <= n_lists) {
                // ... for larger k (the shadow scan's k' = 32) a warp's worth of heads says little (its k-th is its
                // largest); the k-th smallest of ALL the heads does: ranked by counting in the still unused candidate
                // array.  Without it ~1000 of 148 x 32 keys survived and went through the bitonic network (16 us).
                for (uint32_t l = tid; l < n_lists; l += nthr) cand[l] = __ldcg(keys + (size_t)l * k);
                named_bar_sync(1, CW * 32);
                for (uint32_t l = tid; l < n_lists; l += nthr) {
                    const uint64_t key = cand[l];
                    uint32_t rank = 0;
#pragma unroll 8
                    for (uint32_t i = 0; i < n_lists; i++) {
                        const uint64_t o = cand[i];
                        rank += (o < key) || (o == key && i < l);
                    }
                    if (rank == k - 1 && key != KEY_SENTINEL) atomicMin(&s_T, (unsigned long long)key);
                }
            } else if (k <= 32) {
                for (uint32_t l0 = (uint32_t)warp * 32u; l0 < n_lists; l0 += nthr) {
                    const uint32_t l = l0 + (uint32_t)lane;
                    uint64_t hd = l < n_lists ? __ldcg(keys + (size_t)l * k) : KEY_SENTINEL;
                    hd = warp_bitonic_sort_u64(hd, lane);
                    const uint64_t kth = shfl_u64(hd, (int)k - 1);
                    if (lane == 0 && kth != KEY_SENTINEL) atomicMin(&s_T, (unsigned long long)kth);
                }
            }
            named_bar_sync(1, CW * 32);
            if (p.timeline && tid == 0) p.timeline[blockIdx.x * 16 + 11] = global_timer_ns();   // threshold known
            const uint64_t T = s_T;
            // four independent loads per thread and step: with k' = 32 keys per block list (shadow scan) and few consumer
            // warps this loop was 10 us of dependent L2 round trips
            constexpr int GU = HALF ? 4 : 1;   // (the fp32 instantiations have no registers to spare and 3x fewer keys)
            for (uint32_t i0 = tid; i0 < n; i0 += GU * nthr) {
                uint64_t key[GU];
#pragma unroll
                for (int u = 0; u < GU; u++) key[u] = i0 + u * nthr < n ? __ldcg(keys + i0 + u * nthr) : KEY_SENTINEL;
#pragma unroll
                for (int u = 0; u < GU; u++)
                    if (i0 + u * nthr < n && key[u] <= T) cand[atomicAdd(&s_m, 1u)] = key[u];
            }
            named_bar_sync(1, CW * 32);
            if (p.timeline && tid == 0) p.timeline[blockIdx.x * 16 + 12] = global_timer_ns();   // survivors gathered
            const uint32_t m = s_m;
            if (m <= 512) {
                // few survivors: rank by counting
                for (uint32_t e = tid; e < m; e += nthr) {
                    const uint64_t key = cand[e];
                    uint32_t rank = 0;
#pragma unroll 8
                    for (uint32_t i = 0; i < m; i++) {
                        const uint64_t o = cand[i];
                        rank += (o < key) || (o == key && i < e);
                    }
                    if (rank < k) top[qi * k + rank] = key;
                }
                named_bar_sync(1, CW * 32);
            } else {
                // many survivors (larger k): bitonic network over the consumer threads
                uint32_t P = 1024;
                while (P < m) P <<= 1;
                for (uint32_t i = m + tid; i < P; i += nthr) cand[i] = KEY_SENTINEL;
                for (uint32_t size = 2; size <= P; size <<= 1) {
                    for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
                        named_bar_sync(1, CW * 32);
                        for (uint32_t t = tid; t < (P >> 1); t += nthr) {
                            const uint32_t i = 2 * t - (t & (stride - 1));
                            const uint32_t j = i + stride;
                            const bool up = (i & size) == 0;
                            const uint64_t a = cand[i], b = cand[j];
                            if ((a > b) == up) {
                                cand[i] = b;
                                cand[j] = a;
                            }
                        }
                    }
                }
                named_bar_sync(1, CW * 32);
                for (uint32_t j = tid; j < k; j += nthr) top[qi * k + j] = cand[j];
                named_bar_sync(1, CW * 32);
            }
        }
        // what the output stage below reads: the final keys, kf per query
        const uint64_t* fin = top;
        uint32_t kf = k;
        uint32_t my_uncert = 0;   // HALF: bit qi = query qi is not certified on this rank (same in every thread)
        if (HALF) {
            // ---- exact re-rank of the k' <= 64 candidates + certificate (see ScanParams) ----
            __shared__ uint32_t s_uncert;
            uint64_t* ex = top + (size_t)p.nq_valid * k;        // [nq][64] exact keys, unsorted
            uint64_t* fx = ex + (size_t)p.nq_valid * 64;        // [nq][k_out] exact keys, ascending
            if (tid == 0) s_uncert = 0;
            // four candidates per warp at a time: their rows are four independent HBM round trips (a candidate at a time
            // cost ~1.5 us each, 8 per warp); per candidate the scan's own arithmetic -- lane l sums float4 columns l,
            // l + 32, ..., butterfly over the lanes
            for (uint32_t e0 = (uint32_t)warp * 4u; e0 < p.nq_valid * k; e0 += (uint32_t)CW * 4u) {
                uint64_t keys[4];
                const float4* xrow[4];
                float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    keys[u] = e0 + u < p.nq_valid * k ? top[e0 + u] : KEY_SENTINEL;
                    xrow[u] = p.rows_exact + (size_t)(keys[u] != KEY_SENTINEL ? key_row(keys[u]) : 0u) * p.ld4_exact;
                }
                const float4* qv = qs + (size_t)(e0 / k) * ldq4;   // k is a multiple of 4: the four share their query
                for (uint32_t j = lane; j < p.ld4_exact; j += 32) {
                    const float4 q4 = qv[j];
#pragma unroll
                    for (int u = 0; u < 4; u++) acc[u] = accum4<METRIC>(acc[u], __ldg(xrow[u] + j), q4);
                }
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    float a = acc[u];
#pragma unroll
                    for (int off = 16; off >= 1; off >>= 1) a += __shfl_xor_sync(0xffffffffu, a, off);
                    if (lane == 0 && e0 + u < p.nq_valid * k) {
                        const uint32_t qi = (e0 + u) / k, i = (e0 + u) - qi * k;
                        ex[qi * 64 + i] = keys[u] != KEY_SENTINEL ? make_key((METRIC == METRIC_IP) ? 1.0f - a : a, key_row(keys[u])) : KEY_SENTINEL;
                    }
                }
            }
            named_bar_sync(1, CW * 32);
            if ((uint32_t)warp < p.nq_valid) {
                const uint32_t qi = (uint32_t)warp;
                uint64_t* xs = ex + qi * 64;
                warp_sort_list(xs, k, 64, lane);
                if ((uint32_t)lane < p.k_out) fx[qi * p.k_out + lane] = xs[lane];
                const uint64_t last = top[qi * k + k - 1];                 // k'-th approximate key: sentinel = every row is a candidate
                const uint64_t ek = xs[p.k_out - 1];                       // exact k-th best among the candidates
                bool certified = true;
                if (last != KEY_SENTINEL) {
                    float delta = q8_del;
                    if (!Q8) {
                        float scale = 1.0f;
                        if (!p.cosine) {
                            const float xmax = sqrtf(__uint_as_float(*p.max_norm2_bits)), qsn = sqrtf(half_qn);
                            scale = (METRIC == METRIC_L2) ? (xmax + qsn) * (xmax + qsn) : xmax * qsn;
                        }
                        delta = p.delta_rel * scale;
                    }
                    certified = (key_dist(last) - delta > key_dist(ek));   // false for NaN
                }
                if (!Q8 && __ldg(p.half_state + 2)) certified = false;   // the shadow overflowed fp16: nothing it selected can be trusted
                if (lane == 0 && !certified) atomicOr(&s_uncert, 1u << qi);
            }
            named_bar_sync(1, CW * 32);
            my_uncert = s_uncert;
            fin = fx;
            kf = p.k_out;
        }
        if (p.timeline && tid == 0) p.timeline[blockIdx.x * 16 + 5] = global_timer_ns();   // last CTA: final select done
        const ExchangeView& x = p.xchg;
        uint32_t any_uncert = my_uncert;
        if (x.world <= 1 && p.tagged_out) {
            for (uint32_t i = tid; i <= k; i += nthr) {
                uint4 rec;
                if (i < k) {
                    const uint64_t key = top[i];
                    const bool valid = key != KEY_SENTINEL;
                    const unsigned long long row = valid ? (unsigned long long)(p.row_base + key_row(key)) : ~0ull;
                    rec = make_uint4(valid ? __float_as_uint(key_dist(key)) : 0x7f800000u, p.tag, (uint32_t)row, (uint32_t)(row >> 32));
                } else {
                    uint32_t c = 0;
                    for (uint32_t j = 0; j < k; j++) c += top[j] != KEY_SENTINEL;
                    rec = make_uint4(c, p.tag, 0u, 0u);
                }
                asm volatile("st.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p.tagged_out + i), "r"(rec.x), "r"(rec.y), "r"(rec.z), "r"(rec.w)
                             : "memory");
            }
        } else if (x.world <= 1) {
            for (uint32_t i = tid; i < p.nq_valid * kf; i += nthr) {
                const uint64_t key = fin[i];
                const bool valid = key != KEY_SENTINEL;
                p.out_dists[i] = valid ? key_dist(key) : __int_as_float(0x7f800000);
                p.out_rows[i] = valid ? (int64_t)(p.row_base + key_row(key)) : -1;
            }
            for (uint32_t qi = tid; qi < p.nq_valid; qi += nthr) {
                int c = 0;
                for (uint32_t j = 0; j < kf; j++) c += fin[qi * kf + j] != KEY_SENTINEL;
                p.out_counts[qi] = c;
            }
        } else {
            // p.cert: this launch is the first of a {first tier, conditional fp32} pair -- the ranks also agree on whether
            // any of them failed to certify (an fp32 first launch always certifies)
            any_uncert = exchange_and_merge(x, fin, p.nq_valid, kf, p.out_dists, p.out_rows, p.out_counts, tid, nthr, &s_valid,
                                            NQ == 1 && p.cert != nullptr, my_uncert);
        }
        if (NQ == 1 && p.cert && tid == 0) {
            *p.cert = any_uncert ? 1u : 0u;
            if (HALF) {
                uint32_t* cnt = p.half_stats + (Q8 ? 2 : 0);
                const uint32_t a = atomicAdd(cnt, p.nq_valid) + p.nq_valid;
                const uint32_t b = atomicAdd(cnt + 1, (uint32_t)__popc(my_uncert)) + (uint32_t)__popc(my_uncert);
                if (p.half_stats_host) {
                    p.half_stats_host[Q8 ? 4 : 0] = a;
                    p.half_stats_host[Q8 ? 5 : 1] = b;
                    if (!Q8) p.half_stats_host[2] = __ldg(p.half_state + 2);
                }
            }
        }
    }
    if (RANGE && p.fused) {
        // range search across row shards: this rank's hits (appended to range_keys by every CTA; the ticket made them
        // visible) are sorted here, exchanged over peer memory and merged -- one launch per query, no NCCL call
        uint64_t* a = reinterpret_cast<uint64_t*>(smem);
        const unsigned long long found = *reinterpret_cast<volatile unsigned long long*>(p.range_counts);
        const unsigned long long share = XCHG_SLOT_KEYS / p.xchg.world;
        const uint32_t n_local = (uint32_t)(found <= share ? found : 0);
        for (uint32_t i = tid; i < n_local; i += nthr) a[i] = __ldcg(p.range_keys + i);
        named_bar_sync(1, CW * 32);
        range_exchange_and_merge(p.xchg, a, n_local, found, p.out_dists, p.out_rows, p.range_out_count, tid, nthr, s_rcnt);
    }
    if (p.timeline && tid == 0) p.timeline[blockIdx.x * 16 + 6] = global_timer_ns();       // last CTA: outputs written
    if (p.done_flag) {   // results (possibly in mapped host memory) before the flag
        __threadfence_system();
        named_bar_sync(1, CW * 32);
        if (tid == 0) asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p.done_flag), "r"(p.done_value) : "memory");
        if (p.timeline && tid == 0) p.timeline[blockIdx.x * 16 + 7] = global_timer_ns();   // flag raised
    }
    if (tid == 0) {
        p.sched[0] = 0;
        p.sched[1] = 0;
    }
}

template <int METRIC, int NQ, int R, bool RANGE>
__global__ void __launch_bounds__(scan_max_threads<NQ>(), 1) scan_kernel(const ScanParams p) {
    scan_body<METRIC, NQ, R, RANGE, false>(p, nullptr);
}
// one query over the fp16 shadow of the rows, exact re-rank + certificate in the fused tail (ScanParams::rows_exact)
template <int METRIC, int R, bool RANGE = false>
__global__ void __launch_bounds__(scan_max_threads<4>(), 1) scan_kernel_half(const ScanParams p) {   // <= 8 consumer warps
    scan_body<METRIC, 1, R, RANGE, false, 1>(p, nullptr);
}
// ... with tensor-core consumers (rows of a multiple of 64 halves): 16 rows per warp step
template <int METRIC, bool RANGE = false>
__global__ void __launch_bounds__(256, 1) scan_kernel_half_mma(const ScanParams p) {   // <= 7 consumer warps + 1 producer
    scan_body<METRIC, 1, 16, RANGE, false, 2>(p, nullptr);
}
// one query over the int8 shadow (rows of a multiple of 128 bytes), int8 tensor-core consumers, k' <= 64
template <int METRIC>
__global__ void __launch_bounds__(256, 1) scan_kernel_q8(const ScanParams p) {   // <= 7 consumer warps + 1 producer
    scan_body<METRIC, 1, 16, false, false, 3>(p, nullptr);
}
// tests only (mlv_index_debug_half_scan): the approximate distance of every live row, from the consumers above
template <int METRIC, int R>
__global__ void __launch_bounds__(scan_max_threads<4>(), 1) scan_kernel_half_debug(const ScanParams p) {
    scan_body<METRIC, 1, R, true, false, 1, true>(p, nullptr);
}
template <int METRIC>
__global__ void __launch_bounds__(256, 1) scan_kernel_half_mma_debug(const ScanParams p) {
    scan_body<METRIC, 1, 16, true, false, 2, true>(p, nullptr);
}
// tests only (mlv_index_debug_q8_scan): the int8 consumers' approximate distance of every live row, then {|q|^2, t, delta}
template <int METRIC>
__global__ void __launch_bounds__(256, 1) scan_kernel_q8_debug(const ScanParams p) {
    scan_body<METRIC, 1, 16, true, false, 3, true>(p, nullptr);
}
// one query whose raw values travel in the launch parameters (batch-1 latency path)
template <int METRIC, int R, bool RANGE>
__global__ void __launch_bounds__(SCAN_MAX_THREADS, 1) scan_kernel_iq(const __grid_constant__ ScanParams p,
                                                                      const __grid_constant__ InlineQuery iq) {
    scan_body<METRIC, 1, R, RANGE, true>(p, iq.v);
}

}  // namespace mlv
