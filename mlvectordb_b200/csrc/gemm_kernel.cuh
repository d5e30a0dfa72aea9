// gemm_kernel.cuh -- large query batches: the distance matrix as a tensor-core contraction
// (tcgen05.mma kind::tf32, 3xTF32 split, accumulators in TMEM, operands staged by TMA) with the
// metric transform, tombstone/filter mask and candidate selection fused into the epilogue.
//
// The reference has no batch API (Index.search takes one query: src/mlvectordb/implementations/
// index.py:91-129); BASELINE.json configs[2] (10M x 768, k=100, 4096-query batches) is this path.
//
// A GEMM computes l2 as |x|^2 + |q|^2 - 2 x.q, which is not the reference's arithmetic
// (hnswlib: sum (x_i - q_i)^2), so this kernel only SELECTS: it keeps, per query, the k' = k + slack
// rows with the smallest approximate distance `a`.  rerank_kernel then recomputes those rows in the
// reference's form with the scan kernel's exact summation order (bit-identical scores) and
// certifies the result:  every row outside the candidate set has a >= a_k', hence an exact distance
// >= a_k' - delta; if the exact k-th best is below that, no outside row can belong to the top-k.
// Queries that fail the certificate (or overflow their candidate buffer) are re-run by the exact
// scan; the host does that, so results never depend on which path ran.
//
// Structure (one CTA per SM, 320 threads):
//   warp 0      TMA producer: per K chunk of 32 floats one X tile [128 rows] and the Qhi/Qlo tiles
//               [256 queries] -> 128B-swizzled shared memory, 2-stage ring, full/empty mbarriers
//   warps 2-5   split X in place into hi = x & 0xffffe000 (what kind::tf32 consumes) and
//               lo = x - hi (second buffer); elementwise, so the swizzle is irrelevant to them
//   warp 1      MMA issuer: per 8-float K step  D += Xhi.Qhi + Xhi.Qlo + Xlo.Qhi  (M=128, N=256);
//               two accumulators (2 x 256 TMEM columns) so the epilogue overlaps the next tile
//   warps 6-9   epilogue: tcgen05.ld 32 columns at a time; thread = row, column = query;
//               a = metric(dot); rows passing the query's current threshold are appended to the
//               query's candidate buffer (atomic slot claim)
// Thresholds only change between launches: the host runs the scan of the rows as a sequence of
// geometrically growing rounds, each followed by refine_kernel (keep the best k', set thr = a_k').
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>

#include "common.cuh"
#include "scan_kernel.cuh"
#include "select_kernel.cuh"

namespace mlv {

constexpr int GEMM_BM = 128;  // rows per tile      (UMMA M)
constexpr int GEMM_BK = 32;   // floats per K chunk (one 128-byte swizzle row)
constexpr int GEMM_THREADS = 320;
constexpr uint32_t GEMM_X_BYTES = GEMM_BM * GEMM_BK * 4;   // 16 KB
// Three shapes: BN = 256 queries per tile with a 2-stage ring (96 KB stages) for large batches (tensor-
// bound); BN = 128 / 3 stages and BN = 64 / 4 stages for small batches, where a pass over the rows
// is HBM-bound and padding the query tile to 256 columns would only burn tensor time.
//
// PASSES = 3 is the 3xTF32 split described above.  PASSES = 1 is the fast first tier: ONE kind::tf32 MMA per K
// step on the raw fp32 tiles (the tensor core reads the top 19 bits of each operand, i.e. the same truncation as
// `hi`), no split of X, no Qlo tile -- a third of the tensor work and 60 % of the shared-memory fill.  Its
// approximate distances are coarser (|a - exact| <= 2^-9 |x||q| instead of 2^-13), which the certificate
// accounts for with a larger delta and the host with a larger candidate slack; queries it cannot certify are
// re-run by the PASSES = 3 tier, and only what that cannot certify either goes to the scan.
//
// PASSES = 2 is the HALF tier: the same one-MMA-per-K-step pipeline on an fp16 SHADOW of the rows (kind::f16, K = 16 per
// instruction: twice the products per tensor cycle and per operand byte of kind::tf32, so a pass over the rows costs
// half of PASSES = 1 at the same shared-memory traffic per cycle).  fp16 keeps the same 10 explicit mantissa bits as
// TF32, rounded to nearest instead of truncated, so its approximate distances are TWICE as tight as PASSES = 1's; its
// 5-bit exponent is dealt with by power-of-two scales (one per matrix, one per query) that the epilogue divides out
// exactly.  A K chunk is 64 halves (one 128-byte swizzle row), tiles are the same 16 KB / BN * 128 B.
// per-warp queue of candidate hits (see hitq_flush below): CAP entries, filled and flushed by its warp alone.  The hits
// of one column (= one query) enter together as a GROUP; fc[e] = first entry of e's group << 16 | the group's size.
template <uint32_t CAP>
struct HitQueue {
    uint64_t key[CAP];
    uint32_t q[CAP];
    uint32_t fc[CAP];
    uint32_t gbase[CAP];   // slot the group's first hit got in its query's candidate buffer (indexed by the first entry)
};
constexpr int GEMM_TIER_F16 = 2;
template <int BN, int PASSES = 3>
struct GemmShape {
    static constexpr uint32_t Q_BYTES = BN * GEMM_BK * 4;
    static constexpr uint32_t STAGE_BYTES = PASSES == 3 ? 2 * GEMM_X_BYTES + 2 * Q_BYTES : GEMM_X_BYTES + Q_BYTES;
    static constexpr int STAGES = PASSES == 3 ? (BN == 256 ? 2 : (BN == 128 ? 3 : 4)) : (BN == 256 ? 4 : 6);
    static constexpr uint32_t HITQ = 256;   // queue entries per epilogue warp (4 warps x 5 KB)
    static constexpr uint32_t SMEM_BYTES = 1024 + STAGES * STAGE_BYTES + 5 * BN * 4 + 256 + 4 * sizeof(HitQueue<HITQ>);
    // fp32 accumulate, A and B K-major, M = 128, N = BN; operand format TF32 (kind::tf32) or F16 (kind::f16)
    static constexpr uint32_t FMT = PASSES == GEMM_TIER_F16 ? 0u : 2u;
    static constexpr uint32_t IDESC = (1u << 4) | (FMT << 7) | (FMT << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(GEMM_BM >> 4) << 24);
    static constexpr uint32_t CHUNK_ELEMS = PASSES == GEMM_TIER_F16 ? 64 : 32;   // elements per 128-byte K chunk
};
constexpr float GEMM_DELTA_REL = 1.220703125e-4f;  // 2^-13: bound on |a - exact| / scale (see rerank_kernel), PASSES = 3
// PASSES = 1: both operands truncated to 10 explicit mantissa bits -> |x~q~ - xq| < (2^-9 + 2^-20) |xq|, so the dot
// product is off by < 2^-9 (1 + 2^-11) |x||q| (Cauchy-Schwarz); the products are exact in fp32 and each of the d
// accumulation steps may lose up to 2 ulp of the running sum (tensor cores align and truncate), <= d 2^-22 |x||q|.
// ip / cosine: a = 1 - dot, scale = |x|max |q|.  l2: a = |x|^2 + |q|^2 - 2 dot is off by twice that, and
// 2 |x||q| <= (|x|max + |q|)^2 / 2, so the same bound halves relative to the l2 scale.
__host__ __device__ inline float gemm_delta_rel_1pass(bool l2, uint32_t d) {
    const float e = 1.953125e-3f * (1.0f + 4.8828125e-4f) + (float)d * 2.384185791015625e-7f + 9.5367431640625e-7f;
    return l2 ? 0.5f * e : e;
}
// PASSES = 2 (fp16 shadow): both operands ROUNDED to 11 significant bits -> |x~q~ - xq| <= (2^-10 + 2^-22) |xq|, i.e. the
// dot product is off by <= 2^-10 (1 + 2^-12) |x||q|; elements below the fp16 normal range of the scaled matrix (less than
// 2^-28 of the largest row norm) add at most 2^-25 / scale each, <= 2^-38 sqrt(d) |x|max |q| in total; products of
// halves are exact in fp32 and the accumulation is bounded like the TF32 tier's (fewer, wider steps: the bound is kept).
__host__ __device__ inline float gemm_delta_rel_f16(bool l2, uint32_t d) {
    const float e = 9.765625e-4f * (1.0f + 2.44140625e-4f) + (float)d * 2.384185791015625e-7f + 9.5367431640625e-7f;
    return l2 ? 0.5f * e : e;
}
// The int8 shadow's bound (q8_delta) is in scan_kernel.cuh, next to the kernel that uses it.

struct GemmParams {
    uint32_t n_rows;
    uint32_t row_tile0, row_tile1;  // row tiles [t0, t1) of this round
    uint32_t nq;                    // valid queries (padded ones never pass: thr = -inf)
    uint32_t n_qtiles;
    uint32_t n_kchunks;
    const float* row_norms;  // [n_rows] |x|^2   (l2 only)
    const float* q_norms;    // [nq_pad] |q|^2
    const float* thr;        // [nq_pad] current threshold on the approximate distance
    const uint32_t* live;
    const uint32_t* filter;
    uint64_t* cand;          // [nq_pad][cap]
    uint32_t* cand_cnt;      // [nq_pad]
    uint32_t cap;
    // PASSES = 2: the accumulator holds (x * 2^sx) . (q * 2^sq); dot = acc * *x_unscale * q_unscale[query]
    const float* x_unscale;  // device scalar 2^-sx, frozen when the shadow was converted
    const float* q_unscale;  // [nq_pad] 2^-sq
    int debug;               // profiling only (set_tuning "gemm_debug"): bit 0 = the epilogue drains nothing (results are wrong)
};

// ---- PTX wrappers ---------------------------------------------------------------------------
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, int32_t c0, int32_t c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
            smem_u32(smem_dst)),
        "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_mma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tc_mma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// K-major operand tile, rows of 128 bytes, SWIZZLE_128B (what the TMA box {32 floats, rows} writes):
// 8-row groups are 1024 bytes apart (SBO); LBO is unused for swizzled K-major layouts.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
    uint64_t d = (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;  // descriptor version (sm_100)
    d |= (uint64_t)2 << 61;  // SWIZZLE_128B
    return d;
}

// wait for every tcgen05.ld issued so far; the registers of the load being waited for are in/out operands, so no use
// of them can be scheduled above the wait
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&v)[32]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]), "+r"(v[8]),
                   "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15]), "+r"(v[16]),
                   "+r"(v[17]), "+r"(v[18]), "+r"(v[19]), "+r"(v[20]), "+r"(v[21]), "+r"(v[22]), "+r"(v[23]), "+r"(v[24]),
                   "+r"(v[25]), "+r"(v[26]), "+r"(v[27]), "+r"(v[28]), "+r"(v[29]), "+r"(v[30]), "+r"(v[31])
                 :
                 : "memory");
}
// issue only: the registers are valid after the next tmem_ld_wait()
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}

// One column of the warp's 32 lanes (collective), waited for: the hit path re-reads the few values that passed the pre-test
// instead of keeping the chunk's 32 registers addressable by a run-time index.  The wait also completes any chunk load
// in flight, which is harmless (its own wait then returns at once).
__device__ __forceinline__ uint32_t tmem_ld1_wait(uint32_t taddr) {
    uint32_t v;
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];\n\t"
        "tcgen05.wait::ld.sync.aligned;"
        : "=r"(v)
        : "r"(taddr)
        : "memory");
    return v;
}

// ---- epilogue pieces shared by both GEMM kernels ---------------------------------------------------------------------
// Per query: the threshold test a <= thr solved so that a value costs ONE FFMA and half a three-input max
// (dot = us * v, us the power-of-two unscale of the fp16 tier, 1 otherwise):
//   l2      xn + qn - 2 us v <= thr   <=>   u = v d + e >= xn,   d = 2 us,  e = thr - qn
//   ip      1 - us v <= thr           <=>   u = v d + e >= 0,    d = us,    e = thr - 1
// A lane keeps the running max of u over a 32-column chunk and compares it ONCE with its row's right-hand side; only a
// warp with a passing lane goes on to find the columns.  The chip runs this kernel at its power limit (1000 W, SM
// clocks ~1.35-1.5 GHz; scripts/drain_diag.py), where the epilogue's instructions cost throughput even though they
// overlap the MMAs in time: the previous form (FFMA + FSETP + SEL + LOP3 per value) was 2.3 of 20.7 ms.
// The pre-test is RELAXED by 2^-19 of the magnitudes involved (e upwards, the row's side downwards: 8x the rounding of
// either form), so it never rejects a value the exact test (epilogue_drain) would accept -- the candidate sets are those of
// the plain loop, bit for bit.  Called by the 128 threads (et = 0..127) that are about to drain a tile of query tile
// qt; the caller synchronises them afterwards.  c1_s = e, c2_s = d (d is not read where it is the constant 1 or 2).
template <int METRIC, bool F16, int BN>
__device__ __forceinline__ void epilogue_constants(const GemmParams& p, uint32_t qt, int et, float* thr_s, float* qn_s, float* us_s,
                                                   float* c1_s, float* c2_s) {
    const float xus = F16 ? __ldg(p.x_unscale) : 1.0f;
    for (int i = et; i < BN; i += 128) {
        const float thr = p.thr[qt * BN + i], qn = p.q_norms[qt * BN + i];
        const float us = F16 ? p.q_unscale[qt * BN + i] * xus : 1.0f;   // powers of two: the product is exact
        thr_s[i] = thr;
        qn_s[i] = qn;
        if (F16) us_s[i] = us;
        const bool fin = fabsf(thr) <= 3.0e38f;   // +inf = no threshold yet, -inf = padding query: nothing to relax
        if (METRIC == METRIC_L2) {
            const float e = thr - qn;
            c1_s[i] = fin ? e + 1.9073486328125e-6f * (qn + fabsf(thr)) : e;
            if (F16) c2_s[i] = 2.0f * us;
        } else {
            const float e = thr - 1.0f;
            c1_s[i] = fin ? e + 1.9073486328125e-6f * (1.0f + fabsf(thr)) : e;
            if (F16) c2_s[i] = us;
        }
    }
}

__device__ __forceinline__ float fmax3(float a, float b, float c) {
    float r;
    asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));   // FMNMX3; a NaN operand is ignored
    return r;
}

// One thread = one row (TMEM lane) of a 128 x BN accumulator at taddr0: BN values, 32 per tcgen05.ld, two register
// buffers so the load of chunk c + 1 is in flight while chunk c is tested.
// Hits are queued per warp in shared memory and appended to the queries' candidate buffers a queue at a time: an append
// needs the value its global atomicAdd returns, and waiting ~1000 cycles for that once per hit made the drain 2-3x longer
// than the tile's MMAs.  The queue belongs to its warp alone and the hits of one column are found together (a ballot),
// so the fill count is a warp-uniform REGISTER (no shared-memory atomics) and a column's hits reserve their slots with
// ONE atomicAdd of their number: in the first rounds of a batch (no thresholds yet) every row is a hit, and 32 lanes
// adding 1 to the same counter were serialised by the memory system at ~60 ns each -- 2 us per column, 250 us for a
// single tile (scripts/dense_probe.py).
template <uint32_t CAP>
__device__ __forceinline__ void hitq_flush(const GemmParams& p, HitQueue<CAP>* hq, uint32_t n, int lane) {
    __syncwarp();
#pragma unroll 4
    for (uint32_t i = (uint32_t)lane; i < n; i += 32) {
        const uint32_t fc = hq->fc[i];
        if ((fc >> 16) == i) hq->gbase[i] = atomicAdd(p.cand_cnt + hq->q[i], fc & 0xffffu);
    }
    __syncwarp();
#pragma unroll 4
    for (uint32_t i = (uint32_t)lane; i < n; i += 32) {
        const uint32_t first = hq->fc[i] >> 16;
        const uint32_t pos = hq->gbase[first] + (i - first);
        if (pos < p.cap) p.cand[(size_t)hq->q[i] * p.cap + pos] = hq->key[i];
    }
    __syncwarp();
}

template <int METRIC, bool F16, int BN, uint32_t QCAP>
__device__ __forceinline__ void epilogue_drain(const GemmParams& p, uint32_t taddr0, uint32_t qt, uint32_t row, bool row_ok, float xn,
                                               const float* thr_s, const float* qn_s, const float* us_s, const float* c1_s,
                                               const float* c2_s, HitQueue<QCAP>* hq, uint32_t c_begin = 0, uint32_t c_end = BN / 32) {
    const int lane = threadIdx.x & 31;
    // the row's side of the pre-test; NaN for a row that takes no part (tombstoned, filtered out, beyond the matrix or
    // the round): every comparison with it is false
    const float xr = !row_ok ? __int_as_float(0x7fc00000) : (METRIC == METRIC_L2 ? xn * (1.0f - 1.9073486328125e-6f) : 0.0f);
    // A value that passes the relaxed pre-test is examined with the exact test below.  About one value in a
    // thousand does, i.e. many 32 x 32 warp chunks hold one: walking a lane's 32 registers for its set bits (an unrolled
    // chain of 32 predicated calls -- registers cannot be indexed at run time) cost ~200 issue slots per hit, 4.3 of
    // 24.7 ms on 4M x 768 x 4096 (profiles/r02_drain_diag.jsonl).  Instead the warp walks the UNION of its lanes' bits and
    // re-reads each such column from TMEM (one collective single-column tcgen05.ld): a handful of instructions per hit.
    uint32_t queued = 0;   // entries in this warp's queue (warp-uniform)
    const uint32_t lt_mask = (1u << lane) - 1u;
    auto u_of = [&](uint32_t bits, float d, float e) -> float {
        const float v = __uint_as_float(bits);
        if (F16) return fmaf(v, d, e);
        return METRIC == METRIC_L2 ? fmaf(v, 2.0f, e) : v + e;
    };
    const bool drain_off = p.debug & 1;   // profiling: TMEM loads only
    auto process = [&](const uint32_t(&v)[32], uint32_t c) {
        if (drain_off) return;
        const float4* ke = reinterpret_cast<const float4*>(c1_s + c * 32);
        const float4* kd = reinterpret_cast<const float4*>(c2_s + c * 32);
        float mx = __int_as_float(0xff800000);
#pragma unroll
        for (int j4 = 0; j4 < 8; j4++) {
            const float4 e = ke[j4];
            const float4 d = F16 ? kd[j4] : make_float4(0.f, 0.f, 0.f, 0.f);
            mx = fmax3(mx, u_of(v[4 * j4], d.x, e.x), u_of(v[4 * j4 + 1], d.y, e.y));
            mx = fmax3(mx, u_of(v[4 * j4 + 2], d.z, e.z), u_of(v[4 * j4 + 3], d.w, e.w));
        }
        if (!__any_sync(0xffffffffu, mx >= xr)) return;   // warp-uniform
        // some lane holds a value that passes: one bit per column (the same arithmetic as above, so the same verdicts)
        uint32_t m = 0;
#pragma unroll
        for (int j4 = 0; j4 < 8; j4++) {
            const float4 e = ke[j4];
            const float4 d = F16 ? kd[j4] : make_float4(0.f, 0.f, 0.f, 0.f);
            m |= u_of(v[4 * j4], d.x, e.x) >= xr ? 1u << (4 * j4) : 0u;
            m |= u_of(v[4 * j4 + 1], d.y, e.y) >= xr ? 2u << (4 * j4) : 0u;
            m |= u_of(v[4 * j4 + 2], d.z, e.z) >= xr ? 4u << (4 * j4) : 0u;
            m |= u_of(v[4 * j4 + 3], d.w, e.w) >= xr ? 8u << (4 * j4) : 0u;
        }
        uint32_t rest = __reduce_or_sync(0xffffffffu, m);   // warp-uniform
        while (rest) {
            const uint32_t j = (uint32_t)__ffs((int)rest) - 1u;
            rest &= rest - 1u;
            const uint32_t ql = c * 32 + j;
            const float vj = __uint_as_float(tmem_ld1_wait(taddr0 + ql));
            // the exact test, in the arithmetic the thresholds were made in
            const float dot = F16 ? vj * us_s[ql] : vj;
            const float a = (METRIC == METRIC_L2) ? fmaf(-2.0f, dot, xn + qn_s[ql]) : 1.0f - dot;
            const bool h = ((m >> j) & 1u) && (a <= thr_s[ql]);
            const uint32_t hb = __ballot_sync(0xffffffffu, h);
            if (hb == 0) continue;
            if (queued + 32 > QCAP) {
                hitq_flush<QCAP>(p, hq, queued, lane);
                queued = 0;
            }
            const uint32_t nh = (uint32_t)__popc(hb);
            if (h) {
                const uint32_t slot = queued + __popc(hb & lt_mask);
                hq->key[slot] = make_key(a, row);
                hq->q[slot] = qt * BN + ql;
                hq->fc[slot] = (queued << 16) | nh;
            }
            queued += nh;
        }
    };
    uint32_t va[32], vb[32];
    tmem_ld32_issue(taddr0 + c_begin * 32, va);
    for (uint32_t c = c_begin; c < c_end; c += 2) {   // an even number of 32-column chunks
        tmem_ld_wait(va);
        tmem_ld32_issue(taddr0 + (c + 1) * 32, vb);
        process(va, c);
        tmem_ld_wait(vb);
        if (c + 2 < c_end) tmem_ld32_issue(taddr0 + (c + 2) * 32, va);
        process(vb, c + 1);
    }
    if (queued) hitq_flush<QCAP>(p, hq, queued, lane);
}

// ---- the GEMM + candidate-selection kernel ---------------------------------------------------
template <int METRIC, int GEMM_BN, int PASSES>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_topk_kernel(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_qhi,
                 const __grid_constant__ CUtensorMap tm_qlo, const GemmParams p) {
    constexpr int GEMM_STAGES = GemmShape<GEMM_BN, PASSES>::STAGES;
    constexpr uint32_t GEMM_Q_BYTES = GemmShape<GEMM_BN, PASSES>::Q_BYTES;
    constexpr uint32_t GEMM_STAGE_BYTES = GemmShape<GEMM_BN, PASSES>::STAGE_BYTES;
    constexpr uint32_t GEMM_IDESC = GemmShape<GEMM_BN, PASSES>::IDESC;
    // stage layout: PASSES = 3: Xhi | Xlo | Qhi | Qlo;  PASSES = 1: X | Q
    constexpr uint32_t GEMM_Q_OFF = PASSES == 3 ? 2 * GEMM_X_BYTES : GEMM_X_BYTES;
    extern __shared__ unsigned char gemm_smem_raw[];
    // SWIZZLE_128B tiles need 1024-byte alignment
    unsigned char* smem = gemm_smem_raw + ((1024u - (smem_u32(gemm_smem_raw) & 1023u)) & 1023u);
    constexpr bool F16 = PASSES == GEMM_TIER_F16;
    constexpr uint32_t CHUNK_ELEMS = GemmShape<GEMM_BN, PASSES>::CHUNK_ELEMS;
    float* thr_s = reinterpret_cast<float*>(smem + GEMM_STAGES * GEMM_STAGE_BYTES);  // [256]
    float* qn_s = thr_s + GEMM_BN;                                                    // [256]
    float* us_s = qn_s + GEMM_BN;                                                     // [256] (PASSES = 2)
    float* c1_s = us_s + GEMM_BN;                                                     // [256] pre-test constants
    float* c2_s = c1_s + GEMM_BN;                                                     // [256]
    uint64_t* bars = reinterpret_cast<uint64_t*>(c2_s + GEMM_BN);
    uint64_t* full = bars;                      // [S]  TMA bytes landed
    uint64_t* empty = bars + GEMM_STAGES;       // [S]  MMAs reading the stage retired
    uint64_t* conv = bars + 2 * GEMM_STAGES;    // [S]  hi/lo split written
    uint64_t* tfull = bars + 3 * GEMM_STAGES;   // [2]  accumulator complete
    uint64_t* tempty = tfull + 2;               // [2]  accumulator drained
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
    using HitQ = HitQueue<GemmShape<GEMM_BN, PASSES>::HITQ>;
    HitQ* hqs = reinterpret_cast<HitQ*>(reinterpret_cast<unsigned char*>(bars) + 256);   // [4] one per epilogue warp

    const int tid = threadIdx.x;
    const int warp = tid >> 5;
    const int lane = tid & 31;

    if (tid == 0) {
        for (int s = 0; s < GEMM_STAGES; s++) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 1);
            mbar_init(&conv[s], 4);
        }
        for (int a = 0; a < 2; a++) {
            mbar_init(&tfull[a], 1);
            mbar_init(&tempty[a], 4);
        }
        mbar_fence_init();
        tma_prefetch_desc(&tm_x);
        tma_prefetch_desc(&tm_qhi);
        tma_prefetch_desc(&tm_qlo);
    }
    if (warp == 1) {  // whole warp: allocate all 512 TMEM columns (two 128 x 256 fp32 accumulators)
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    const uint32_t n_items = (p.row_tile1 - p.row_tile0) * p.n_qtiles;

    if (warp == 0) {
        // ------------------------------------------------------------------ TMA producer
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            for (uint32_t it = blockIdx.x; it < n_items; it += gridDim.x) {
                const uint32_t rt = p.row_tile0 + it / p.n_qtiles, qt = it % p.n_qtiles;
                for (uint32_t kc = 0; kc < p.n_kchunks; kc++) {
                    mbar_wait(&empty[stage], phase ^ 1);
                    unsigned char* sb = smem + (size_t)stage * GEMM_STAGE_BYTES;
                    mbar_arrive_expect_tx(&full[stage], GEMM_X_BYTES + (PASSES == 3 ? 2 : 1) * GEMM_Q_BYTES);
                    tma_load_2d(sb, &tm_x, (int32_t)(kc * CHUNK_ELEMS), (int32_t)(rt * GEMM_BM), &full[stage]);
                    tma_load_2d(sb + GEMM_Q_OFF, &tm_qhi, (int32_t)(kc * CHUNK_ELEMS), (int32_t)(qt * GEMM_BN), &full[stage]);
                    if (PASSES == 3)
                        tma_load_2d(sb + GEMM_Q_OFF + GEMM_Q_BYTES, &tm_qlo, (int32_t)(kc * CHUNK_ELEMS), (int32_t)(qt * GEMM_BN),
                                    &full[stage]);
                    if (++stage == GEMM_STAGES) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer
        if (lane == 0) {
            uint32_t stage = 0, phase = 0, local = 0;
            for (uint32_t it = blockIdx.x; it < n_items; it += gridDim.x, local++) {
                const uint32_t acc = local & 1, acc_phase = (local >> 1) & 1;
                mbar_wait(&tempty[acc], acc_phase ^ 1);
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + acc * GEMM_BN;
                for (uint32_t kc = 0; kc < p.n_kchunks; kc++) {
                    mbar_wait(&full[stage], phase);
                    if (PASSES == 3) mbar_wait(&conv[stage], phase);
                    tc_fence_after();
                    const uint32_t sb = smem_u32(smem + (size_t)stage * GEMM_STAGE_BYTES);
                    const uint64_t d_xhi = umma_desc_sw128(sb);
                    const uint64_t d_xlo = umma_desc_sw128(sb + GEMM_X_BYTES);
                    const uint64_t d_qhi = umma_desc_sw128(sb + GEMM_Q_OFF);
                    const uint64_t d_qlo = umma_desc_sw128(sb + GEMM_Q_OFF + GEMM_Q_BYTES);
#pragma unroll
                    for (uint32_t ks = 0; ks < GEMM_BK / 8; ks++) {
                        const uint64_t adv = (uint64_t)(ks * 2);  // 8 floats = 32 bytes = 2 x 16-byte units
                        if (PASSES == 3) {
                            // small terms first, the dominant hi.hi product last
                            tc_mma_tf32(tmem_d, d_xlo + adv, d_qhi + adv, GEMM_IDESC, (kc | ks) != 0);
                            tc_mma_tf32(tmem_d, d_xhi + adv, d_qlo + adv, GEMM_IDESC, 1);
                            tc_mma_tf32(tmem_d, d_xhi + adv, d_qhi + adv, GEMM_IDESC, 1);
                        } else if (F16) {
                            // fp16 shadow tiles: 16 halves (the same 32 bytes) per instruction
                            tc_mma_f16(tmem_d, d_xhi + adv, d_qhi + adv, GEMM_IDESC, (kc | ks) != 0);
                        } else {
                            // raw fp32 tiles: the tensor core truncates both operands to TF32 itself
                            tc_mma_tf32(tmem_d, d_xhi + adv, d_qhi + adv, GEMM_IDESC, (kc | ks) != 0);
                        }
                    }
                    tc_commit(&empty[stage]);  // stage reusable once these MMAs have read it
                    if (++stage == GEMM_STAGES) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
                tc_commit(&tfull[acc]);
            }
        }
    } else if (warp < 6) {
        // ------------------------------------------------------------------ hi/lo split of X (PASSES = 3 only)
        const int ct = tid - 64;  // 0..127
        uint32_t stage = 0, phase = 0;
        for (uint32_t it = blockIdx.x; PASSES == 3 && it < n_items; it += gridDim.x) {
            for (uint32_t kc = 0; kc < p.n_kchunks; kc++) {
                mbar_wait(&full[stage], phase);
                uint4* xh = reinterpret_cast<uint4*>(smem + (size_t)stage * GEMM_STAGE_BYTES);
                float4* xl = reinterpret_cast<float4*>(smem + (size_t)stage * GEMM_STAGE_BYTES + GEMM_X_BYTES);
#pragma unroll
                for (int i = 0; i < (int)(GEMM_X_BYTES / 16 / 128); i++) {
                    const int idx = ct + 128 * i;
                    const uint4 v = xh[idx];
                    uint4 hi;
                    hi.x = v.x & 0xFFFFE000u;
                    hi.y = v.y & 0xFFFFE000u;
                    hi.z = v.z & 0xFFFFE000u;
                    hi.w = v.w & 0xFFFFE000u;
                    float4 lo;
                    lo.x = __uint_as_float(v.x) - __uint_as_float(hi.x);
                    lo.y = __uint_as_float(v.y) - __uint_as_float(hi.y);
                    lo.z = __uint_as_float(v.z) - __uint_as_float(hi.z);
                    lo.w = __uint_as_float(v.w) - __uint_as_float(hi.w);
                    xh[idx] = hi;
                    xl[idx] = lo;
                }
                fence_proxy_async_smem();  // generic-proxy writes -> visible to the tensor core's async proxy
                __syncwarp();
                if (lane == 0) mbar_arrive(&conv[stage]);
                if (++stage == GEMM_STAGES) {
                    stage = 0;
                    phase ^= 1;
                }
            }
        }
    } else {
        // ------------------------------------------------------------------ epilogue
        const int et = tid - 192;        // 0..127
        const uint32_t quarter = warp & 3;  // TMEM lanes this warp may read: 32*quarter .. +31
        HitQ* hq = hqs + (warp - 6);
        uint32_t local = 0;
        for (uint32_t it = blockIdx.x; it < n_items; it += gridDim.x, local++) {
            const uint32_t rt = p.row_tile0 + it / p.n_qtiles, qt = it % p.n_qtiles;
            const uint32_t acc = local & 1, acc_phase = (local >> 1) & 1;
            named_bar_sync(2, 128);  // everyone finished reading thr_s / qn_s of the previous item
            epilogue_constants<METRIC, F16, GEMM_BN>(p, qt, et, thr_s, qn_s, us_s, c1_s, c2_s);
            const uint32_t row = rt * GEMM_BM + quarter * 32 + lane;
            bool row_ok = row < p.n_rows && !(p.debug & 1);
            float xn = 0.f;
            if (row_ok) {
                if (p.live) row_ok = (__ldg(p.live + (row >> 5)) >> (row & 31)) & 1u;
                if (row_ok && p.filter) row_ok = (__ldg(p.filter + (row >> 5)) >> (row & 31)) & 1u;
                if (METRIC == METRIC_L2 && row_ok) xn = __ldg(p.row_norms + row);
            }
            named_bar_sync(2, 128);
            mbar_wait(&tfull[acc], acc_phase);
            tc_fence_after();
            const uint32_t taddr0 = tmem_base + ((quarter * 32u) << 16) + acc * GEMM_BN;
            epilogue_drain<METRIC, F16, GEMM_BN, GemmShape<GEMM_BN, PASSES>::HITQ>(p, taddr0, qt, row, row_ok, xn, thr_s, qn_s, us_s, c1_s, c2_s, hq);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty[acc]);
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// (A "wide" single-CTA kernel -- two row tiles per staged query tile, 16 drain warps, optionally clusters of two sharing the
// query tile by TMA multicast -- lived here during round 2: 57.5k q/s on config 3 against the CTA-pair kernel's 65 - 70k on
// every shape measured, and its 576 threads left the rewritten epilogue 130 bytes of spills.  Removed; the numbers are in
// profiles/README.md.)

__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}

// ---- the CTA-pair one-pass kernel (tcgen05 cta_group::2) ----------------------------------------------------------
// What bounds the one-pass tiers once the epilogue is cheap is the rate at which operand bytes ENTER an SM (~43 B/clk each
// when all 148 pull from L2; r02 ncu: xbar2l1tex 11.2 TB/s whatever the kernel): a 128 x 256 tile per SM needs 96 B/clk at
// full tensor rate, two row tiles per query tile 64 B/clk.  A CTA pair shares the B operand inside the tensor cores: the
// pair computes D[256 x 256] per instruction, each SM holds its own 128 rows of X and only HALF of the query tile, so an
// SM takes in (128 + 128) operand rows for its 128 x 256 products -- 64 B/clk with the accumulators still double-buffered
// (the drain overlaps the next tile's MMAs), against 96 B/clk for gemm_topk_kernel.
// 320 threads per CTA: warp 0 TMA producer (both CTAs; every load completes on the LEADER's barrier) | warp 1 MMA issuer
// (leader CTA only) | warps 2-9 epilogue (two warps per TMEM lane quarter, 128 columns each).
constexpr int GEMMP_BN = 256;
constexpr int GEMMP_STAGES = 6;
constexpr uint32_t GEMMP_QH_BYTES = (GEMMP_BN / 2) * GEMM_BK * 4;            // this CTA's half of the query tile: 16 KB
constexpr uint32_t GEMMP_STAGE_BYTES = GEMM_X_BYTES + GEMMP_QH_BYTES;          // 32 KB
constexpr uint32_t GEMMP_HITQ = 176;   // 8 warps x 3.4 KB
constexpr uint32_t GEMMP_SMEM_BYTES = 1024 + GEMMP_STAGES * GEMMP_STAGE_BYTES + 5 * GEMMP_BN * 4 + 256 + 8 * sizeof(HitQueue<GEMMP_HITQ>);

__device__ __forceinline__ uint32_t mapa_shared(uint32_t local_addr, uint32_t cta_rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(cta_rank));
    return r;
}
// 2-D tile load of a CTA pair: the bytes land in THIS CTA's shared memory, the transaction count on `bar_cluster_addr`
// (a shared::cluster address: the leader's barrier)
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* map, int32_t c0, int32_t c1, uint32_t bar_cluster_addr) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
            smem_u32(smem_dst)),
        "l"(map), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tc_commit_pair(uint64_t* bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
                 "h"(mask)
                 : "memory");
}
__device__ __forceinline__ void tc_mma_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate, bool f16) {
    if (f16)
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "setp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
            "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
            : "memory");
    else
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "setp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
            "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
            : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar_cluster_addr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(bar_cluster_addr) : "memory");
}

template <int METRIC, int PASSES>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_topk_pair_kernel(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_q, const GemmParams p) {
    static_assert(PASSES == 1 || PASSES == GEMM_TIER_F16, "one-pass tiers only");
    constexpr bool F16 = PASSES == GEMM_TIER_F16;
    constexpr uint32_t CHUNK_ELEMS = F16 ? 64 : 32;
    // fp32 accumulate, K-major operands, M = 256 (the pair), N = 256
    constexpr uint32_t FMT = F16 ? 0u : 2u;
    constexpr uint32_t IDESC = (1u << 4) | (FMT << 7) | (FMT << 10) | ((uint32_t)(GEMMP_BN >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
    extern __shared__ unsigned char gemm_smem_raw[];
    unsigned char* smem = gemm_smem_raw + ((1024u - (smem_u32(gemm_smem_raw) & 1023u)) & 1023u);
    float* thr_s = reinterpret_cast<float*>(smem + GEMMP_STAGES * GEMMP_STAGE_BYTES);
    float* qn_s = thr_s + GEMMP_BN;
    float* us_s = qn_s + GEMMP_BN;
    float* c1_s = us_s + GEMMP_BN;
    float* c2_s = c1_s + GEMMP_BN;
    uint64_t* bars = reinterpret_cast<uint64_t*>(c2_s + GEMMP_BN);
    uint64_t* full = bars;                       // [S]  leader only: both CTAs' loads of the stage have landed
    uint64_t* empty = bars + GEMMP_STAGES;       // [S]  both CTAs: the pair's MMAs reading the stage have retired
    uint64_t* tfull = bars + 2 * GEMMP_STAGES;   // [2]  both CTAs: accumulator complete
    uint64_t* tempty = tfull + 2;                // [2]  leader only: accumulator drained by both CTAs' epilogue warps
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
    using HitQ = HitQueue<GEMMP_HITQ>;
    HitQ* hqs = reinterpret_cast<HitQ*>(reinterpret_cast<unsigned char*>(bars) + 256);   // [8] one per epilogue warp

    const int tid = threadIdx.x;
    const int warp = tid >> 5;
    const int lane = tid & 31;
    const uint32_t crank = cluster_ctarank();
    const bool leader = crank == 0;

    if (tid == 0) {
        for (int s = 0; s < GEMMP_STAGES; s++) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 1);
        }
        for (int a = 0; a < 2; a++) {
            mbar_init(&tfull[a], 1);
            mbar_init(&tempty[a], 16);   // 8 epilogue warps in each of the two CTAs
        }
        mbar_fence_init();
        tma_prefetch_desc(&tm_x);
        tma_prefetch_desc(&tm_q);
    }
    if (warp == 1) {   // one warp of EACH CTA: the pair's allocation (same columns in both tensor memories)
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();   // both CTAs' barriers exist before any load / commit / arrive crosses over
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    // items: (pair of consecutive row tiles) x (query tile); CTA `crank` of the pair owns row tile 2 * grp + crank
    const uint32_t tiles = p.row_tile1 - p.row_tile0;
    const uint32_t n_items = ((tiles + 1) / 2) * p.n_qtiles;
    const uint32_t pair_id = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;

    if (warp == 0) {
        // ------------------------------------------------------------------ TMA producer (both CTAs)
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            for (uint32_t it = pair_id; it < n_items; it += n_pairs) {
                const uint32_t grp = it / p.n_qtiles, qt = it % p.n_qtiles;
                const uint32_t rt = p.row_tile0 + grp * 2 + crank;
                for (uint32_t kc = 0; kc < p.n_kchunks; kc++) {
                    mbar_wait(&empty[stage], phase ^ 1);
                    unsigned char* sb = smem + (size_t)stage * GEMMP_STAGE_BYTES;
                    const uint32_t lead_full = mapa_shared(smem_u32(&full[stage]), 0);
                    if (leader) mbar_arrive_expect_tx(&full[stage], 2 * GEMMP_STAGE_BYTES);   // this CTA's bytes and the peer's
                    tma_load_2d_pair(sb, &tm_x, (int32_t)(kc * CHUNK_ELEMS), (int32_t)(rt * GEMM_BM), lead_full);
                    tma_load_2d_pair(sb + GEMM_X_BYTES, &tm_q, (int32_t)(kc * CHUNK_ELEMS),
                                     (int32_t)(qt * GEMMP_BN + crank * (GEMMP_BN / 2)), lead_full);
                    if (++stage == GEMMP_STAGES) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer (leader CTA, one thread, for both SMs)
        if (leader && lane == 0) {
            uint32_t stage = 0, phase = 0, local = 0;
            for (uint32_t it = pair_id; it < n_items; it += n_pairs, local++) {
                const uint32_t acc = local & 1, acc_phase = (local >> 1) & 1;
                mbar_wait(&tempty[acc], acc_phase ^ 1);
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + acc * GEMMP_BN;
                for (uint32_t kc = 0; kc < p.n_kchunks; kc++) {
                    mbar_wait(&full[stage], phase);
                    tc_fence_after();
                    const uint32_t sb = smem_u32(smem + (size_t)stage * GEMMP_STAGE_BYTES);
                    const uint64_t d_x = umma_desc_sw128(sb), d_q = umma_desc_sw128(sb + GEMM_X_BYTES);
#pragma unroll
                    for (uint32_t ks = 0; ks < GEMM_BK / 8; ks++) {
                        const uint64_t adv = (uint64_t)(ks * 2);
                        tc_mma_pair(tmem_d, d_x + adv, d_q + adv, IDESC, (kc | ks) != 0, F16);
                    }
                    tc_commit_pair(&empty[stage], 3);   // the stage is free again in both CTAs
                    if (++stage == GEMMP_STAGES) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
                tc_commit_pair(&tfull[acc], 3);          // both CTAs' epilogue warps may drain their 128 rows
            }
        }
    } else {
        // ------------------------------------------------------------------ epilogue (both CTAs): 8 warps, 128 rows x 256 queries
        const int et = tid - 64;            // 0..255
        const uint32_t half = ((uint32_t)(warp - 2) >> 2) & 1u;
        const uint32_t quarter = warp & 3;
        HitQ* hq = hqs + (warp - 2);
        uint32_t local = 0;
        for (uint32_t it = pair_id; it < n_items; it += n_pairs, local++) {
            const uint32_t grp = it / p.n_qtiles, qt = it % p.n_qtiles;
            const uint32_t tile = p.row_tile0 + grp * 2 + crank;
            const uint32_t acc = local & 1, acc_phase = (local >> 1) & 1;
            named_bar_sync(2, 256);
            if (et < 128) epilogue_constants<METRIC, F16, GEMMP_BN>(p, qt, et, thr_s, qn_s, us_s, c1_s, c2_s);
            const uint32_t row = tile * GEMM_BM + quarter * 32 + lane;
            bool row_ok = tile < p.row_tile1 && row < p.n_rows && !(p.debug & 1);
            float xn = 0.f;
            if (row_ok) {
                if (p.live) row_ok = (__ldg(p.live + (row >> 5)) >> (row & 31)) & 1u;
                if (row_ok && p.filter) row_ok = (__ldg(p.filter + (row >> 5)) >> (row & 31)) & 1u;
                if (METRIC == METRIC_L2 && row_ok) xn = __ldg(p.row_norms + row);
            }
            named_bar_sync(2, 256);
            mbar_wait(&tfull[acc], acc_phase);
            tc_fence_after();
            const uint32_t taddr0 = tmem_base + ((quarter * 32u) << 16) + acc * GEMMP_BN;
            epilogue_drain<METRIC, F16, GEMMP_BN, GEMMP_HITQ>(p, taddr0, qt, row, row_ok, xn, thr_s, qn_s, us_s, c1_s, c2_s, hq, half * (GEMMP_BN / 64),
                                                  (half + 1) * (GEMMP_BN / 64));
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(mapa_shared(smem_u32(&tempty[acc]), 0));   // the leader's barrier
        }
    }

    tc_fence_before();
    __syncthreads();
    cluster_sync_all();   // nobody leaves while the peer may still load, commit or arrive across
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// ---- helpers around the GEMM -------------------------------------------------------------------
// dense copy of the listed rows (one warp per row) and of their squared norms: the matrix a filtered batch multiplies
__global__ void gather_rows_kernel(const float4* __restrict__ src, const uint32_t* __restrict__ list, uint32_t m, uint32_t ld4,
                                   float4* __restrict__ dst, const float* __restrict__ norms, float* __restrict__ out_norms) {
    const uint32_t w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (w >= m) return;
    const uint32_t r = list[w];
    for (uint32_t j = lane; j < ld4; j += 32) dst[(size_t)w * ld4 + j] = src[(size_t)r * ld4 + j];
    if (lane == 0 && norms) out_norms[w] = norms[r];
}
// second tier works on the queries the first could not certify: dst[i] = src[idx[i]] (rows of ld floats)
__global__ void gather_queries_kernel(const float* __restrict__ src, const uint32_t* __restrict__ idx, float* __restrict__ dst,
                                      uint32_t n, uint32_t ld) {
    const uint32_t total = n * ld;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const uint32_t r = i / ld;
        dst[i] = src[(size_t)idx[r] * ld + (i - r * ld)];
    }
}
// ... and its results go back to the queries' own slots: dst[idx[i]] = src[i]
__global__ void scatter_results_kernel(const uint32_t* __restrict__ idx, uint32_t n, uint32_t k, const float* __restrict__ sd,
                                       const int64_t* __restrict__ sr, const int32_t* __restrict__ sc, float* __restrict__ dd,
                                       int64_t* __restrict__ dr, int32_t* __restrict__ dc) {
    const uint32_t total = n * k;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const uint32_t r = i / k, j = i - r * k;
        const size_t o = (size_t)idx[r] * k + j;
        dd[o] = sd[i];
        dr[o] = sr[i];
        if (j == 0) dc[idx[r]] = sc[r];
    }
}

// ---- fp16 shadow of the rows (PASSES = 2) ---------------------------------------------------------
// st[0] = 2^-s (float, what the epilogue multiplies by), st[1] = s (int), st[2] = overflow flag (cleared).
// max_norm2_bits == nullptr: unit rows (cosine).
__global__ void f16_freeze_scale_kernel(const uint32_t* max_norm2_bits, uint32_t* st) {
    const float xmax = max_norm2_bits ? sqrtf(__uint_as_float(*max_norm2_bits)) : 1.0f;
    const int s = f16_scale_exp(xmax);
    st[0] = __float_as_uint(ldexpf(1.0f, -s));
    st[1] = (uint32_t)s;
    st[2] = 0;
}
// rows [first, first + n) of the fp32 matrix -> halves (round to nearest) of value * 2^s, ld16 halves per row (zero padded).
// A value the frozen scale cannot hold (rows much larger than any present when it was frozen) raises st[2].
__global__ void convert_rows_f16_kernel(const float* __restrict__ rows, uint64_t first, uint64_t n, uint32_t ld, uint32_t ld16,
                                        __half* __restrict__ out, uint32_t* st) {
    const float scale = ldexpf(1.0f, (int)st[1]);
    const uint32_t pairs = ld16 >> 1;
    const uint64_t total = n * pairs;
    bool over = false;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t r = i / pairs;
        const uint32_t c = (uint32_t)(i - r * pairs) * 2;
        const float* src = rows + (first + r) * ld;
        const float a = c < ld ? src[c] * scale : 0.f, b = c + 1 < ld ? src[c + 1] * scale : 0.f;
        over |= fabsf(a) > 65000.f || fabsf(b) > 65000.f;
        reinterpret_cast<__half2*>(out + (first + r) * ld16)[c >> 1] = __floats2half2_rn(a, b);
    }
    if (over) st[2] = 1;
}
// ---- int8 shadow of the rows (scan_kernel_q8, see q8_delta in scan_kernel.cuh) ------------------------------------
// rows [first, first + n) -> int8 digits x^ = rint(x / s_x) with s_x = max |x| / 127 (one scale per row, so appended rows
// cannot overflow), ld8 bytes per row (zero padded).  sx[row] = s_x; *e_bits = max over the rows of e_x >= |x - s_x x^|_2
// (float bits: non-negative floats order as uints, a NaN row wins and leaves every query uncertified).  One warp per row.
__global__ void convert_rows_q8_kernel(const float* __restrict__ rows, uint64_t first, uint64_t n, uint32_t ld, uint32_t ld8,
                                       int8_t* __restrict__ out, float* __restrict__ sx, uint32_t* e_bits) {
    const uint64_t w = (uint64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (w >= n) return;
    const float4* src = reinterpret_cast<const float4*>(rows + (first + w) * ld);
    const uint32_t ld4 = ld >> 2;
    float m = 0.f;
    for (uint32_t j = lane; j < ld4; j += 32) {
        const float4 x = src[j];
        m = fmaxf(m, fmaxf(fmaxf(fabsf(x.x), fabsf(x.y)), fmaxf(fabsf(x.z), fabsf(x.w))));
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, off));
    const float s = m / 127.0f;
    const float inv = m > 0.f ? 127.0f / m : 0.f;
    uint32_t* dst = reinterpret_cast<uint32_t*>(out + (first + w) * ld8);
    float ss = 0.f;
    for (uint32_t j = lane; j < ld8 / 4; j += 32) {
        const float4 x = j < ld4 ? src[j] : make_float4(0.f, 0.f, 0.f, 0.f);
        const float v[4] = {x.x, x.y, x.z, x.w};
        uint32_t packed = 0;
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const float dq = fminf(fmaxf(rintf(v[i] * inv), -127.f), 127.f);
            const float r = fmaf(-s, dq, v[i]);
            ss = fmaf(r, r, ss);
            packed |= ((uint32_t)(int32_t)dq & 0xffu) << (8 * i);
        }
        dst[j] = packed;
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, off);
    if (lane == 0) {
        // rounded up: each residual is one fma (relative 2^-24), the fp32 sum of ld squares is off by <= ld 2^-23 of itself,
        // squares below the normal range add < 2^-60 in total
        const float e = sqrtf(ss) * (1.0f + (float)(ld + 4) * 2.384185791015625e-7f) + 8.673617379884035e-19f;
        sx[first + w] = s;
        atomicMax(e_bits, __float_as_uint(e));
    }
}
// Prepared queries [nq, ld] -> halves of q * 2^sq [nq_pad, ld16] (pad rows / columns zero), 2^-sq, |q|^2, initial thresholds,
// cleared counters and flags.  One warp per (padded) query.
__global__ void split_queries_f16_kernel(const float* __restrict__ q, __half* __restrict__ q16, float* __restrict__ unscale,
                                         float* __restrict__ qn, float* __restrict__ thr, uint32_t* __restrict__ cnt,
                                         uint32_t* __restrict__ flags, uint32_t* __restrict__ sorted_n, uint32_t nq, uint32_t nq_pad,
                                         uint32_t ld, uint32_t ld16) {
    const uint32_t w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (w >= nq_pad) return;
    float s = 0.f, m = 0.f;
    for (uint32_t j = lane; j < ld; j += 32) {
        const float v = w < nq ? q[(size_t)w * ld + j] : 0.f;
        s = fmaf(v, v, s);
        m = fmaxf(m, fabsf(v));
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, off);
        m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, off));
    }
    const int sq = f16_scale_exp(m);
    const float scale = ldexpf(1.0f, sq);
    for (uint32_t j = lane; j < ld16; j += 32)
        q16[(size_t)w * ld16 + j] = __float2half_rn((w < nq && j < ld) ? q[(size_t)w * ld + j] * scale : 0.f);
    if (lane == 0) {
        unscale[w] = ldexpf(1.0f, -sq);
        qn[w] = s;
        thr[w] = w < nq ? __int_as_float(0x7f800000) : __int_as_float(0xff800000);
        cnt[w] = 0;
        flags[w] = 0;
        sorted_n[w] = 0;
    }
}

// |x|^2 per row (one warp per row) and the running maximum (non-negative floats order as uints).
__global__ void row_norms_kernel(const float* __restrict__ rows, uint64_t first, uint64_t n, uint32_t ld, float* norms,
                                 uint32_t* max_norm2_bits) {
    const uint64_t w = (uint64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (w >= n) return;
    const float4* r = reinterpret_cast<const float4*>(rows + (first + w) * ld);
    const uint32_t ld4 = ld >> 2;
    float s = 0.f;
    for (uint32_t j = lane; j < ld4; j += 32) {
        const float4 x = r[j];
        s = fmaf(x.x, x.x, s);
        s = fmaf(x.y, x.y, s);
        s = fmaf(x.z, x.z, s);
        s = fmaf(x.w, x.w, s);
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
    if (lane == 0) {
        norms[first + w] = s;
        if (s == s) atomicMax(max_norm2_bits, __float_as_uint(s));
    }
}

// Prepared queries [nq, ld] -> Qhi / Qlo [nq_pad, ld] (pad rows zero), |q|^2, initial thresholds,
// cleared candidate counters and flags.  One warp per (padded) query.
__global__ void split_queries_kernel(const float* __restrict__ q, float* __restrict__ qhi, float* __restrict__ qlo,
                                     float* __restrict__ qn, float* __restrict__ thr, uint32_t* __restrict__ cnt,
                                     uint32_t* __restrict__ flags, uint32_t* __restrict__ sorted_n, uint32_t nq, uint32_t nq_pad, uint32_t ld) {
    const uint32_t w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (w >= nq_pad) return;
    float s = 0.f;
    for (uint32_t j = lane; j < ld; j += 32) {
        const float v = w < nq ? q[(size_t)w * ld + j] : 0.f;
        const float hi = __uint_as_float(__float_as_uint(v) & 0xFFFFE000u);
        qhi[(size_t)w * ld + j] = hi;
        qlo[(size_t)w * ld + j] = v - hi;
        s = fmaf(v, v, s);
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
    if (lane == 0) {
        qn[w] = s;
        thr[w] = w < nq ? __int_as_float(0x7f800000) : __int_as_float(0xff800000);
        cnt[w] = 0;
        flags[w] = 0;
        sorted_n[w] = 0;
    }
}

// After a round: keep the kprime smallest keys of each query's buffer and tighten its threshold to the jrank-th smallest.
// jrank == kprime is the plain rule (a threshold no tighter than the k'-th best seen can never lose a top-k' row).
// jrank < kprime PREDICTS the final k'-th best from the rows seen so far -- with S of N rows seen, the jrank-th best of S
// sits where about jrank N / S rows of the whole matrix will, and the host keeps that at 4 k' or more -- so later rounds
// append a fraction of the hits.  A prediction can be wrong (rows stored in an order that correlates with the query):
// the last round's refine (final != 0) checks it -- k' candidates at or below the tightest threshold any round used,
// which makes the kept k' exactly the k' best of ALL rows -- and sets flags[q] bit 2 otherwise (the query is answered by
// the next tier, whose thresholds are the plain rule).  Thresholds only tighten (min), so the last one is the tightest.
// flags[q] bit 0 = the buffer overflowed (candidates were lost: the query falls back as well).
// The first sorted_n[q] slots are what the previous refine kept -- already ascending -- so only the round's NEW hits are
// sorted (a bitonic network in shared memory is bound by shared-memory bandwidth: 4096 queries x 1024 keys cost 190 us
// per round) and the two ascending lists are merged by rank (binary search).  Shared memory: P + kprime keys.
__global__ void __launch_bounds__(SELECT_THREADS, 1)
refine_kernel(uint64_t* cand, uint32_t* cnt, float* thr, uint32_t* flags, uint32_t* sorted_n, uint32_t cap, uint32_t P, uint32_t kprime,
              uint32_t jrank, int final) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint64_t* a = reinterpret_cast<uint64_t*>(smem_raw);   // new hits, padded to a power of two
    const uint32_t q = blockIdx.x;
    const uint32_t c = cnt[q];
    const uint32_t n = min(c, cap);
    const float thr_old = thr[q];
    if (n < jrank && c <= cap) {  // too few candidates for a threshold: keep all (uniform per block)
        // ... fine while no threshold was ever applied (every passing row is here); otherwise a prediction starved it
        // (the host passes jrank == kprime with final, and the re-rank does not need a short buffer sorted)
        if (final && thr_old < __int_as_float(0x7f800000) && threadIdx.x == 0) atomicOr(&flags[q], 4u);
        return;
    }
    const uint32_t s = min(sorted_n[q], n);
    const uint32_t m = n - s;
    uint64_t* mine = cand + (size_t)q * cap;
    uint32_t Pm = 2;
    while (Pm < m) Pm <<= 1;
    Pm = min(Pm, P);
    uint64_t* o = a + Pm;                                   // the previous survivors (ascending), s <= kprime of them
    for (uint32_t i = threadIdx.x; i < Pm; i += blockDim.x) a[i] = i < m ? mine[s + i] : KEY_SENTINEL;
    for (uint32_t i = threadIdx.x; i < s; i += blockDim.x) o[i] = mine[i];
    bitonic_sort_smem(a, Pm);
    const uint32_t keep = min(n, kprime);
    for (uint32_t e = threadIdx.x; e < n; e += blockDim.x) {
        uint64_t key;
        uint32_t rank;
        if (e < s) {
            key = o[e];
            rank = e + sorted_count_below(a, m, key, true);
        } else {
            key = a[e - s];
            rank = (e - s) + sorted_count_below(o, s, key, false);
        }
        if (rank < keep) mine[rank] = key;
        if (rank == jrank - 1) thr[q] = fminf(thr_old, key_dist(key));
        if (final && rank == kprime - 1 && !(key_dist(key) <= thr_old)) atomicOr(&flags[q], 4u);
    }
    if (threadIdx.x == 0) {
        cnt[q] = keep;
        sorted_n[q] = keep;
        if (c > cap) atomicOr(&flags[q], 1u);
    }
}

struct RerankParams {
    const float4* rows;
    uint32_t ld4;
    const float4* queries;  // prepared [nq, ld]
    const float* q_norms;
    const uint32_t* max_norm2_bits;  // max |x|^2 over the rows (null for cosine: unit rows)
    const uint64_t* cand;
    const uint32_t* cnt;
    uint32_t* flags;
    uint32_t cap, kprime, k, P;
    float* out_dists;
    int64_t* out_rows;
    int32_t* out_counts;
    uint64_t row_base;
    const uint32_t* rowmap;  // candidate row (position in `rows`) -> index row; nullptr = identity
    int metric;  // MLV metric: 0 l2, 1 ip, 2 cosine
    float delta_rel;  // bound on |a - exact| / scale of the GEMM tier that selected the candidates
};

// One CTA per query: exact reference-form distances of the candidates with the scan kernel's
// summation order (lane l sums float4 columns l, l+32, ...; butterfly over the lanes), final
// top-k, and the certificate described at the top of this file.  flags[q] bit 1 = not certified.
template <int METRIC>
__global__ void __launch_bounds__(256, 1) rerank_kernel(const RerankParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint64_t* a = reinterpret_cast<uint64_t*>(smem_raw);
    const uint32_t q = blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t n = min(p.cnt[q], p.kprime);  // refine_kernel left them sorted by approximate key
    const uint64_t* mine = p.cand + (size_t)q * p.cap;
    const float4* qv = p.queries + (size_t)q * p.ld4;
    for (uint32_t i = threadIdx.x; i < p.P; i += blockDim.x) a[i] = KEY_SENTINEL;
    __syncthreads();
    // four candidates per warp at a time: four independent row reads in flight (one at a time ran the 2.8 GB of a
    // 4096 x 224-candidate batch at 4.3 TB/s); per candidate the arithmetic is unchanged
    const uint32_t nw = blockDim.x >> 5;
    for (uint32_t i0 = (uint32_t)warp * 4u; i0 < n; i0 += nw * 4u) {
        uint32_t rows4[4];
        const float4* x[4];
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int u = 0; u < 4; u++) {
            rows4[u] = key_row(mine[min(i0 + u, n - 1)]);
            x[u] = p.rows + (size_t)rows4[u] * p.ld4;
        }
        for (uint32_t j = lane; j < p.ld4; j += 32) {
            const float4 q4 = qv[j];
#pragma unroll
            for (int u = 0; u < 4; u++) acc[u] = accum4<METRIC>(acc[u], x[u][j], q4);
        }
#pragma unroll
        for (int u = 0; u < 4; u++) {
            float s = acc[u];
#pragma unroll
            for (int off = 16; off >= 1; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
            const float dist = (METRIC == METRIC_IP) ? 1.0f - s : s;
            if (lane == 0 && i0 + u < n) a[i0 + u] = make_key(dist, rows4[u]);
        }
    }
    bitonic_sort_smem(a, p.P);
    __shared__ int cnt_s;
    if (threadIdx.x == 0) cnt_s = 0;
    __syncthreads();
    int local = 0;
    for (uint32_t i = threadIdx.x; i < p.k; i += blockDim.x) {
        const uint64_t key = a[i];
        const bool valid = key != KEY_SENTINEL;
        p.out_dists[(size_t)q * p.k + i] = valid ? key_dist(key) : __int_as_float(0x7f800000);
        p.out_rows[(size_t)q * p.k + i] = valid ? (int64_t)(p.row_base + (p.rowmap ? p.rowmap[key_row(key)] : key_row(key))) : -1;
        local += valid;
    }
    if (local) atomicAdd(&cnt_s, local);
    __syncthreads();
    if (threadIdx.x == 0) {
        p.out_counts[q] = cnt_s;
        bool certified = true;
        if (n >= p.kprime && p.k <= n) {  // rows may exist outside the candidate set
            const float qn = p.q_norms[q];
            float scale;
            if (p.metric == 2) {
                scale = 1.0f;
            } else {
                const float xmax = sqrtf(__uint_as_float(*p.max_norm2_bits));
                const float qs = sqrtf(qn);
                scale = (p.metric == 0) ? (xmax + qs) * (xmax + qs) : xmax * qs;
            }
            const float delta = p.delta_rel * scale;
            const float a_last = key_dist(mine[p.kprime - 1]);  // largest approximate distance kept
            const float e_k = key_dist(a[p.k - 1]);             // exact k-th best among the candidates
            certified = (a_last - delta > e_k);                 // false for NaN
        }
        if (!certified) p.flags[q] |= 2u;
    }
}

}  // namespace mlv
