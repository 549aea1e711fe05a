// Tensor-core candidate pass of the cosine top-k (the only tensor-core path of the trainer): for a tile of 256 query
// rows (two M = 128 halves that share every table tile: the pass is bound by streaming the table, so operand reuse is
// what counts), stream the normalised bf16 table through tcgen05.mma (accumulators in TMEM, operands staged in shared memory by
// TMA with 128-byte swizzle) and keep, per query row, the KP best approximate similarities in a fused epilogue that
// reads the accumulator straight out of TMEM.  The candidates are re-scored exactly in fp32 (same routine as the fp32
// scan) and a query whose k-th exact score is not safely above the bf16 cut-off of the candidate lists is sent through the
// exact scan, so the returned ids are the exact fp32 top-k in every case
// [replaces cosine_similarity + tf.math.top_k, ref src/models/utils.py:12-19, src/models/model_utils.py:97-99].
//
// Warp roles (320 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer (one elected lane),
// warps 2..9 = epilogue (warps 2-5 drain the accumulators of query half 0, warps 6-9 those of half 1; each owns the
// 32-lane quarter of TMEM given by warp % 4; thread = one query row).
#include <stdlib.h>

#include <cuda.h>
#include <cudaTypedefs.h>
#include <cuda_bf16.h>

#include "glove_topk.cuh"

namespace glove {

constexpr int TC_M = 128;     // UMMA M
constexpr int TC_MQ = 256;    // query rows per CTA = 2 x UMMA M
constexpr int TC_N = 128;     // table rows per accumulator tile (UMMA N)
constexpr int TC_KC = 64;     // bf16 elements per K chunk = 128 bytes = one SWIZZLE_128B row
constexpr int TC_STAGES = 3;  // B-operand pipeline depth
constexpr int TC_KP = 32;     // candidates kept per (query, table slice)
constexpr int TC_THREADS = 320;
constexpr int TC_MAX_KCH = 5;  // Kp <= 320
constexpr uint32_t TC_A_HALF_BYTES = TC_M * TC_KC * 2;    // 16 KB
constexpr uint32_t TC_A_CHUNK_BYTES = TC_MQ * TC_KC * 2;  // 32 KB: rows 0-127 then rows 128-255
constexpr uint32_t TC_B_STAGE_BYTES = TC_N * TC_KC * 2;   // 16 KB
// Bound on |bf16 MMA similarity - fp32 similarity| of two rows normalised in fp32 (the guarantee check of rescore_kernel):
//  * bf16 keeps 8 significant bits, so rounding to nearest moves each factor by up to 2^-8 of itself, and a product of
//    two rounded factors by up to (1 + 2^-8)^2 - 1 = 2^-7 + 2^-16 of |q_c t_c|.  Summed over the columns, with
//    sum |q_c t_c| <= |q| |t| (Cauchy-Schwarz), that is 7.83e-3 for unit vectors.  The bound is attained when every
//    component sits just below a rounding midpoint (tests/test_topk_bound.py builds such a table): 2^-8 is NOT enough.
//  * fp32 normalisation: the sum of squares is at most ~15 roundings deep (per-lane sum + butterfly), so |q|, |t| are
//    within ~1e-6 of 1 -- a negligible change of the term above.
//  * fp32 accumulation of the MMA and of cos_dot, Kp <= 320 products each: n u sum |q_c t_c| <= 320 * 2^-24 = 1.9e-5
//    per sum with IEEE rounding; allowing twice that for the tensor core's own accumulation order, 6e-5 for both.
// 7.83e-3 + 6e-5 < 7.9e-3; rounded up to 8e-3.
constexpr float TC_DELTA = 8.0e-3f;

// ---- PTX wrappers ----------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}\n" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap *map, uint32_t bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum) : "memory");
}
// K-major operand tile in shared memory, 128-byte rows, SWIZZLE_128B: 8-row groups are 1024 bytes apart
__device__ __forceinline__ uint64_t sw128_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);  // start address
    d |= (uint64_t)1 << 16;                       // leading byte offset (unused for swizzled K-major)
    d |= (uint64_t)(1024 >> 4) << 32;             // stride byte offset
    d |= (uint64_t)1 << 46;                       // descriptor version (sm_100)
    d |= (uint64_t)2 << 61;                       // SWIZZLE_128B
    return d;
}
// kind::f16: D = F32, A = B = BF16, both K-major, M = 128, N = 128
constexpr uint32_t TC_IDESC = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(TC_N >> 3) << 17) | ((uint32_t)(TC_M >> 4) << 24);

struct TcSmem {  // offsets inside the 1024-byte aligned dynamic shared memory
    static constexpr uint32_t A = 0;
    static constexpr uint32_t B = TC_MAX_KCH * TC_A_CHUNK_BYTES;
    static constexpr uint32_t BARS = B + TC_STAGES * TC_B_STAGE_BYTES;
    static constexpr uint32_t TOTAL = BARS + 128;
};

__global__ void __launch_bounds__(TC_THREADS, 1)
topk_tc_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_t, int64_t V,
               int32_t kch, int32_t tiles_total, int32_t tiles_per_slice, float *cand_val, int32_t *cand_idx,
               float *cutoff) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t *gen = smem_raw + (base - smem_u32(smem_raw));
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int qt = blockIdx.x, slice = blockIdx.y, n_slices = gridDim.y;
    const int t0 = slice * tiles_per_slice, t1 = min(t0 + tiles_per_slice, tiles_total);
    const int n_tiles = max(t1 - t0, 0);

    const uint32_t bar0 = base + TcSmem::BARS;
    const uint32_t bar_a = bar0;                                       // queries landed
    auto bar_full = [&](int s) { return bar0 + 8u * (1 + s); };        // B stage filled by TMA
    auto bar_empty = [&](int s) { return bar0 + 8u * (1 + TC_STAGES + s); };  // B stage consumed by MMA
    auto bar_tfull = [&](int b) { return bar0 + 8u * (1 + 2 * TC_STAGES + b); };   // accumulator ready
    auto bar_tempty = [&](int b) { return bar0 + 8u * (3 + 2 * TC_STAGES + b); };  // accumulator drained
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(gen + TcSmem::BARS + 8 * (5 + 2 * TC_STAGES));

    if (threadIdx.x == 0) {
        mbar_init(bar_a, 1);
        for (int s = 0; s < TC_STAGES; ++s) { mbar_init(bar_full(s), 1); mbar_init(bar_empty(s), 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(bar_tfull(b), 1); mbar_init(bar_tempty(b), 8); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {  // TMEM: all 512 columns (2 buffers x 2 query halves of 128 x 128 fp32 accumulators)
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            mbar_expect_tx(bar_a, kch * TC_A_CHUNK_BYTES);
            for (int kc = 0; kc < kch; ++kc) tma_load_2d(base + TcSmem::A + kc * TC_A_CHUNK_BYTES, &map_q, bar_a, kc * TC_KC, qt * TC_MQ);
            int stage = 0;
            uint32_t phase = 0;
            for (int t = t0; t < t1; ++t) {
                for (int kc = 0; kc < kch; ++kc) {
                    mbar_wait(bar_empty(stage), phase ^ 1);
                    mbar_expect_tx(bar_full(stage), TC_B_STAGE_BYTES);
                    tma_load_2d(base + TcSmem::B + stage * TC_B_STAGE_BYTES, &map_t, bar_full(stage), kc * TC_KC, t * TC_N);
                    if (++stage == TC_STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        if (lane == 0) {
            mbar_wait(bar_a, 0);
            tc_fence_after();
            int stage = 0;
            uint32_t phase = 0;
            for (int j = 0; j < n_tiles; ++j) {
                const int buf = j & 1;
                mbar_wait(bar_tempty(buf), ((j >> 1) & 1) ^ 1);
                tc_fence_after();
                for (int kc = 0; kc < kch; ++kc) {
                    mbar_wait(bar_full(stage), phase);
                    tc_fence_after();
                    const uint64_t bdesc = sw128_desc(base + TcSmem::B + stage * TC_B_STAGE_BYTES);
#pragma unroll
                    for (int h = 0; h < 2; ++h) {            // both query halves consume the same table tile
                        const uint32_t d_tmem = tmem_base + (buf * 2 + h) * TC_N;
                        const uint64_t adesc = sw128_desc(base + TcSmem::A + kc * TC_A_CHUNK_BYTES + h * TC_A_HALF_BYTES);
#pragma unroll
                        for (int kk = 0; kk < TC_KC / 16; ++kk)  // UMMA_K = 16 bf16 = 32 bytes: +2 in the address field
                            tc_mma_bf16(d_tmem, adesc + 2 * kk, bdesc + 2 * kk, TC_IDESC, (kc | kk) != 0);
                    }
                    tc_commit(bar_empty(stage));  // frees the stage when these MMAs have read it
                    if (++stage == TC_STAGES) { stage = 0; phase ^= 1; }
                }
                tc_commit(bar_tfull(buf));        // accumulator complete
            }
        }
    } else {
        // ===== epilogue: thread = one query row; running top-KP of the approximate similarities =====
        const int quarter = warp & 3;                 // TMEM lane quarter this warp may access
        const int half = (warp - 2) >> 2;             // query half whose accumulators this warp drains
        const int row = half * TC_M + quarter * 32 + lane;
        // the running top-KP list lives in registers, sorted (descending): inserting is one pass of compare-and-swap over
        // statically indexed registers, the cut-off is the last entry.  No memory traffic until the list is published.
        const int64_t q = (int64_t)qt * TC_MQ + row;
        float lv[TC_KP];
        int32_t li[TC_KP];
#pragma unroll
        for (int e = 0; e < TC_KP; ++e) { lv[e] = -INFINITY; li[e] = -1; }
        float thr = -INFINITY;                        // KP-th best so far (-inf until the list is full)
        for (int j = 0; j < n_tiles; ++j) {
            const int buf = j & 1;
            mbar_wait(bar_tfull(buf), (j >> 1) & 1);
            tc_fence_after();
            const int64_t tile_row0 = (int64_t)(t0 + j) * TC_N;
#pragma unroll 1
            for (int c = 0; c < TC_N / 32; ++c) {
                uint32_t r[32];
                const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (buf * 2 + half) * TC_N + c * 32;
                asm volatile(
                    "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                    "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                    "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                    : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                      "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
                      "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
                      "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                    : "r"(taddr));
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                float m = __uint_as_float(r[0]);
#pragma unroll
                for (int e = 1; e < 32; ++e) m = fmaxf(m, __uint_as_float(r[e]));
                if (m > thr) {
                    const int64_t g0 = tile_row0 + c * 32;
                    uint32_t hits = 0;                             // entries of this chunk that beat the cut-off
#pragma unroll
                    for (int e = 0; e < 32; ++e) hits |= (uint32_t)(__uint_as_float(r[e]) > thr) << e;
                    while (hits) {
                        const int e = __ffs(hits) - 1;
                        hits &= hits - 1;
                        // r[] is statically indexed only in fully unrolled code: pick entry e with a select chain
                        float v = -INFINITY;
#pragma unroll
                        for (int u = 0; u < 32; ++u) v = (u == e) ? __uint_as_float(r[u]) : v;
                        if (v > thr && g0 + e < V) {
                            int32_t vi = (int32_t)(g0 + e);
#pragma unroll
                            for (int u = 0; u < TC_KP; ++u) {      // ties keep the earlier (lower) table row in front
                                const bool up = v > lv[u];
                                const float tv = lv[u];
                                const int32_t ti = li[u];
                                lv[u] = up ? v : tv;
                                li[u] = up ? vi : ti;
                                v = up ? tv : v;
                                vi = up ? ti : vi;
                            }
                            thr = lv[TC_KP - 1];
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_tempty(buf));
        }
        // publish the candidate list of this (query, slice)
        const int64_t o = (q * n_slices + slice) * TC_KP;
#pragma unroll
        for (int e = 0; e < TC_KP; ++e) {
            cand_val[o + e] = lv[e];
            cand_idx[o + e] = li[e];
        }
        cutoff[q * n_slices + slice] = thr;
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
    }
}

// normalised bf16 query rows, gathered from the normalised table copy (rows >= nq are zero)
__global__ void gather_queries_kernel(const __nv_bfloat16 *__restrict__ tn, int32_t Kp, const int32_t *__restrict__ query_ids,
                                      int32_t nq, int32_t nq_pad, __nv_bfloat16 *qn) {
    const int64_t total = (int64_t)nq_pad * Kp;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t q = i / Kp;
        const int c = (int)(i % Kp);
        qn[i] = q < nq ? tn[(int64_t)query_ids[q] * Kp + c] : __float2bfloat16(0.0f);
    }
}

// exact fp32 re-score of the candidates (one warp per query) + guarantee check
template <int NV>
__global__ void __launch_bounds__(256) rescore_kernel(const float *__restrict__ table, int32_t d, int32_t S, int32_t P,
                                                      const float *__restrict__ inv_norm, const float *__restrict__ qtable,
                                                      int32_t qP, const int32_t *__restrict__ query_ids,
                                                      int32_t nq, int32_t k, const int32_t *__restrict__ cand_idx,
                                                      const float *__restrict__ cutoff, int32_t n_slices, float *out_sim,
                                                      int32_t *out_idx, int32_t *flags) {
    extern __shared__ float qn_all[];  // [8 warps][S]
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int q = blockIdx.x * 8 + wid;
    if (q >= nq) return;
    float *qn = qn_all + wid * S;
    {
        const float *row = qtable + (int64_t)query_ids[q] * qP * S;
        const float rn = row_inv_norm(row, d, lane);
        for (int c = lane; c < S; c += 32) qn[c] = c < d ? row[c] * rn : 0.0f;
    }
    __syncwarp();
    const int S4 = S >> 2;
    LaneTopK top;
    top.init();
    const int n_cand = n_slices * TC_KP;
    for (int c = 0; c < n_cand; ++c) {
        const int32_t v = cand_idx[(int64_t)q * n_cand + c];
        if (v < 0) continue;
        float4 x[NV];
        const float *row = table + (int64_t)v * P * S;
#pragma unroll
        for (int r = 0; r < NV; ++r) x[r] = ld4_emb(row, lane + 32 * r, d);
        top.insert(cos_dot<NV>(qn, x, inv_norm[v], lane, S4), v, lane, k);
    }
    if (lane < k) {
        out_sim[(int64_t)q * k + lane] = top.sim;
        out_idx[(int64_t)q * k + lane] = top.idx;
    }
    // Anything outside the candidate lists has bf16 similarity <= cut-off, hence exact similarity <= cut-off + delta.
    // If the k-th exact score clears that, no outsider can belong to the top-k; otherwise re-run this query exactly.
    float cut = -INFINITY;
    for (int s = lane; s < n_slices; s += 32) cut = fmaxf(cut, cutoff[(int64_t)q * n_slices + s]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cut = fmaxf(cut, __shfl_xor_sync(0xffffffffu, cut, o));
    if (lane == 0) flags[q] = (top.thr > cut + TC_DELTA) ? 0 : 1;
}

static PFN_cuTensorMapEncodeTiled get_encode() {
    static PFN_cuTensorMapEncodeTiled fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = (PFN_cuTensorMapEncodeTiled)p;
    }
    return fn;
}

static int make_map(CUtensorMap *map, const void *ptr, uint64_t rows, uint64_t cols, uint32_t box_rows) {
    PFN_cuTensorMapEncodeTiled enc = get_encode();
    if (!enc) return set_error(GLOVE_ECUDA, "topk: cuTensorMapEncodeTiled entry point not available");
    cuuint64_t gdim[2] = {cols, rows};
    cuuint64_t gstride[1] = {cols * 2};
    cuuint32_t box[2] = {(cuuint32_t)TC_KC, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void *>(ptr), gdim, gstride, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return set_error(GLOVE_ECUDA, "topk: cuTensorMapEncodeTiled failed (%d)", (int)r);
    return GLOVE_OK;
}

struct TcWs {
    __nv_bfloat16 *qn;
    float *cand_val;
    int32_t *cand_idx;
    float *cutoff;
    int32_t *flags;
    void *scan_ws;
    size_t scan_bytes;
    size_t bytes;
    int32_t nq_pad, n_slices, tiles_per_slice;
};
static TcWs tc_ws_view(void *base, int64_t V, int32_t d, int32_t nq, int32_t k) {
    TcWs w;
    char *p = (char *)base;
    size_t off = 0;
    auto take = [&](size_t bytes) { char *r = p ? p + off : nullptr; off += align_up(bytes); return r; };
    const int32_t Kp = glove_topk_kpad(d);
    const int64_t tiles = glove_topk_vpad(V) / TC_N;
    w.nq_pad = (nq + TC_MQ - 1) / TC_MQ * TC_MQ;
    const int q_tiles = w.nq_pad / TC_MQ;
    // one CTA per SM: at least one full wave, and among 1..8 x that the slice count that wastes least of its last wave
    int slices = (kNumSMs + q_tiles - 1) / q_tiles;
    {
        const int lo = slices;
        double best = -1.0;
        for (int s = lo; s <= 8 * lo && s <= lo + 7; ++s) {
            const int ctas = q_tiles * s, waves = (ctas + kNumSMs - 1) / kNumSMs;
            const double eff = (double)ctas / ((double)waves * kNumSMs);
            if (eff > best + 0.02) { best = eff; slices = s; }
        }
    }
    if (const char *e = getenv("GLOVE_TOPK_SLICES")) {   // tuning aid
        const int n = atoi(e);
        if (n > 0) slices = n;
    }
    if (slices > tiles) slices = (int)tiles;
    if (slices < 1) slices = 1;
    w.tiles_per_slice = (int32_t)((tiles + slices - 1) / slices);
    w.n_slices = (int32_t)((tiles + w.tiles_per_slice - 1) / w.tiles_per_slice);
    w.qn = (__nv_bfloat16 *)take((size_t)w.nq_pad * Kp * 2);
    w.cand_val = (float *)take((size_t)w.nq_pad * w.n_slices * TC_KP * 4);
    w.cand_idx = (int32_t *)take((size_t)w.nq_pad * w.n_slices * TC_KP * 4);
    w.cutoff = (float *)take((size_t)w.nq_pad * w.n_slices * 4);
    w.flags = (int32_t *)take((size_t)w.nq_pad * 4);
    w.scan_bytes = scan_fp32_workspace(nq, k);
    w.scan_ws = take(w.scan_bytes);
    w.bytes = off;
    return w;
}

__global__ void count_flags_kernel(const int32_t *flags, int32_t n, int32_t *out) {
    int c = 0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) c += flags[i] != 0;
    c = (int)warp_sum((float)c);  // n_queries < 2^24
    __shared__ int sh[8];
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) { int t = 0; for (int w = 0; w < 8; ++w) t += sh[w]; *out = t; }
}

}  // namespace glove

using namespace glove;

extern "C" {

int glove_topk_flagged(const void *workspace, int64_t V, int32_t d, int32_t n_queries, int32_t k, int32_t *host_count,
                       void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GLOVE_REQUIRE(workspace && host_count && V > 0 && d > 0 && n_queries > 0 && k > 0, "glove_topk_flagged: bad arguments");
    TcWs w = tc_ws_view(const_cast<void *>(workspace), V, d, n_queries, k);
    int32_t *dev = w.flags + w.nq_pad - 1;  // last padding slot doubles as the counter when nq < nq_pad; else use cutoff[0]
    if (n_queries == w.nq_pad) dev = reinterpret_cast<int32_t *>(w.cutoff);
    count_flags_kernel<<<1, 256, 0, stream>>>(w.flags, n_queries, dev);
    GLOVE_CHECK_LAUNCH();
    GLOVE_CHECK_CUDA(cudaMemcpyAsync(host_count, dev, 4, cudaMemcpyDeviceToHost, stream));
    GLOVE_CHECK_CUDA(cudaStreamSynchronize(stream));
    return GLOVE_OK;
}

size_t glove_topk_workspace_bytes(int64_t V, int32_t d, int32_t n_queries, int32_t k) {
    if (V <= 0 || d <= 0 || n_queries <= 0 || k <= 0) return 0;
    return tc_ws_view(nullptr, V, d, n_queries, k).bytes;
}

int glove_topk_cosine_queries(const float *table, int64_t V, int32_t d, int32_t planes, const void *norm_bf16,
                              const float *inv_norm, const float *qtable, int32_t qplanes, const void *qnorm_bf16,
                              const int32_t *query_ids, int32_t n_queries, int32_t k, float *out_sim, int32_t *out_idx,
                              void *workspace, size_t workspace_bytes, void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GLOVE_REQUIRE(table && inv_norm && query_ids && out_sim && out_idx && workspace && qtable && qplanes >= 1,
                  "glove_topk_cosine: null pointer");
    GLOVE_REQUIRE(V > 0 && d > 0 && planes >= 1 && n_queries > 0, "glove_topk_cosine: bad sizes");
    if (k < 1 || k > 32 || k > V) return set_error(GLOVE_EUNSUPPORTED, "topk: k=%d not in [1, min(32, V)]", k);
    const int32_t Kp = glove_topk_kpad(d), S = table_stride(d);
    const int kch = Kp / TC_KC;
    TcWs w = tc_ws_view(workspace, V, d, n_queries, k);
    if (workspace_bytes < w.bytes)
        return set_error(GLOVE_EWORKSPACE, "glove_topk_cosine: workspace %zu < required %zu", workspace_bytes, w.bytes);
    // shapes the tensor-core pass does not cover go straight to the exact scan
    if (!norm_bf16 || !qnorm_bf16 || kch > TC_MAX_KCH || k > TC_KP - 8 || V < 1024)
        return scan_fp32_launch(table, V, d, planes, inv_norm, qtable, qplanes, query_ids, n_queries, k, nullptr, out_sim,
                                out_idx, w.scan_ws, w.scan_bytes, stream);
    const int64_t Vp = glove_topk_vpad(V);
    gather_queries_kernel<<<kNumSMs * 4, 256, 0, stream>>>((const __nv_bfloat16 *)qnorm_bf16, Kp, query_ids, n_queries,
                                                           w.nq_pad, w.qn);
    GLOVE_CHECK_LAUNCH();
    CUtensorMap map_q, map_t;
    int rc = make_map(&map_q, w.qn, (uint64_t)w.nq_pad, (uint64_t)Kp, TC_MQ);
    if (rc != GLOVE_OK) return rc;
    rc = make_map(&map_t, norm_bf16, (uint64_t)Vp, (uint64_t)Kp, TC_N);
    if (rc != GLOVE_OK) return rc;
    const size_t smem = TcSmem::TOTAL + 1024;
    GLOVE_CHECK_CUDA(cudaFuncSetAttribute(topk_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid(w.nq_pad / TC_MQ, w.n_slices);
    topk_tc_kernel<<<grid, TC_THREADS, smem, stream>>>(map_q, map_t, V, kch, (int32_t)(Vp / TC_N), w.tiles_per_slice,
                                                       w.cand_val, w.cand_idx, w.cutoff);
    GLOVE_CHECK_LAUNCH();
    const int nv = (S / 4 + 31) / 32;
    const size_t rs_smem = sizeof(float) * 8 * S;
    const int rs_blocks = (n_queries + 7) / 8;
#define LAUNCH_RESCORE(NV)                                                                                            \
    rescore_kernel<NV><<<rs_blocks, 256, rs_smem, stream>>>(table, d, S, planes, inv_norm, qtable, qplanes, query_ids,  \
                                                            n_queries, k, w.cand_idx, w.cutoff, w.n_slices, out_sim,  \
                                                            out_idx, w.flags)
    switch (nv) {
        case 1: LAUNCH_RESCORE(1); break;
        case 2: LAUNCH_RESCORE(2); break;
        case 3: LAUNCH_RESCORE(3); break;
        default: LAUNCH_RESCORE(4); break;
    }
#undef LAUNCH_RESCORE
    GLOVE_CHECK_LAUNCH();
    // guarantee fallback: flagged queries (none in the common case; the scan kernel exits at once for unflagged tiles)
    return scan_fp32_launch(table, V, d, planes, inv_norm, qtable, qplanes, query_ids, n_queries, k, w.flags, out_sim,
                            out_idx, w.scan_ws, w.scan_bytes, stream);
}

int glove_topk_cosine(const float *table, int64_t V, int32_t d, int32_t planes, const void *norm_bf16,
                      const float *inv_norm, const int32_t *query_ids, int32_t n_queries, int32_t k, float *out_sim,
                      int32_t *out_idx, void *workspace, size_t workspace_bytes, void *stream) {
    return glove_topk_cosine_queries(table, V, d, planes, norm_bf16, inv_norm, table, planes, norm_bf16, query_ids, n_queries,
                                     k, out_sim, out_idx, workspace, workspace_bytes, stream);
}

}  // extern "C"
