// PREDICT: cosine top-k -- cosine_similarity + tf.math.top_k of the reference
// [ref src/models/utils.py:12-19, src/models/model_utils.py:81-110]:
//     sim[q, v] = l2norm(R[q]) . l2norm(R[v]),  top_k(sim, k, sorted): values descending, ties -> lower index.
//
// Two implementations of the same contract:
//   * glove_topk_cosine_fp32 : exact fp32 CUDA-core scan (this file).
//   * glove_topk_cosine      : tcgen05 / TMA bf16 candidate pass (glove_topk_tc.cu) + exact fp32 re-score of the
//                              candidates with the SAME dot-product routine as the scan, + a guarantee check that sends
//                              a query back through the exact scan when the bf16 cut-off is too close to its k-th score.
#include <cuda_bf16.h>

#include "glove_topk.cuh"

namespace glove {

// ---- normalisation ---------------------------------------------------------------------------------------------------
// inv_norm[v] = rsqrt(max(sum x^2, 1e-12))  (tf.math.l2_normalize), bf16 copy of x * inv_norm for the tensor-core pass
__global__ void __launch_bounds__(256) normalize_kernel(const float *__restrict__ table, int64_t V, int32_t d, int32_t S,
                                                        int32_t P, __nv_bfloat16 *out, int32_t Kp, int64_t Vp,
                                                        float *inv_norm) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t v = warp; v < Vp; v += nwarps) {
        float rn = 0.0f;
        const float *row = table + v * P * S;
        if (v < V) {
            rn = row_inv_norm(row, d, lane);
            if (lane == 0 && inv_norm) inv_norm[v] = rn;
        }
        if (out)
            for (int c = lane; c < Kp; c += 32)
                out[v * Kp + c] = __float2bfloat16((v < V && c < d) ? row[c] * rn : 0.0f);
    }
}

// ---- exact fp32 scan ---------------------------------------------------------------------------------------------------
// grid (query tiles of kScanQT, V slices); 8 warps stride the rows of the slice; every warp keeps, per query, a sorted
// top-k list spread over its lanes (k <= 32).
template <int NV>
__global__ void __launch_bounds__(256) scan_fp32_kernel(const float *__restrict__ table, int64_t V, int32_t d, int32_t S,
                                                        int32_t P, const float *__restrict__ inv_norm,
                                                        const float *__restrict__ qtable, int32_t qP,
                                                        const int32_t *__restrict__ query_ids, int32_t nq, int32_t k,
                                                        const int32_t *__restrict__ only_flagged, int64_t rows_per_slice,
                                                        float *cand_sim, int32_t *cand_idx) {
    extern __shared__ float qn[];  // [kScanQT][S] normalised queries, zero outside columns < d
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int q0 = blockIdx.x * kScanQT;
    if (only_flagged) {  // guarantee-check fallback: skip tiles with no flagged query
        bool any = false;
        for (int t = 0; t < kScanQT; ++t) any |= (q0 + t < nq) && only_flagged[q0 + t];
        if (!any) return;
    }
    for (int t = wid; t < kScanQT; t += 8) {
        const int q = q0 + t;
        const float *row = qtable + (int64_t)(q < nq ? query_ids[q] : 0) * qP * S;   // queries may live in another table
        const float rn = q < nq ? row_inv_norm(row, d, lane) : 0.0f;
        for (int c = lane; c < S; c += 32) qn[t * S + c] = (q < nq && c < d) ? row[c] * rn : 0.0f;
    }
    __syncthreads();
    const int S4 = S >> 2;
    LaneTopK top[kScanQT];
#pragma unroll
    for (int t = 0; t < kScanQT; ++t) top[t].init();
    const int64_t v0 = blockIdx.y * rows_per_slice, v1 = min(v0 + rows_per_slice, V);
    for (int64_t v = v0 + wid; v < v1; v += 8) {
        float4 x[NV];
        const float *row = table + v * P * S;
        const float rn = inv_norm[v];
#pragma unroll
        for (int r = 0; r < NV; ++r) x[r] = ld4_emb(row, lane + 32 * r, d);
#pragma unroll
        for (int t = 0; t < kScanQT; ++t) {
            const float sim = cos_dot<NV>(qn + t * S, x, rn, lane, S4);
            top[t].insert(sim, (int32_t)v, lane, k);
        }
    }
    // cand[q][slice][warp][k]
    const int n_lists = gridDim.y * 8;
#pragma unroll
    for (int t = 0; t < kScanQT; ++t) {
        const int q = q0 + t;
        if (q < nq && lane < k) {
            const int64_t o = (((int64_t)q * n_lists) + blockIdx.y * 8 + wid) * k + lane;
            cand_sim[o] = top[t].sim;
            cand_idx[o] = top[t].idx;
        }
    }
}

// one warp per query merges n_lists sorted-or-not candidate lists of k entries (empty entries have idx < 0)
__global__ void __launch_bounds__(256) merge_kernel(const float *__restrict__ cand_sim, const int32_t *__restrict__ cand_idx,
                                                    int32_t nq, int32_t n_cand, int32_t k,
                                                    const int32_t *__restrict__ only_flagged, float *out_sim,
                                                    int32_t *out_idx) {
    const int lane = threadIdx.x & 31;
    const int q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (q >= nq) return;
    if (only_flagged && !only_flagged[q]) return;
    LaneTopK top;
    top.init();
    for (int c0 = 0; c0 < n_cand; c0 += 32) {
        const int c = c0 + lane;
        const float s = c < n_cand ? cand_sim[(int64_t)q * n_cand + c] : 0.0f;
        const int32_t i = c < n_cand ? cand_idx[(int64_t)q * n_cand + c] : -1;
        for (int l = 0; l < 32 && c0 + l < n_cand; ++l) {
            const float sl = __shfl_sync(0xffffffffu, s, l);
            const int32_t il = __shfl_sync(0xffffffffu, i, l);
            if (il >= 0) top.insert(sl, il, lane, k);
        }
    }
    if (lane < k) {
        out_sim[(int64_t)q * k + lane] = top.sim;
        out_idx[(int64_t)q * k + lane] = top.idx;
    }
}

int scan_fp32_launch(const float *table, int64_t V, int32_t d, int32_t planes, const float *inv_norm,
                     const float *qtable, int32_t qplanes, const int32_t *query_ids, int32_t nq, int32_t k,
                     const int32_t *only_flagged, float *out_sim, int32_t *out_idx, void *workspace, size_t workspace_bytes,
                     cudaStream_t stream) {
    const int32_t S = table_stride(d);
    const int nv = (S / 4 + 31) / 32;
    const int q_tiles = (nq + kScanQT - 1) / kScanQT;
    int slices = (2 * kNumSMs + q_tiles - 1) / q_tiles;
    if (slices < 1) slices = 1;
    if (slices > 64) slices = 64;
    if ((int64_t)slices * 64 > V) slices = (int)((V + 63) / 64);
    const int64_t rows_per_slice = (V + slices - 1) / slices;
    const int n_cand = slices * 8 * k;
    const size_t need = align_up((size_t)nq * n_cand * 4) * 2;
    if (workspace_bytes < need)
        return set_error(GLOVE_EWORKSPACE, "topk fp32: workspace %zu < required %zu", workspace_bytes, need);
    float *cand_sim = (float *)workspace;
    int32_t *cand_idx = (int32_t *)((char *)workspace + align_up((size_t)nq * n_cand * 4));
    const size_t smem = sizeof(float) * kScanQT * S;
    dim3 grid(q_tiles, slices);
#define LAUNCH_SCAN(NV)                                                                                              \
    scan_fp32_kernel<NV><<<grid, 256, smem, stream>>>(table, V, d, S, planes, inv_norm, qtable, qplanes, query_ids, nq, k, \
                                                      only_flagged, rows_per_slice, cand_sim, cand_idx)
    switch (nv) {
        case 1: LAUNCH_SCAN(1); break;
        case 2: LAUNCH_SCAN(2); break;
        case 3: LAUNCH_SCAN(3); break;
        case 4: LAUNCH_SCAN(4); break;
        default: return set_error(GLOVE_EUNSUPPORTED, "topk: embedding size %d > 510 not supported", d);
    }
#undef LAUNCH_SCAN
    GLOVE_CHECK_LAUNCH();
    merge_kernel<<<(nq + 7) / 8, 256, 0, stream>>>(cand_sim, cand_idx, nq, n_cand, k, only_flagged, out_sim, out_idx);
    GLOVE_CHECK_LAUNCH();
    return GLOVE_OK;
}

size_t scan_fp32_workspace(int32_t nq, int32_t k) { return 2 * align_up((size_t)nq * 64 * 8 * k * 4); }

}  // namespace glove

using namespace glove;

extern "C" {

int32_t glove_topk_kpad(int32_t d) { return (d + 63) / 64 * 64; }
int64_t glove_topk_vpad(int64_t V) { return (V + 255) / 256 * 256; }

int glove_normalize_rows(const float *table, int64_t V, int32_t d, int32_t planes, void *out_bf16, float *inv_norm,
                         void *stream) {
    GLOVE_REQUIRE(table && V > 0 && d > 0 && planes >= 1 && (out_bf16 || inv_norm), "glove_normalize_rows: bad arguments");
    const int64_t Vp = out_bf16 ? glove_topk_vpad(V) : V;
    int64_t blocks = (Vp + 7) / 8;
    if (blocks > kNumSMs * 8) blocks = kNumSMs * 8;
    normalize_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(table, V, d, table_stride(d), planes,
                                                                    (__nv_bfloat16 *)out_bf16, glove_topk_kpad(d), Vp,
                                                                    inv_norm);
    GLOVE_CHECK_LAUNCH();
    return GLOVE_OK;
}

int glove_topk_cosine_fp32(const float *table, int64_t V, int32_t d, int32_t planes, const float *inv_norm,
                           const int32_t *query_ids, int32_t n_queries, int32_t k, float *out_sim, int32_t *out_idx,
                           void *workspace, size_t workspace_bytes, void *stream) {
    GLOVE_REQUIRE(table && inv_norm && query_ids && out_sim && out_idx && workspace, "glove_topk_cosine_fp32: null pointer");
    GLOVE_REQUIRE(V > 0 && d > 0 && planes >= 1 && n_queries > 0, "glove_topk_cosine_fp32: bad sizes");
    if (k < 1 || k > 32 || k > V) return set_error(GLOVE_EUNSUPPORTED, "topk: k=%d not in [1, min(32, V)]", k);
    return scan_fp32_launch(table, V, d, planes, inv_norm, table, planes, query_ids, n_queries, k, nullptr, out_sim, out_idx,
                            workspace, workspace_bytes, (cudaStream_t)stream);
}

// Merge n_cand candidates per query (idx < 0 = empty) into the k best: descending similarity, ties -> lower id.  The last
// step of a row-sharded top-k: every shard contributes the top-k of its own rows (ids already made global).
int glove_topk_merge(const float *cand_sim, const int32_t *cand_idx, int32_t n_queries, int32_t n_cand, int32_t k,
                     float *out_sim, int32_t *out_idx, void *stream) {
    GLOVE_REQUIRE(cand_sim && cand_idx && out_sim && out_idx && n_queries > 0 && n_cand > 0, "glove_topk_merge: bad arguments");
    if (k < 1 || k > 32) return set_error(GLOVE_EUNSUPPORTED, "topk: k=%d not in [1, 32]", k);
    merge_kernel<<<(n_queries + 7) / 8, 256, 0, (cudaStream_t)stream>>>(cand_sim, cand_idx, n_queries, n_cand, k, nullptr,
                                                                         out_sim, out_idx);
    GLOVE_CHECK_LAUNCH();
    return GLOVE_OK;
}

}  // extern "C"
