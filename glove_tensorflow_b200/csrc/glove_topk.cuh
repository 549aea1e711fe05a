// Shared pieces of the cosine top-k path: the exact fp32 similarity routine (one definition, used by the scan and by the
// re-score of tensor-core candidates, so both produce bit-identical similarities) and a warp-distributed sorted list.
#pragma once
#include <limits.h>
#include <math.h>

#include "glove_common.cuh"

namespace glove {

constexpr int kScanQT = 8;  // queries per CTA of the fp32 scan

// 1 / sqrt(max(sum_{c<d} x_c^2, 1e-12))  -- tf.math.l2_normalize's scale [ref src/models/utils.py:13-15]
__device__ __forceinline__ float row_inv_norm(const float *__restrict__ row, int d, int lane) {
    float ss = 0.0f;
    for (int c = lane; c < d; c += 32) ss = fmaf(row[c], row[c], ss);
    ss = warp_sum(ss);
    return 1.0f / sqrtf(fmaxf(ss, 1e-12f));
}

// float4 number f of a packed row with the columns >= d (bias, last_step, padding) read as zero: nothing stored there, not
// even a non-finite bias, reaches a similarity (0 * inf is NaN).  Bit-identical to the plain load for finite values.
__device__ __forceinline__ float4 ld4_emb(const float *__restrict__ row, int f, int d) {
    const int c = 4 * f;
    float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
    if (c < d) {
        x = ld4(row + c);
        if (c + 1 >= d) x.y = 0.0f;
        if (c + 2 >= d) x.z = 0.0f;
        if (c + 3 >= d) x.w = 0.0f;
    }
    return x;
}

// sim = sum_c qn[c] * (x[c] * rn): qn = normalised query (zero outside columns < d), x = packed table row held as NV
// float4 per lane (ld4_emb: zero outside columns < d), rn = its inverse norm.
template <int NV>
__device__ __forceinline__ float cos_dot(const float *__restrict__ qn, const float4 (&x)[NV], float rn, int lane, int S4) {
    float p = 0.0f;
#pragma unroll
    for (int r = 0; r < NV; ++r) {
        const int f = lane + 32 * r;
        if (f < S4) {
            const float4 q = *reinterpret_cast<const float4 *>(qn + 4 * f);
            p = fmaf(q.x, x[r].x * rn, p);
            p = fmaf(q.y, x[r].y * rn, p);
            p = fmaf(q.z, x[r].z * rn, p);
            p = fmaf(q.w, x[r].w * rn, p);
        }
    }
    return warp_sum(p);
}

// Sorted (similarity descending, ties -> lower id) list of up to 32 entries, entry l in lane l.  insert() takes
// warp-uniform arguments.
struct LaneTopK {
    float sim;
    int32_t idx;
    float thr;  // similarity of entry k-1 (warp-uniform): anything strictly below cannot enter
    __device__ __forceinline__ void init() { sim = -INFINITY; idx = INT_MAX; thr = -INFINITY; }
    __device__ __forceinline__ void insert(float s, int32_t i, int lane, int k) {
        if (!(s >= thr)) return;
        const bool beaten = (s > sim) || (s == sim && i < idx);
        const unsigned ballot = __ballot_sync(0xffffffffu, beaten && lane < k);
        if (ballot == 0) return;
        const int pos = __ffs(ballot) - 1;
        const float us = __shfl_up_sync(0xffffffffu, sim, 1);
        const int32_t ui = __shfl_up_sync(0xffffffffu, idx, 1);
        if (lane > pos) { sim = us; idx = ui; }
        else if (lane == pos) { sim = s; idx = i; }
        thr = __shfl_sync(0xffffffffu, sim, k - 1);
    }
};

int scan_fp32_launch(const float *table, int64_t V, int32_t d, int32_t planes, const float *inv_norm,
                     const float *qtable, int32_t qplanes, const int32_t *query_ids, int32_t nq, int32_t k,
                     const int32_t *only_flagged, float *out_sim, int32_t *out_idx, void *workspace, size_t workspace_bytes,
                     cudaStream_t stream);
size_t scan_fp32_workspace(int32_t nq, int32_t k);

}  // namespace glove
