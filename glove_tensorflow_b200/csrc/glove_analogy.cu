// Intrinsic evaluation of the row embeddings: word analogies and word-pair similarity
// [conventions of Stanford GloVe eval/python/evaluate.py; 3CosMul: Levy & Goldberg 2014].
//
//   * 3CosAdd: q = b^ - a^ + c^ (x^ = x * row_inv_norm(x)) is written as a packed one-plane table and ranked with the
//     cosine top-k (glove_topk_cosine_queries) for k + 3 entries; drop_abc_kernel then removes the ids a, b, c and keeps
//     the first k.  Exact: the order (score descending, id ascending) is total, so the k best ids outside {a, b, c} are
//     the k first survivors of the k + 3 best overall.
//   * 3CosMul: an exact fp32 scan of its own (mul_scan_kernel), since its score combines three cosines per candidate.
//   * pair cosine: the similarity routine of the top-k (query normalised with row_inv_norm, cos_dot against the
//     candidate row and its inv_norm), so cos(w1, w2) equals the similarity topk(w1) reports for w2, bit for bit.
#include "glove_topk.cuh"

namespace glove {

// 3CosMul tiling: a CTA holds kMulQT questions (a^, b^, c^ in shared memory) and sweeps its slice of the table in tiles of
// kMulTV rows, one row per thread; each tile is staged through shared memory kMulDC columns at a time, transposed, so a
// thread reads its row's column from shared memory once and its 3 kMulQT accumulators take one FFMA each per broadcast
// question element.  Every table row is read once per kMulQT questions.
constexpr int kMulQT = 8;
constexpr int kMulTV = 256;
constexpr int kMulDC = 32;
constexpr float kMulEps = 1e-3f;  // Levy & Goldberg's epsilon

// normalised query vector of table row `id` in dst[0, width), zero outside columns < d (as scan_fp32_kernel builds it)
__device__ __forceinline__ void load_unit_row(const float *__restrict__ table, int32_t S, int32_t P, int32_t d, int32_t id,
                                              float *dst, int32_t width, int lane) {
    const float *row = table + (int64_t)id * P * S;
    const float rn = row_inv_norm(row, d, lane);
    for (int c = lane; c < width; c += 32) dst[c] = c < d ? row[c] * rn : 0.0f;
}

// one warp per question: q[c] = (b^[c] - a^[c]) + c^[c] for c < d, 0 for d <= c < S; ids[i] = i
__global__ void __launch_bounds__(256) add_query_kernel(const float *__restrict__ table, int32_t d, int32_t S, int32_t P,
                                                        const int32_t *__restrict__ abc, int32_t n, float *q, int32_t *ids) {
    const int lane = threadIdx.x & 31;
    const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (i >= n) return;
    const float *ra = table + (int64_t)abc[3 * i] * P * S;
    const float *rb = table + (int64_t)abc[3 * i + 1] * P * S;
    const float *rc = table + (int64_t)abc[3 * i + 2] * P * S;
    const float na = row_inv_norm(ra, d, lane), nb = row_inv_norm(rb, d, lane), nc = row_inv_norm(rc, d, lane);
    float *out = q + (int64_t)i * S;
    for (int c = lane; c < S; c += 32)
        out[c] = c < d ? __fadd_rn(__fsub_rn(__fmul_rn(rb[c], nb), __fmul_rn(ra[c], na)), __fmul_rn(rc[c], nc)) : 0.0f;
    if (lane == 0) ids[i] = i;
}

// thread per question: the first k entries of the (k + 3)-list whose id is not a, b or c
__global__ void drop_abc_kernel(const float *__restrict__ sim, const int32_t *__restrict__ idx, int32_t kk,
                                const int32_t *__restrict__ abc, int32_t n, int32_t k, float *out_score, int32_t *out_idx) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int32_t a = abc[3 * i], b = abc[3 * i + 1], c = abc[3 * i + 2];
    int o = 0;
    for (int j = 0; j < kk && o < k; ++j) {
        const int32_t v = idx[(int64_t)i * kk + j];
        if (v == a || v == b || v == c) continue;
        out_score[(int64_t)i * k + o] = sim[(int64_t)i * kk + j];
        out_idx[(int64_t)i * k + o] = v;
        ++o;
    }
}

// 3CosMul scan: grid (question tiles of kMulQT, V slices), 256 threads.  For candidate x and question (a, b, c), in
// this fp32 order:  dot_a = fmaf chain over the columns c = 0, 1, ..., d-1 of a^[c] * x[c] (likewise b, c),
//     ca = dot_a * inv_norm[x],  pa = (1 + ca) * 0.5,  pb, pc alike,  score = (pb * pc) / (pa + 1e-3)
// every operation rounded to nearest (explicit intrinsics: no contraction into FMA).  x in {a, b, c} is skipped.
// Output: per (question, slice, warp) a sorted list of k (LaneTopK), merged by glove_topk_merge.
__global__ void __launch_bounds__(256) mul_scan_kernel(const float *__restrict__ table, int64_t V, int32_t d, int32_t S,
                                                       int32_t P, int32_t Sp, const float *__restrict__ inv_norm,
                                                       const int32_t *__restrict__ abc, int32_t n, int32_t k,
                                                       int64_t rows_per_slice, float *cand_sim, int32_t *cand_idx) {
    extern __shared__ float mul_smem[];
    float *qs = mul_smem;                             // [kMulQT * 3][Sp]: a^, b^, c^ per question, zero past d
    float *xs = mul_smem + kMulQT * 3 * Sp;           // [kMulDC][kMulTV + 1]: a column chunk of the tile, transposed
    __shared__ int32_t qid[kMulQT][3];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int q0 = blockIdx.x * kMulQT;
    for (int j = wid; j < kMulQT * 3; j += 8) {
        const int t = j / 3, w = j % 3, q = q0 + t;
        const int32_t id = q < n ? abc[3 * q + w] : 0;
        load_unit_row(table, S, P, d, id, qs + j * Sp, Sp, lane);
        if (lane == 0) qid[t][w] = q < n ? id : -1;
    }
    LaneTopK top[kMulQT];
#pragma unroll
    for (int t = 0; t < kMulQT; ++t) top[t].init();
    const int64_t s0 = blockIdx.y * rows_per_slice, s1 = min(s0 + rows_per_slice, V);
    for (int64_t t0 = s0; t0 < s1; t0 += kMulTV) {
        float acc[kMulQT * 3];
#pragma unroll
        for (int j = 0; j < kMulQT * 3; ++j) acc[j] = 0.0f;
        for (int c0 = 0; c0 < Sp; c0 += kMulDC) {
            __syncthreads();                          // the previous chunk is consumed (and qs / qid are written)
            for (int e = tid; e < kMulTV * (kMulDC / 4); e += 256) {
                const int r = e / (kMulDC / 4), c = c0 + 4 * (e % (kMulDC / 4));
                const int64_t v = t0 + r;
                float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
                if (v < s1 && c < d) {                // c + 3 < S: inside the row; columns >= d (bias, last step) -> 0
                    x = ld4(table + v * P * S + c);
                    if (c + 1 >= d) x.y = 0.0f;
                    if (c + 2 >= d) x.z = 0.0f;
                    if (c + 3 >= d) x.w = 0.0f;
                }
                float *col = xs + (c - c0) * (kMulTV + 1) + r;
                col[0] = x.x;
                col[kMulTV + 1] = x.y;
                col[2 * (kMulTV + 1)] = x.z;
                col[3 * (kMulTV + 1)] = x.w;
            }
            __syncthreads();
#pragma unroll 1
            for (int c = 0; c < kMulDC; c += 4) {
                const float x0 = xs[c * (kMulTV + 1) + tid], x1 = xs[(c + 1) * (kMulTV + 1) + tid];
                const float x2 = xs[(c + 2) * (kMulTV + 1) + tid], x3 = xs[(c + 3) * (kMulTV + 1) + tid];
#pragma unroll
                for (int j = 0; j < kMulQT * 3; ++j) {
                    const float4 q = *reinterpret_cast<const float4 *>(qs + j * Sp + c0 + c);
                    acc[j] = fmaf(q.x, x0, acc[j]);
                    acc[j] = fmaf(q.y, x1, acc[j]);
                    acc[j] = fmaf(q.z, x2, acc[j]);
                    acc[j] = fmaf(q.w, x3, acc[j]);
                }
            }
        }
        const int64_t v = t0 + tid;
        const float rn = v < s1 ? inv_norm[v] : 0.0f;
#pragma unroll
        for (int t = 0; t < kMulQT; ++t) {
            const int32_t ia = qid[t][0], ib = qid[t][1], ic = qid[t][2];
            const bool ok = v < s1 && ia >= 0 && v != ia && v != ib && v != ic;
            const float pa = __fmul_rn(__fadd_rn(1.0f, __fmul_rn(acc[3 * t], rn)), 0.5f);
            const float pb = __fmul_rn(__fadd_rn(1.0f, __fmul_rn(acc[3 * t + 1], rn)), 0.5f);
            const float pc = __fmul_rn(__fadd_rn(1.0f, __fmul_rn(acc[3 * t + 2], rn)), 0.5f);
            const float score = __fdiv_rn(__fmul_rn(pb, pc), __fadd_rn(pa, kMulEps));
            unsigned m = __ballot_sync(0xffffffffu, ok && score >= top[t].thr);
            while (m) {                               // lanes in order: a fixed insertion sequence
                const int l = __ffs(m) - 1;
                m &= m - 1;
                top[t].insert(__shfl_sync(0xffffffffu, score, l), (int32_t)__shfl_sync(0xffffffffu, (int32_t)v, l), lane, k);
            }
        }
    }
    const int n_lists = gridDim.y * 8;
#pragma unroll
    for (int t = 0; t < kMulQT; ++t) {
        const int q = q0 + t;
        if (q < n && lane < k) {
            const int64_t o = (((int64_t)q * n_lists) + blockIdx.y * 8 + wid) * k + lane;
            cand_sim[o] = top[t].sim;
            cand_idx[o] = top[t].idx;  // an empty entry (INT_MAX, -inf) never beats a real one in the merge
        }
    }
}

// one warp per pair: w1 normalised as the query of the top-k, cos_dot against the row of w2 and inv_norm[w2]
template <int NV>
__global__ void __launch_bounds__(256) pair_cosine_kernel(const float *__restrict__ table, int32_t d, int32_t S, int32_t P,
                                                          const float *__restrict__ inv_norm,
                                                          const int32_t *__restrict__ pairs, int32_t n, float *out) {
    extern __shared__ float qn_all[];  // [8 warps][S]
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int i = blockIdx.x * 8 + wid;
    if (i >= n) return;
    float *qn = qn_all + wid * S;
    load_unit_row(table, S, P, d, pairs[2 * i], qn, S, lane);
    __syncwarp();
    const int32_t v = pairs[2 * i + 1];
    const float *row = table + (int64_t)v * P * S;
    float4 x[NV];
#pragma unroll
    for (int r = 0; r < NV; ++r) x[r] = ld4_emb(row, lane + 32 * r, d);
    const float s = cos_dot<NV>(qn, x, inv_norm[v], lane, S >> 2);
    if (lane == 0) out[i] = s;
}

struct MulPlan {
    int q_tiles, slices;
    int64_t rows_per_slice;
};
static MulPlan mul_plan(int64_t V, int32_t n) {
    MulPlan p;
    p.q_tiles = (n + kMulQT - 1) / kMulQT;
    int slices = (2 * kNumSMs + p.q_tiles - 1) / p.q_tiles;  // at least two CTAs per SM
    if (slices > 64) slices = 64;
    if ((int64_t)slices * kMulTV > V) slices = (int)((V + kMulTV - 1) / kMulTV);  // at least one full tile per slice
    if (slices < 1) slices = 1;
    p.slices = slices;
    p.rows_per_slice = (V + slices - 1) / slices;
    return p;
}

struct AnalogyWs {
    float *q;                // ADD: [n][S] query rows
    void *q_bf16;            // ADD: [vpad(n)][Kp] normalised bf16 copy
    int32_t *ids;            // ADD: arange(n)
    float *sim;              // ADD: [n][k+3]; MUL: candidate lists
    int32_t *idx;
    void *topk_ws;           // ADD: workspace of glove_topk_cosine_queries
    size_t topk_bytes;
    size_t bytes;
};
static AnalogyWs analogy_ws_view(void *base, int64_t V, int32_t d, int32_t n, int32_t k, int32_t method) {
    AnalogyWs w{};
    char *p = (char *)base;
    size_t off = 0;
    auto take = [&](size_t bytes) { char *r = p ? p + off : nullptr; off += align_up(bytes); return r; };
    if (method == GLOVE_ANALOGY_ADD) {
        const int32_t kk = k + 3;
        w.q = (float *)take((size_t)n * table_stride(d) * 4);
        w.q_bf16 = take((size_t)glove_topk_vpad(n) * glove_topk_kpad(d) * 2);
        w.ids = (int32_t *)take((size_t)n * 4);
        w.sim = (float *)take((size_t)n * kk * 4);
        w.idx = (int32_t *)take((size_t)n * kk * 4);
        w.topk_bytes = glove_topk_workspace_bytes(V, d, n, kk);
        w.topk_ws = take(w.topk_bytes);
    } else {
        const MulPlan pl = mul_plan(V, n);
        const size_t n_cand = (size_t)n * pl.slices * 8 * k;
        w.sim = (float *)take(n_cand * 4);
        w.idx = (int32_t *)take(n_cand * 4);
    }
    w.bytes = off;
    return w;
}

static int analogy_check_args(int64_t V, int32_t d, int32_t n, int32_t k, int32_t method) {
    GLOVE_REQUIRE(V > 0 && d > 0 && n > 0, "glove_analogy: bad sizes (V=%lld, d=%d, n=%d)", (long long)V, d, n);
    if (method != GLOVE_ANALOGY_ADD && method != GLOVE_ANALOGY_MUL)
        return set_error(GLOVE_EUNSUPPORTED, "glove_analogy: unknown method %d", method);
    if (k < 1 || k > 29 || (int64_t)k + 3 > V)
        return set_error(GLOVE_EUNSUPPORTED, "glove_analogy: k=%d not in [1, min(29, V - 3)]", k);
    if ((table_stride(d) / 4 + 31) / 32 > 4)
        return set_error(GLOVE_EUNSUPPORTED, "glove_analogy: embedding size %d > 510 not supported", d);
    return GLOVE_OK;
}

}  // namespace glove

using namespace glove;

extern "C" {

size_t glove_analogy_workspace_bytes(int64_t V, int32_t d, int32_t n_questions, int32_t k, int32_t method) {
    if (V <= 0 || d <= 0 || n_questions <= 0 || k <= 0) return 0;
    if (method != GLOVE_ANALOGY_ADD && method != GLOVE_ANALOGY_MUL) return 0;
    return analogy_ws_view(nullptr, V, d, n_questions, k, method).bytes;
}

int glove_analogy_topk(const float *table, int64_t V, int32_t d, int32_t planes, const void *norm_bf16,
                       const float *inv_norm, const int32_t *abc, int32_t n_questions, int32_t method, int32_t k,
                       float *out_score, int32_t *out_idx, void *workspace, size_t workspace_bytes, void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GLOVE_REQUIRE(table && inv_norm && abc && out_score && out_idx && workspace, "glove_analogy_topk: null pointer");
    GLOVE_REQUIRE(planes >= 1, "glove_analogy_topk: planes=%d", planes);
    int rc = analogy_check_args(V, d, n_questions, k, method);
    if (rc != GLOVE_OK) return rc;
    const AnalogyWs w = analogy_ws_view(workspace, V, d, n_questions, k, method);
    if (workspace_bytes < w.bytes)
        return set_error(GLOVE_EWORKSPACE, "glove_analogy_topk: workspace %zu < required %zu", workspace_bytes, w.bytes);
    const int32_t S = table_stride(d);
    if (method == GLOVE_ANALOGY_ADD) {
        const int32_t kk = k + 3;
        add_query_kernel<<<(n_questions + 7) / 8, 256, 0, stream>>>(table, d, S, planes, abc, n_questions, w.q, w.ids);
        GLOVE_CHECK_LAUNCH();
        if (norm_bf16) {
            rc = glove_normalize_rows(w.q, n_questions, d, 1, w.q_bf16, nullptr, stream);
            if (rc != GLOVE_OK) return rc;
        }
        rc = glove_topk_cosine_queries(table, V, d, planes, norm_bf16, inv_norm, w.q, 1, norm_bf16 ? w.q_bf16 : nullptr,
                                       w.ids, n_questions, kk, w.sim, w.idx, w.topk_ws, w.topk_bytes, stream);
        if (rc != GLOVE_OK) return rc;
        drop_abc_kernel<<<(n_questions + 255) / 256, 256, 0, stream>>>(w.sim, w.idx, kk, abc, n_questions, k, out_score,
                                                                       out_idx);
        GLOVE_CHECK_LAUNCH();
        return GLOVE_OK;
    }
    const MulPlan pl = mul_plan(V, n_questions);
    const int32_t Sp = (d + kMulDC - 1) / kMulDC * kMulDC;
    const size_t smem = sizeof(float) * (kMulQT * 3 * Sp + kMulDC * (kMulTV + 1));
    GLOVE_CHECK_CUDA(cudaFuncSetAttribute(mul_scan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    mul_scan_kernel<<<dim3(pl.q_tiles, pl.slices), 256, smem, stream>>>(table, V, d, S, planes, Sp, inv_norm, abc,
                                                                        n_questions, k, pl.rows_per_slice, w.sim, w.idx);
    GLOVE_CHECK_LAUNCH();
    return glove_topk_merge(w.sim, w.idx, n_questions, pl.slices * 8 * k, k, out_score, out_idx, stream);
}

int glove_pair_cosine(const float *table, int64_t V, int32_t d, int32_t planes, const float *inv_norm,
                      const int32_t *pairs, int32_t n_pairs, float *out, void *stream) {
    GLOVE_REQUIRE(table && inv_norm && pairs && out, "glove_pair_cosine: null pointer");
    GLOVE_REQUIRE(V > 0 && d > 0 && planes >= 1 && n_pairs > 0, "glove_pair_cosine: bad sizes");
    const int32_t S = table_stride(d);
    const int nv = (S / 4 + 31) / 32;
    if (nv > 4) return set_error(GLOVE_EUNSUPPORTED, "glove_pair_cosine: embedding size %d > 510 not supported", d);
    const size_t smem = sizeof(float) * 8 * S;
    const int blocks = (n_pairs + 7) / 8;
#define LAUNCH_PAIR(NV)                                                                                               \
    pair_cosine_kernel<NV><<<blocks, 256, smem, (cudaStream_t)stream>>>(table, d, S, planes, inv_norm, pairs, n_pairs, out)
    switch (nv) {
        case 1: LAUNCH_PAIR(1); break;
        case 2: LAUNCH_PAIR(2); break;
        case 3: LAUNCH_PAIR(3); break;
        default: LAUNCH_PAIR(4); break;
    }
#undef LAUNCH_PAIR
    GLOVE_CHECK_LAUNCH();
    return GLOVE_OK;
}

}  // extern "C"
