// PREPROCESS (SURVEY §8 f.4): token-id stream -> symmetric co-occurrence table with the GloVe columns, i.e.
// create_interaction_dataframe + create_glove_dataframe of the reference preprocessor [ref src/data/text8.py:84-139]
// without the position cross-join (2-3 min and 21 GB of pandas at text8 scale):
//
//   cooc_chunk    emit, for every position p and distance k = 1..context, the pair (id[p], id[p+k]) (right context only,
//                 equal ids dropped) [ref text8.py:90-95]; radix-sort the packed (row, col) keys with k as payload;
//                 reduce-by-key to {count, numer} where numer = sum L/k, L = lcm(1..context): the sum of 1/k is carried
//                 as an exact integer [ref text8.py:98-102]
//   cooc_merge    union of two sorted partial tables (chunks of a corpus larger than one sort)
//   cooc_finish   union with the transposed table and sum [ref text8.py:105-110], count >= count_minimum
//                 [ref text8.py:129], value = numer / L (one rounding), neg_weight = count_row * proportion_col
//                 [ref text8.py:113-117], glove_weight = clip((count/100)^0.75, 0, 1), glove_value = log(value)
//                 [ref text8.py:130-139]; records come out in a keyed-hash order (the reference orders them by Python's
//                 per-process salted hash() of the token pair, i.e. randomly [ref text8.py:119-124])
//
// The Stanford GloVe scheme (vocab_count / cooccur, corpus.py scheme "stanford") shares the sort, reduce, route and
// finish code: emit_line_pairs_kernel emits (left, right) at distances 1..window (<= 15) within one line of the
// in-vocabulary token stream, self pairs kept, weights lcm(1..window)/k or 1; route sends one or both orientations;
// every pair becomes a record.
//
// Integer / sort work, HBM-bound: CUB radix sort + reduce-by-key around small hand-written kernels; no tensor cores.
#include <cub/cub.cuh>
#include <thrust/iterator/transform_iterator.h>

#include "glove_common.cuh"

namespace glove {

constexpr int kCoocMaxPartBits = 12;   // glove_cooc_route: at most 4096 partitions

struct Agg { long long count, numer; };
struct AggSum {
    __host__ __device__ __forceinline__ Agg operator()(const Agg &a, const Agg &b) const {
        return Agg{a.count + b.count, a.numer + b.numer};
    }
};
// payload k-1 of a sorted pair -> its contribution {1, w[k-1]}; N = 8 (reference contexts 1..8) or 16 (Stanford windows
// 1..15), so that the reference pass carries no more payload table than it needs
template <int N> struct KToAggN {
    long long w[N];
    __host__ __device__ __forceinline__ Agg operator()(const uint8_t &k1) const { return Agg{1, w[k1 & (N - 1)]}; }
};
using KToAgg = KToAggN<8>;
using KToAgg16 = KToAggN<16>;
constexpr int kStanfordMaxWindow = 15;

static int vbits_of(int64_t V) {
    int b = 1;
    while ((1ll << b) < V) ++b;
    return b;
}
static long long lcm_upto(int n) {
    long long l = 1;
    for (int k = 2; k <= n; ++k) {
        long long a = l, b = k;
        while (b) { const long long t = a % b; a = b; b = t; }
        l = l / a * k;
    }
    return l;
}

struct CoocWs {
    uint64_t *keys[4];
    uint32_t *idx[2];
    uint8_t *kk[2];
    Agg *agg, *agg2;
    uint8_t *flags;
    long long *count_out;   // device scalar written by CUB
    void *cub_temp;
    size_t cub_bytes;
    size_t bytes;
};
static CoocWs cooc_ws_view(void *base, int64_t n) {
    CoocWs w;
    char *p = (char *)base;
    size_t off = 0;
    auto take = [&](size_t bytes) { char *r = p ? p + off : nullptr; off += align_up(bytes); return r; };
    for (int i = 0; i < 4; ++i) w.keys[i] = (uint64_t *)take(sizeof(uint64_t) * n);
    for (int i = 0; i < 2; ++i) w.idx[i] = (uint32_t *)take(sizeof(uint32_t) * n);
    for (int i = 0; i < 2; ++i) w.kk[i] = (uint8_t *)take(n);
    w.agg = (Agg *)take(sizeof(Agg) * n);
    w.agg2 = (Agg *)take(sizeof(Agg) * n);
    w.flags = (uint8_t *)take(n);
    w.count_out = (long long *)take(sizeof(long long));
    size_t a = 0, b = 0, c = 0, d = 0, e = 0;
    const int ni = (int)n;
    cub::DeviceRadixSort::SortPairs(nullptr, a, (uint64_t *)nullptr, (uint64_t *)nullptr, (uint8_t *)nullptr, (uint8_t *)nullptr, ni);
    cub::DeviceRadixSort::SortPairs(nullptr, b, (uint64_t *)nullptr, (uint64_t *)nullptr, (uint32_t *)nullptr, (uint32_t *)nullptr, ni);
    thrust::transform_iterator<KToAgg, const uint8_t *> it((const uint8_t *)nullptr, KToAgg());
    cub::DeviceReduce::ReduceByKey(nullptr, c, (uint64_t *)nullptr, (uint64_t *)nullptr, it, (Agg *)nullptr, (long long *)nullptr, AggSum(), ni);
    size_t c16 = 0;
    thrust::transform_iterator<KToAgg16, const uint8_t *> it16((const uint8_t *)nullptr, KToAgg16());
    cub::DeviceReduce::ReduceByKey(nullptr, c16, (uint64_t *)nullptr, (uint64_t *)nullptr, it16, (Agg *)nullptr, (long long *)nullptr, AggSum(), ni);
    if (c16 > c) c = c16;
    cub::DeviceReduce::ReduceByKey(nullptr, d, (uint64_t *)nullptr, (uint64_t *)nullptr, (Agg *)nullptr, (Agg *)nullptr, (long long *)nullptr, AggSum(), ni);
    cub::DeviceSelect::Flagged(nullptr, e, (uint32_t *)nullptr, (uint8_t *)nullptr, (uint32_t *)nullptr, (long long *)nullptr, ni);
    w.cub_bytes = a;
    if (b > w.cub_bytes) w.cub_bytes = b;
    if (c > w.cub_bytes) w.cub_bytes = c;
    if (d > w.cub_bytes) w.cub_bytes = d;
    if (e > w.cub_bytes) w.cub_bytes = e;
    w.cub_temp = take(w.cub_bytes);
    w.bytes = off;
    return w;
}

// pair (p, k): row = id[p], col = id[p + k]; ids outside [0, V) are an error of the caller (flag)
__global__ void __launch_bounds__(256) emit_pairs_kernel(const int32_t *__restrict__ ids, int64_t n_positions, int64_t n_tokens,
                                                         int32_t context, int vbits, int32_t V, uint64_t *keys, uint8_t *kk,
                                                         int32_t *bad) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_positions * context) return;
    const int64_t p = t / context;
    const int k = (int)(t - p * context) + 1;
    const uint64_t none = (1ull << (2 * vbits)) - 1;   // row == col == 2^vbits - 1: never a valid pair, sorts last
    uint64_t key = none;
    if (p + k < n_tokens) {
        const int32_t a = ids[p], b = ids[p + k];
        if (a < 0 || a >= V || b < 0 || b >= V) *bad = 1;
        else if (a != b) key = ((uint64_t)(uint32_t)a << vbits) | (uint32_t)b;
    }
    keys[t] = key;
    kk[t] = (uint8_t)(k - 1);
}

// Stanford GloVe's cooccur: pair (p, k): left = id of tok[p], right = id of tok[p + k], emitted only when both lie on one
// line (equal segment ids); self pairs are kept.  tok[i] = (segment << 32) | id, the in-vocabulary tokens in text order
// (glove_tokens_stream), so out-of-vocabulary words take no position.
__global__ void __launch_bounds__(256) emit_line_pairs_kernel(const uint64_t *__restrict__ tok, int64_t n_positions,
                                                              int64_t n_tokens, int32_t window, int vbits, int32_t V,
                                                              uint64_t *keys, uint8_t *kk, int32_t *bad) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_positions * window) return;
    const int64_t p = t / window;
    const int k = (int)(t - p * window) + 1;
    uint64_t key = (1ull << (2 * vbits)) - 1;          // as in emit_pairs_kernel: never a valid pair, sorts last
    if (p + k < n_tokens) {
        const uint64_t x = tok[p], y = tok[p + k];
        const int32_t a = (int32_t)(uint32_t)x, b = (int32_t)(uint32_t)y;
        if (a < 0 || a >= V || b < 0 || b >= V) *bad = 1;
        else if ((x >> 32) == (y >> 32)) key = ((uint64_t)(uint32_t)a << vbits) | (uint32_t)b;
    }
    keys[t] = key;
    kk[t] = (uint8_t)(k - 1);
}

__global__ void __launch_bounds__(256) iota_kernel(uint32_t *idx, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) idx[i] = (uint32_t)i;
}
// concatenated tables A | B addressed by one index
__global__ void __launch_bounds__(256) gather_agg_kernel(const uint32_t *__restrict__ idx, int64_t n, const Agg *__restrict__ a,
                                                         int64_t na, const Agg *__restrict__ b, Agg *out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t j = idx[i];
    out[i] = j < na ? a[j] : b[j - na];
}
__global__ void __launch_bounds__(256) transpose_keys_kernel(const uint64_t *__restrict__ keys, int64_t n, int vbits,
                                                             uint64_t *out, uint32_t *idx) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t k = keys[i], mask = (1ull << vbits) - 1;
    out[i] = k;
    out[n + i] = ((k & mask) << vbits) | (k >> vbits);
    idx[i] = (uint32_t)i;
    idx[n + i] = (uint32_t)i;   // both orientations carry the same {count, numer}
}
__device__ __forceinline__ uint64_t mix64(uint64_t x) {
    x ^= x >> 30; x *= 0xbf58476d1ce4e5b9ull;
    x ^= x >> 27; x *= 0x94d049bb133111ebull;
    return x ^ (x >> 31);
}
__global__ void __launch_bounds__(256) flag_min_count_kernel(const Agg *__restrict__ agg, int64_t n, long long count_min,
                                                             uint8_t *flags, uint32_t *idx) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    flags[i] = agg[i].count >= count_min && agg[i].count != 0 && agg[i].numer != 0;
    idx[i] = (uint32_t)i;
}
__global__ void __launch_bounds__(256) order_keys_kernel(const uint64_t *__restrict__ keys, const uint32_t *__restrict__ sel,
                                                         int64_t n, uint64_t salt, uint64_t *hashed) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) hashed[i] = mix64(keys[sel[i]] + salt * 0x9e3779b97f4a7c15ull);
}
__global__ void __launch_bounds__(256) columns_kernel(const uint64_t *__restrict__ keys, const Agg *__restrict__ agg,
                                                      const uint32_t *__restrict__ order, int64_t n, int vbits, double inv_unit,
                                                      long long unit, const long long *__restrict__ vocab_count,
                                                      double total, int32_t *row, int32_t *col, long long *count,
                                                      double *value, double *neg_weight, double *glove_weight,
                                                      double *glove_value) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t j = order[i];
    const uint64_t k = keys[j];
    const int32_t a = (int32_t)(k >> vbits), b = (int32_t)(k & ((1ull << vbits) - 1));
    const Agg g = agg[j];
    const double v = (double)g.numer / (double)unit;          // exact integer / small integer: one rounding
    row[i] = a;
    col[i] = b;
    count[i] = g.count;
    value[i] = v;
    neg_weight[i] = (double)vocab_count[a] * ((double)vocab_count[b] / total);
    glove_weight[i] = fmin(fmax(pow((double)g.count / 100.0, 0.75), 0.0), 1.0);
    glove_value[i] = log(v);
}

// partition of a directed key: the top part_bits bits of its order hash, so that the partitions taken in ascending order
// and each sorted by the full hash give the single-table record order
__device__ __forceinline__ uint32_t part_of(uint64_t key, uint64_t salt, int part_bits) {
    return part_bits ? (uint32_t)(mix64(key + salt * 0x9e3779b97f4a7c15ull) >> (64 - part_bits)) : 0u;
}
__device__ __forceinline__ uint64_t directed_key(const uint64_t *keys, int64_t n, int64_t t, int vbits) {
    const uint64_t k = keys[t < n ? t : t - n], mask = (1ull << vbits) - 1;
    return t < n ? k : ((k & mask) << vbits) | (k >> vbits);
}
// t < n: entry t as (a, b); t >= n: entry t - n as (b, a); n_orient = 2 routes both orientations, 1 only (a, b)
__global__ void __launch_bounds__(256) route_parts_kernel(const uint64_t *__restrict__ keys, int64_t n, int n_orient, int vbits,
                                                          uint64_t salt, int part_bits, uint32_t *part, uint32_t *idx) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_orient * n) return;
    part[t] = part_of(directed_key(keys, n, t, vbits), salt, part_bits);
    idx[t] = (uint32_t)t;
}
__global__ void __launch_bounds__(256) route_scatter_kernel(const uint64_t *__restrict__ keys, const Agg *__restrict__ agg,
                                                            int64_t n, int n_orient, int vbits, const uint32_t *__restrict__ order,
                                                            uint64_t *out_keys, Agg *out_agg) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_orient * n) return;
    const int64_t t = order[i];
    out_keys[i] = directed_key(keys, n, t, vbits);
    out_agg[i] = agg[t < n ? t : t - n];
}

struct RouteWs {
    uint32_t *part[2], *idx[2];
    int *hist;
    void *cub_temp;
    size_t cub_bytes, bytes;
};
static RouteWs route_ws_view(void *base, int64_t n2, int part_bits) {
    RouteWs w;
    char *p = (char *)base;
    size_t off = 0;
    auto take = [&](size_t bytes) { char *r = p ? p + off : nullptr; off += align_up(bytes); return r; };
    for (int i = 0; i < 2; ++i) w.part[i] = (uint32_t *)take(4 * n2);
    for (int i = 0; i < 2; ++i) w.idx[i] = (uint32_t *)take(4 * n2);
    w.hist = (int *)take(sizeof(int) << part_bits);
    size_t a = 0, b = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, a, (uint32_t *)nullptr, (uint32_t *)nullptr, (uint32_t *)nullptr, (uint32_t *)nullptr,
                                    (int)n2);
    cub::DeviceHistogram::HistogramEven(nullptr, b, (uint32_t *)nullptr, (int *)nullptr, (1 << part_bits) + 1, 0u,
                                        (uint32_t)(1 << part_bits), (int)n2);
    w.cub_bytes = a > b ? a : b;
    w.cub_temp = take(w.cub_bytes);
    w.bytes = off;
    return w;
}

static int read_count(const long long *dev, long long *host, cudaStream_t stream) {
    GLOVE_CHECK_CUDA(cudaMemcpyAsync(host, dev, sizeof(long long), cudaMemcpyDeviceToHost, stream));
    GLOVE_CHECK_CUDA(cudaStreamSynchronize(stream));
    return GLOVE_OK;
}

// sorts the n emitted (key, k-1) pairs of a chunk and reduces them to {count, sum of w[k-1]} per key into the caller's
// buffers, dropping the sentinel run
template <class Conv>
static int reduce_chunk_pairs(const char *who, const CoocWs &w, int64_t n, int vbits, const Conv &conv, int32_t V,
                              const int32_t *bad, uint64_t *out_keys, int64_t *out_agg, int64_t capacity,
                              int64_t *n_unique_host, cudaStream_t stream) {
    size_t tb = w.cub_bytes;
    GLOVE_CHECK_CUDA(cub::DeviceRadixSort::SortPairs(w.cub_temp, tb, w.keys[0], w.keys[1], w.kk[0], w.kk[1], (int)n, 0,
                                                     2 * vbits, stream));
    thrust::transform_iterator<Conv, const uint8_t *> vals(w.kk[1], conv);
    tb = w.cub_bytes;
    GLOVE_CHECK_CUDA(cub::DeviceReduce::ReduceByKey(w.cub_temp, tb, w.keys[1], w.keys[0], vals, w.agg, w.count_out, AggSum(),
                                                    (int)n, stream));
    long long runs = 0;
    int32_t bad_h = 0;
    GLOVE_CHECK_CUDA(cudaMemcpyAsync(&bad_h, bad, sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
    if (int rc = read_count(w.count_out, &runs, stream)) return rc;
    if (bad_h) return set_error(GLOVE_EINVAL, "%s: token id outside [0, %d)", who, V);
    // the sentinel run (dropped pairs), when present, is the last one
    uint64_t last_key = 0;
    if (runs > 0) {
        GLOVE_CHECK_CUDA(cudaMemcpyAsync(&last_key, w.keys[0] + runs - 1, sizeof(uint64_t), cudaMemcpyDeviceToHost, stream));
        GLOVE_CHECK_CUDA(cudaStreamSynchronize(stream));
        if (last_key == (1ull << (2 * vbits)) - 1) --runs;
    }
    if (runs > capacity)
        return set_error(GLOVE_EINVAL, "%s: %lld distinct pairs > capacity %lld", who, runs, (long long)capacity);
    GLOVE_CHECK_CUDA(cudaMemcpyAsync(out_keys, w.keys[0], sizeof(uint64_t) * runs, cudaMemcpyDeviceToDevice, stream));
    GLOVE_CHECK_CUDA(cudaMemcpyAsync(out_agg, w.agg, sizeof(Agg) * runs, cudaMemcpyDeviceToDevice, stream));
    GLOVE_CHECK_CUDA(cudaStreamSynchronize(stream));
    *n_unique_host = runs;
    return GLOVE_OK;
}

// routes n_orient orientations of every entry of a table to its partition (glove_cooc_route*); arguments checked
static int route_entries(const char *who, const uint64_t *keys, const int64_t *agg, int64_t n, int n_orient, int32_t V,
                         uint64_t order_key, int32_t part_bits, void *workspace, size_t workspace_bytes, uint64_t *out_keys,
                         int64_t *out_agg, int64_t *part_count_host, cudaStream_t stream) {
    const int vbits = vbits_of((int64_t)V + 1);
    const int64_t n2 = n_orient * n;
    const RouteWs w = route_ws_view(workspace, n2, part_bits);
    if (workspace_bytes < w.bytes)
        return set_error(GLOVE_EWORKSPACE, "%s: workspace %zu < required %zu", who, workspace_bytes, w.bytes);
    const unsigned g = (unsigned)((n2 + 255) / 256);
    route_parts_kernel<<<g, 256, 0, stream>>>(keys, n, n_orient, vbits, order_key, part_bits, w.part[0], w.idx[0]);
    GLOVE_CHECK_LAUNCH();
    const uint32_t *order = w.idx[0];
    const int P = 1 << part_bits;
    if (part_bits) {
        size_t tb = w.cub_bytes;
        GLOVE_CHECK_CUDA(cub::DeviceRadixSort::SortPairs(w.cub_temp, tb, w.part[0], w.part[1], w.idx[0], w.idx[1], (int)n2, 0,
                                                         part_bits, stream));
        tb = w.cub_bytes;
        GLOVE_CHECK_CUDA(cub::DeviceHistogram::HistogramEven(w.cub_temp, tb, w.part[1], w.hist, P + 1, 0u, (uint32_t)P, (int)n2,
                                                             stream));
        order = w.idx[1];
    }
    route_scatter_kernel<<<g, 256, 0, stream>>>(keys, (const Agg *)agg, n, n_orient, vbits, order, out_keys, (Agg *)out_agg);
    GLOVE_CHECK_LAUNCH();
    if (part_bits) {
        int hist[1 << kCoocMaxPartBits];
        GLOVE_CHECK_CUDA(cudaMemcpyAsync(hist, w.hist, sizeof(int) * P, cudaMemcpyDeviceToHost, stream));
        GLOVE_CHECK_CUDA(cudaStreamSynchronize(stream));
        for (int p = 0; p < P; ++p) part_count_host[p] = hist[p];
    } else {
        GLOVE_CHECK_CUDA(cudaStreamSynchronize(stream));
        part_count_host[0] = n2;
    }
    return GLOVE_OK;
}

// records of a summed symmetric table (keys sorted ascending, unique): count >= count_min, in the keyed-hash order
// (a stable sort of the ascending keys by mix64(key + salt phi): equal hashes keep key order), with the GloVe columns
static int finish_records(const char *who, const uint64_t *keys, const Agg *agg, long long m, const CoocWs &w, int vbits,
                          int32_t context, int64_t count_min, const int64_t *vocab_count, int64_t total_tokens,
                          uint64_t order_key, int32_t *row, int32_t *col, int64_t *count, double *value, double *neg_weight,
                          double *glove_weight, double *glove_value, int64_t capacity, int64_t *n_out_host,
                          cudaStream_t stream) {
    // count >= count_minimum
    flag_min_count_kernel<<<(unsigned)((m + 255) / 256), 256, 0, stream>>>(agg, m, count_min, w.flags, w.idx[0]);
    GLOVE_CHECK_LAUNCH();
    size_t tb = w.cub_bytes;
    GLOVE_CHECK_CUDA(cub::DeviceSelect::Flagged(w.cub_temp, tb, w.idx[0], w.flags, w.idx[1], w.count_out, (int)m, stream));
    long long n_out = 0;
    if (int rc = read_count(w.count_out, &n_out, stream)) return rc;
    *n_out_host = n_out;
    if (n_out > capacity)
        return set_error(GLOVE_EINVAL, "%s: %lld records > capacity %lld", who, n_out, (long long)capacity);
    if (n_out == 0) return GLOVE_OK;
    GLOVE_REQUIRE(row && col && count && value && neg_weight && glove_weight && glove_value, "%s: null output", who);
    // keyed-hash record order
    const unsigned go = (unsigned)((n_out + 255) / 256);
    order_keys_kernel<<<go, 256, 0, stream>>>(keys, w.idx[1], n_out, order_key, w.keys[2]);
    GLOVE_CHECK_LAUNCH();
    tb = w.cub_bytes;
    GLOVE_CHECK_CUDA(cub::DeviceRadixSort::SortPairs(w.cub_temp, tb, w.keys[2], w.keys[3], w.idx[1], w.idx[0], (int)n_out, 0, 64,
                                                     stream));
    const long long unit = lcm_upto(context);
    columns_kernel<<<go, 256, 0, stream>>>(keys, agg, w.idx[0], n_out, vbits, 1.0 / (double)unit, unit,
                                           (const long long *)vocab_count, (double)total_tokens, row, col,
                                           (long long *)count, value, neg_weight, glove_weight, glove_value);
    GLOVE_CHECK_LAUNCH();
    GLOVE_CHECK_CUDA(cudaStreamSynchronize(stream));
    return GLOVE_OK;
}

}  // namespace glove

using namespace glove;

extern "C" {

size_t glove_cooc_workspace_bytes(int64_t n_items) { return cooc_ws_view(nullptr, n_items < 1 ? 1 : n_items).bytes; }

int glove_cooc_chunk(const int32_t *token_ids, int64_t n_positions, int64_t n_tokens, int32_t V, int32_t context,
                     void *workspace, size_t workspace_bytes, uint64_t *out_keys, int64_t *out_agg, int64_t capacity,
                     int64_t *n_unique_host, void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GLOVE_REQUIRE(token_ids && workspace && out_keys && out_agg && n_unique_host, "glove_cooc_chunk: null pointer");
    GLOVE_REQUIRE(n_positions > 0 && n_tokens >= n_positions && V > 1 && context >= 1 && context <= 8,
                  "glove_cooc_chunk: bad sizes (context must be 1..8)");
    const int64_t n = n_positions * context;
    GLOVE_REQUIRE(n < (1ll << 31), "glove_cooc_chunk: more than 2^31 pairs in one chunk");
    const int vbits = vbits_of((int64_t)V + 1);
    GLOVE_REQUIRE(2 * vbits <= 62, "glove_cooc_chunk: vocabulary too large");
    const CoocWs w = cooc_ws_view(workspace, n);
    if (workspace_bytes < w.bytes)
        return set_error(GLOVE_EWORKSPACE, "glove_cooc_chunk: workspace %zu < required %zu", workspace_bytes, w.bytes);
    int32_t *bad = (int32_t *)w.flags;
    GLOVE_CHECK_CUDA(cudaMemsetAsync(bad, 0, sizeof(int32_t), stream));
    emit_pairs_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(token_ids, n_positions, n_tokens, context, vbits, V,
                                                                        w.keys[0], w.kk[0], bad);
    GLOVE_CHECK_LAUNCH();
    KToAgg conv;
    const long long unit = lcm_upto(context);
    for (int k = 0; k < 8; ++k) conv.w[k] = k < context ? unit / (k + 1) : 0;
    return reduce_chunk_pairs("glove_cooc_chunk", w, n, vbits, conv, V, bad, out_keys, out_agg, capacity, n_unique_host, stream);
}

int glove_cooc_chunk_stanford(const uint64_t *tokens, int64_t n_positions, int64_t n_tokens, int32_t V, int32_t window,
                           int32_t distance_weighting, void *workspace, size_t workspace_bytes, uint64_t *out_keys,
                           int64_t *out_agg, int64_t capacity, int64_t *n_unique_host, void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GLOVE_REQUIRE(tokens && workspace && out_keys && out_agg && n_unique_host, "glove_cooc_chunk_stanford: null pointer");
    GLOVE_REQUIRE(n_positions > 0 && n_tokens >= n_positions && V > 0 && window >= 1 && window <= kStanfordMaxWindow,
                  "glove_cooc_chunk_stanford: bad sizes (window must be 1..%d)", kStanfordMaxWindow);
    const int64_t n = n_positions * window;
    GLOVE_REQUIRE(n < (1ll << 31), "glove_cooc_chunk_stanford: more than 2^31 pairs in one chunk");
    const int vbits = vbits_of((int64_t)V + 1);
    GLOVE_REQUIRE(2 * vbits <= 62, "glove_cooc_chunk_stanford: vocabulary too large");
    const CoocWs w = cooc_ws_view(workspace, n);
    if (workspace_bytes < w.bytes)
        return set_error(GLOVE_EWORKSPACE, "glove_cooc_chunk_stanford: workspace %zu < required %zu", workspace_bytes, w.bytes);
    int32_t *bad = (int32_t *)w.flags;
    GLOVE_CHECK_CUDA(cudaMemsetAsync(bad, 0, sizeof(int32_t), stream));
    emit_line_pairs_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(tokens, n_positions, n_tokens, window, vbits, V,
                                                                             w.keys[0], w.kk[0], bad);
    GLOVE_CHECK_LAUNCH();
    KToAgg16 conv;
    const long long unit = lcm_upto(window);
    for (int k = 0; k < 16; ++k) conv.w[k] = k >= window ? 0 : distance_weighting ? unit / (k + 1) : 1;
    return reduce_chunk_pairs("glove_cooc_chunk_stanford", w, n, vbits, conv, V, bad, out_keys, out_agg, capacity, n_unique_host,
                              stream);
}

int glove_cooc_merge(const uint64_t *keys_a, const int64_t *agg_a, int64_t n_a, const uint64_t *keys_b, const int64_t *agg_b,
                     int64_t n_b, int32_t V, void *workspace, size_t workspace_bytes, uint64_t *out_keys, int64_t *out_agg,
                     int64_t capacity, int64_t *n_unique_host, void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GLOVE_REQUIRE(workspace && out_keys && out_agg && n_unique_host && n_a >= 0 && n_b >= 0 && n_a + n_b > 0,
                  "glove_cooc_merge: bad arguments");
    const int64_t n = n_a + n_b;
    GLOVE_REQUIRE(n < (1ll << 31), "glove_cooc_merge: more than 2^31 entries");
    const int vbits = vbits_of((int64_t)V + 1);
    const CoocWs w = cooc_ws_view(workspace, n);
    if (workspace_bytes < w.bytes)
        return set_error(GLOVE_EWORKSPACE, "glove_cooc_merge: workspace %zu < required %zu", workspace_bytes, w.bytes);
    if (n_a) GLOVE_CHECK_CUDA(cudaMemcpyAsync(w.keys[0], keys_a, sizeof(uint64_t) * n_a, cudaMemcpyDeviceToDevice, stream));
    if (n_b) GLOVE_CHECK_CUDA(cudaMemcpyAsync(w.keys[0] + n_a, keys_b, sizeof(uint64_t) * n_b, cudaMemcpyDeviceToDevice, stream));
    iota_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(w.idx[0], n);
    GLOVE_CHECK_LAUNCH();
    size_t tb = w.cub_bytes;
    GLOVE_CHECK_CUDA(cub::DeviceRadixSort::SortPairs(w.cub_temp, tb, w.keys[0], w.keys[1], w.idx[0], w.idx[1], (int)n, 0,
                                                     2 * vbits, stream));
    gather_agg_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(w.idx[1], n, (const Agg *)agg_a, n_a, (const Agg *)agg_b,
                                                                        w.agg);
    GLOVE_CHECK_LAUNCH();
    // reduce straight into the caller's buffers when they can hold the worst case, else refuse
    GLOVE_REQUIRE(capacity >= n, "glove_cooc_merge: capacity %lld < n_a + n_b = %lld", (long long)capacity, (long long)n);
    tb = w.cub_bytes;
    GLOVE_CHECK_CUDA(cub::DeviceReduce::ReduceByKey(w.cub_temp, tb, w.keys[1], out_keys, w.agg, (Agg *)out_agg, w.count_out,
                                                    AggSum(), (int)n, stream));
    long long runs = 0;
    if (int rc = read_count(w.count_out, &runs, stream)) return rc;
    *n_unique_host = runs;
    return GLOVE_OK;
}

int glove_cooc_finish(const uint64_t *keys, const int64_t *agg, int64_t n, int32_t V, int32_t context, int64_t count_min,
                      const int64_t *vocab_count, int64_t total_tokens, uint64_t order_key, void *workspace,
                      size_t workspace_bytes, int32_t *row, int32_t *col, int64_t *count, double *value, double *neg_weight,
                      double *glove_weight, double *glove_value, int64_t capacity, int64_t *n_out_host, void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GLOVE_REQUIRE(keys && agg && vocab_count && workspace && n_out_host && n > 0, "glove_cooc_finish: bad arguments");
    GLOVE_REQUIRE(context >= 1 && context <= 8 && total_tokens > 0 && V > 1, "glove_cooc_finish: bad sizes");
    const int64_t n2 = 2 * n;
    GLOVE_REQUIRE(n2 < (1ll << 31), "glove_cooc_finish: more than 2^30 distinct pairs");
    const int vbits = vbits_of((int64_t)V + 1);
    const CoocWs w = cooc_ws_view(workspace, n2);
    if (workspace_bytes < w.bytes)
        return set_error(GLOVE_EWORKSPACE, "glove_cooc_finish: workspace %zu < required %zu", workspace_bytes, w.bytes);
    const unsigned g2 = (unsigned)((n2 + 255) / 256);
    // union with the transposed table, summed per (row, col)
    transpose_keys_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(keys, n, vbits, w.keys[0], w.idx[0]);
    GLOVE_CHECK_LAUNCH();
    size_t tb = w.cub_bytes;
    GLOVE_CHECK_CUDA(cub::DeviceRadixSort::SortPairs(w.cub_temp, tb, w.keys[0], w.keys[1], w.idx[0], w.idx[1], (int)n2, 0,
                                                     2 * vbits, stream));
    gather_agg_kernel<<<g2, 256, 0, stream>>>(w.idx[1], n2, (const Agg *)agg, n2, (const Agg *)agg, w.agg);
    GLOVE_CHECK_LAUNCH();
    tb = w.cub_bytes;
    GLOVE_CHECK_CUDA(cub::DeviceReduce::ReduceByKey(w.cub_temp, tb, w.keys[1], w.keys[0], w.agg, w.agg2, w.count_out, AggSum(),
                                                    (int)n2, stream));
    long long m = 0;
    if (int rc = read_count(w.count_out, &m, stream)) return rc;
    return finish_records("glove_cooc_finish", w.keys[0], w.agg2, m, w, vbits, context, count_min, vocab_count, total_tokens,
                          order_key, row, col, count, value, neg_weight, glove_weight, glove_value, capacity, n_out_host,
                          stream);
}

size_t glove_cooc_route_workspace_bytes(int64_t n, int32_t part_bits) {
    return route_ws_view(nullptr, 2 * (n < 1 ? 1 : n), part_bits < 0 ? 0 : part_bits > kCoocMaxPartBits ? kCoocMaxPartBits : part_bits).bytes;
}

int glove_cooc_route(const uint64_t *keys, const int64_t *agg, int64_t n, int32_t V, uint64_t order_key, int32_t part_bits,
                     void *workspace, size_t workspace_bytes, uint64_t *out_keys, int64_t *out_agg, int64_t capacity,
                     int64_t *part_count_host, void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GLOVE_REQUIRE(keys && agg && workspace && out_keys && out_agg && part_count_host, "glove_cooc_route: null pointer");
    GLOVE_REQUIRE(n > 0 && V > 1 && part_bits >= 0 && part_bits <= kCoocMaxPartBits,
                  "glove_cooc_route: bad sizes (part_bits must be 0..%d)", kCoocMaxPartBits);
    GLOVE_REQUIRE(2 * n < (1ll << 31), "glove_cooc_route: more than 2^30 entries");
    GLOVE_REQUIRE(capacity >= 2 * n, "glove_cooc_route: capacity %lld < 2n = %lld", (long long)capacity, (long long)(2 * n));
    return route_entries("glove_cooc_route", keys, agg, n, 2, V, order_key, part_bits, workspace, workspace_bytes, out_keys,
                         out_agg, part_count_host, stream);
}

int glove_cooc_route_stanford(const uint64_t *keys, const int64_t *agg, int64_t n, int32_t V, uint64_t order_key, int32_t part_bits,
                           int32_t symmetric, void *workspace, size_t workspace_bytes, uint64_t *out_keys, int64_t *out_agg,
                           int64_t capacity, int64_t *part_count_host, void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GLOVE_REQUIRE(keys && agg && workspace && out_keys && out_agg && part_count_host, "glove_cooc_route_stanford: null pointer");
    GLOVE_REQUIRE(n > 0 && V > 0 && part_bits >= 0 && part_bits <= kCoocMaxPartBits,
                  "glove_cooc_route_stanford: bad sizes (part_bits must be 0..%d)", kCoocMaxPartBits);
    GLOVE_REQUIRE(2 * n < (1ll << 31), "glove_cooc_route_stanford: more than 2^30 entries");
    const int n_orient = symmetric ? 2 : 1;
    GLOVE_REQUIRE(capacity >= n_orient * n, "glove_cooc_route_stanford: capacity %lld < %lld", (long long)capacity,
                  (long long)(n_orient * n));
    return route_entries("glove_cooc_route_stanford", keys, agg, n, n_orient, V, order_key, part_bits, workspace, workspace_bytes,
                         out_keys, out_agg, part_count_host, stream);
}

int glove_cooc_finish_sorted(const uint64_t *keys, const int64_t *agg, int64_t n, int32_t V, int32_t context, int64_t count_min,
                             const int64_t *vocab_count, int64_t total_tokens, uint64_t order_key, void *workspace,
                             size_t workspace_bytes, int32_t *row, int32_t *col, int64_t *count, double *value,
                             double *neg_weight, double *glove_weight, double *glove_value, int64_t capacity,
                             int64_t *n_out_host, void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GLOVE_REQUIRE(keys && agg && vocab_count && workspace && n_out_host && n > 0, "glove_cooc_finish_sorted: bad arguments");
    GLOVE_REQUIRE(context >= 1 && context <= 8 && total_tokens > 0 && V > 1, "glove_cooc_finish_sorted: bad sizes");
    GLOVE_REQUIRE(n < (1ll << 31), "glove_cooc_finish_sorted: more than 2^31 entries");
    const int vbits = vbits_of((int64_t)V + 1);
    const CoocWs w = cooc_ws_view(workspace, n);
    if (workspace_bytes < w.bytes)
        return set_error(GLOVE_EWORKSPACE, "glove_cooc_finish_sorted: workspace %zu < required %zu", workspace_bytes, w.bytes);
    return finish_records("glove_cooc_finish_sorted", keys, (const Agg *)agg, n, w, vbits, context, count_min, vocab_count,
                          total_tokens, order_key, row, col, count, value, neg_weight, glove_weight, glove_value, capacity,
                          n_out_host, stream);
}

int glove_cooc_finish_stanford(const uint64_t *keys, const int64_t *agg, int64_t n, int32_t V, int32_t window,
                            int32_t distance_weighting, const int64_t *vocab_count, int64_t total_tokens, uint64_t order_key,
                            void *workspace, size_t workspace_bytes, int32_t *row, int32_t *col, int64_t *count, double *value,
                            double *neg_weight, double *glove_weight, double *glove_value, int64_t capacity,
                            int64_t *n_out_host, void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GLOVE_REQUIRE(keys && agg && vocab_count && workspace && n_out_host && n > 0, "glove_cooc_finish_stanford: bad arguments");
    GLOVE_REQUIRE(window >= 1 && window <= kStanfordMaxWindow && total_tokens > 0 && V > 0,
                  "glove_cooc_finish_stanford: bad sizes (window must be 1..%d)", kStanfordMaxWindow);
    GLOVE_REQUIRE(n < (1ll << 31), "glove_cooc_finish_stanford: more than 2^31 entries");
    const int vbits = vbits_of((int64_t)V + 1);
    const CoocWs w = cooc_ws_view(workspace, n);
    if (workspace_bytes < w.bytes)
        return set_error(GLOVE_EWORKSPACE, "glove_cooc_finish_stanford: workspace %zu < required %zu", workspace_bytes, w.bytes);
    // every pair is a record (count_min 1); value = numer / lcm(1..window), or count with unit weights
    return finish_records("glove_cooc_finish_stanford", keys, (const Agg *)agg, n, w, vbits, distance_weighting ? window : 1, 1,
                          vocab_count, total_tokens, order_key, row, col, count, value, neg_weight, glove_weight, glove_value,
                          capacity, n_out_host, stream);
}

}  // extern "C"
