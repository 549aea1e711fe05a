// Streamed corpus preprocessing (corpus.py): the parts of the two-pass preprocessor that the in-memory path
// (text8.process_data + save_data) does not need.
//
//   vocab_merge   pass 1: merges the distinct tokens of one text chunk (glove_tokens_count) into the global table of
//                 distinct tokens kept on the device, sorted by 64-bit token hash: {hash, count, global byte offset of
//                 the first occurrence, offset and length of the token bytes in a device string pool}.  The bytes are
//                 kept because earlier chunks are no longer resident; equal hashes are compared byte by byte and a
//                 collision fails the call.  Tokens seen for the first time append their bytes to the pool.
//   cooc_csv      interaction.csv lines of a block of finished records, formatted on the device: one kernel measures the
//                 lines, a scan gives their offsets, a second kernel writes them.  Tokens are copied from a pool the host
//                 has already quoted the way pandas' QUOTE_MINIMAL does; float64 columns print as repr(float)
//                 (glove_dtoa.cuh), the way pandas writes them.
//
// Integer / byte work around CUB sorts and scans; no tensor cores.
#include <cub/cub.cuh>

#include "glove_common.cuh"
#include "glove_dtoa.cuh"

namespace glove {

// the token hash of glove_tokens_count (FNV-1a, then a finalising mix)
__device__ __forceinline__ uint64_t token_hash64(const uint8_t *p, int32_t n) {
    uint64_t h = 0xcbf29ce484222325ull;
    for (int32_t i = 0; i < n; ++i) h = (h ^ p[i]) * 0x100000001b3ull;
    h ^= h >> 29; h *= 0xbf58476d1ce4e5b9ull; h ^= h >> 32;
    return h;
}

struct VmWs {
    uint64_t *keys[2];
    uint32_t *idx[2];
    int64_t *head, *head_off, *new_len, *new_off;
    int32_t *bad;
    void *cub_temp;
    size_t cub_bytes, bytes;
};
static VmWs vm_ws_view(void *base, int64_t n) {
    VmWs w;
    char *p = (char *)base;
    size_t off = 0;
    auto take = [&](size_t bytes) { char *r = p ? p + off : nullptr; off += align_up(bytes); return r; };
    for (int i = 0; i < 2; ++i) w.keys[i] = (uint64_t *)take(8 * n);
    for (int i = 0; i < 2; ++i) w.idx[i] = (uint32_t *)take(4 * n);
    w.head = (int64_t *)take(8 * (n + 1));
    w.head_off = (int64_t *)take(8 * (n + 1));
    w.new_len = (int64_t *)take(8 * (n + 1));
    w.new_off = (int64_t *)take(8 * (n + 1));
    w.bad = (int32_t *)take(4);
    size_t a = 0, b = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, a, (uint64_t *)nullptr, (uint64_t *)nullptr, (uint32_t *)nullptr, (uint32_t *)nullptr,
                                    (int)n);
    cub::DeviceScan::ExclusiveSum(nullptr, b, (int64_t *)nullptr, (int64_t *)nullptr, (int)(n + 1));
    w.cub_bytes = a > b ? a : b;
    w.cub_temp = take(w.cub_bytes);
    w.bytes = off;
    return w;
}

// entries 0 .. n_g-1: the global table; n_g .. n_g+m-1: the chunk's distinct tokens
__global__ void __launch_bounds__(256) vm_keys_kernel(const uint8_t *__restrict__ text, const int64_t *__restrict__ first,
                                                      const int32_t *__restrict__ flen, int64_t m,
                                                      const uint64_t *__restrict__ g_hash, int64_t n_g, uint64_t *keys,
                                                      uint32_t *idx) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_g + m) return;
    keys[i] = i < n_g ? g_hash[i] : token_hash64(text + first[i - n_g], flen[i - n_g]);
    idx[i] = (uint32_t)i;
}
// sorted (stable: a global entry precedes the chunk entry of the same hash; each side has distinct hashes, so a run
// holds one or two entries).  head = first of its run; a chunk entry that heads its run is a new token.
__global__ void __launch_bounds__(256) vm_flags_kernel(const uint64_t *__restrict__ keys, const uint32_t *__restrict__ idx,
                                                       int64_t n, int64_t n_g, const uint8_t *__restrict__ text,
                                                       const int64_t *__restrict__ first, const int32_t *__restrict__ flen,
                                                       const uint8_t *__restrict__ pool, const int64_t *__restrict__ g_off,
                                                       const int32_t *__restrict__ g_len, int64_t *head, int64_t *new_len,
                                                       int32_t *bad) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n) return;
    if (i == n) { head[n] = 0; new_len[n] = 0; return; }
    const bool h = i == 0 || keys[i] != keys[i - 1];
    const int64_t j = idx[i];
    head[i] = h;
    new_len[i] = h && j >= n_g ? flen[j - n_g] : 0;
    if (!h) {
        const int64_t a = idx[i - 1], c = j - n_g;
        bool same = a < n_g && c >= 0 && g_len[a] == flen[c];
        for (int32_t k = 0; same && k < flen[c]; ++k) same = pool[g_off[a] + k] == text[first[c] + k];
        if (!same) *bad = 1;
    }
}
__global__ void __launch_bounds__(256) vm_write_kernel(const uint64_t *__restrict__ keys, const uint32_t *__restrict__ idx,
                                                       int64_t n, int64_t n_g, const int64_t *__restrict__ head,
                                                       const int64_t *__restrict__ head_off, const int64_t *__restrict__ new_off,
                                                       const uint8_t *__restrict__ text, int64_t origin,
                                                       const int64_t *__restrict__ first, const int32_t *__restrict__ flen,
                                                       const int64_t *__restrict__ c_count, const int64_t *__restrict__ g_count,
                                                       const int64_t *__restrict__ g_first, const int64_t *__restrict__ g_off,
                                                       const int32_t *__restrict__ g_len, uint8_t *pool, int64_t pool_used,
                                                       uint64_t *o_hash, int64_t *o_count, int64_t *o_first, int64_t *o_off,
                                                       int32_t *o_len) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || !head[i]) return;
    const int64_t o = head_off[i], j = idx[i];
    o_hash[o] = keys[i];
    if (j < n_g) {
        const bool dup = i + 1 < n && !head[i + 1];
        o_count[o] = g_count[j] + (dup ? c_count[idx[i + 1] - n_g] : 0);
        o_first[o] = g_first[j];
        o_off[o] = g_off[j];
        o_len[o] = g_len[j];
        return;
    }
    const int64_t c = j - n_g, dst = pool_used + new_off[i];
    o_count[o] = c_count[c];
    o_first[o] = origin + first[c];
    o_off[o] = dst;
    o_len[o] = flen[c];
    for (int32_t k = 0; k < flen[c]; ++k) pool[dst + k] = text[first[c] + k];
}

// ---- interaction.csv lines --------------------------------------------------------------------------------------------
__device__ __forceinline__ int dec_len(int64_t v) {
    uint64_t u = v < 0 ? (uint64_t)(-(v + 1)) + 1 : (uint64_t)v;
    int n = v < 0 ? 2 : 1;
    while (u >= 10) { u /= 10; ++n; }
    return n;
}
__device__ __forceinline__ uint8_t *put_dec(uint8_t *o, int64_t v) {
    const int n = dec_len(v);
    uint64_t u = v < 0 ? (uint64_t)(-(v + 1)) + 1 : (uint64_t)v;
    if (v < 0) *o = '-';
    for (int k = n - 1; k >= (v < 0 ? 1 : 0); --k) { o[k] = (uint8_t)('0' + u % 10); u /= 10; }
    return o + n;
}
__device__ __forceinline__ int f64_len(double x) {
    char buf[kF64TextMax];
    return format_f64((uint64_t)__double_as_longlong(x), buf);
}
__device__ __forceinline__ uint8_t *put_f64(uint8_t *o, double x) {
    char buf[kF64TextMax];
    const int n = format_f64((uint64_t)__double_as_longlong(x), buf);
    for (int k = 0; k < n; ++k) o[k] = (uint8_t)buf[k];
    return o + n;
}
struct CsvCols {
    const int32_t *row, *col;
    const int64_t *count;
    const double *value, *neg_weight, *glove_weight, *glove_value;
};
// row_token_id,col_token_id,count,value,row_token,col_token,neg_weight,glove_weight,glove_value\n
__global__ void __launch_bounds__(128) csv_len_kernel(CsvCols c, int64_t n, const int64_t *__restrict__ tok_off, int64_t *len) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n) return;
    if (i == n) { len[n] = 0; return; }
    const int32_t a = c.row[i], b = c.col[i];
    len[i] = dec_len(a) + dec_len(b) + dec_len(c.count[i]) + f64_len(c.value[i]) + (tok_off[a + 1] - tok_off[a]) +
             (tok_off[b + 1] - tok_off[b]) + f64_len(c.neg_weight[i]) + f64_len(c.glove_weight[i]) +
             f64_len(c.glove_value[i]) + 9;
}
__global__ void __launch_bounds__(128) csv_write_kernel(CsvCols c, int64_t n, const uint8_t *__restrict__ tok,
                                                        const int64_t *__restrict__ tok_off, const int64_t *__restrict__ offs,
                                                        uint8_t *text) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int32_t a = c.row[i], b = c.col[i];
    uint8_t *o = text + offs[i];
    o = put_dec(o, a); *o++ = ',';
    o = put_dec(o, b); *o++ = ',';
    o = put_dec(o, c.count[i]); *o++ = ',';
    o = put_f64(o, c.value[i]); *o++ = ',';
    for (int64_t k = tok_off[a]; k < tok_off[a + 1]; ++k) *o++ = tok[k];
    *o++ = ',';
    for (int64_t k = tok_off[b]; k < tok_off[b + 1]; ++k) *o++ = tok[k];
    *o++ = ',';
    o = put_f64(o, c.neg_weight[i]); *o++ = ',';
    o = put_f64(o, c.glove_weight[i]); *o++ = ',';
    o = put_f64(o, c.glove_value[i]);
    *o = '\n';
}

__global__ void __launch_bounds__(256) format_f64_kernel(const uint64_t *__restrict__ bits, int64_t n, char *out, int32_t *len) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) len[i] = format_f64(bits[i], out + i * kF64TextMax);
}

struct CsvWs {
    int64_t *len, *offs;
    void *cub_temp;
    size_t cub_bytes, bytes;
};
static CsvWs csvw_view(void *base, int64_t n) {
    CsvWs w;
    char *p = (char *)base;
    size_t off = 0;
    auto take = [&](size_t bytes) { char *r = p ? p + off : nullptr; off += align_up(bytes); return r; };
    w.len = (int64_t *)take(8 * (n + 1));
    w.offs = (int64_t *)take(8 * (n + 1));
    w.cub_bytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, w.cub_bytes, (int64_t *)nullptr, (int64_t *)nullptr, (int)(n + 1));
    w.cub_temp = take(w.cub_bytes);
    w.bytes = off;
    return w;
}

}  // namespace glove

using namespace glove;

extern "C" {

size_t glove_vocab_merge_workspace_bytes(int64_t n_global, int64_t n_chunk) {
    const int64_t n = (n_global < 0 ? 0 : n_global) + (n_chunk < 0 ? 0 : n_chunk);
    return vm_ws_view(nullptr, n < 1 ? 1 : n).bytes;
}

int glove_vocab_merge(const uint8_t *text, int64_t origin, const int64_t *first, const int32_t *first_len, const int64_t *count,
                      int64_t n_chunk, const uint64_t *g_hash, const int64_t *g_count, const int64_t *g_first,
                      const int64_t *g_off, const int32_t *g_len, int64_t n_global, uint8_t *pool, int64_t pool_used,
                      int64_t pool_capacity, void *workspace, size_t workspace_bytes, uint64_t *o_hash, int64_t *o_count,
                      int64_t *o_first, int64_t *o_off, int32_t *o_len, int64_t capacity, int64_t *n_out_host,
                      int64_t *pool_used_host, void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GLOVE_REQUIRE(text && first && first_len && count && pool && workspace && o_hash && o_count && o_first && o_off && o_len &&
                      n_out_host && pool_used_host, "glove_vocab_merge: null pointer");
    GLOVE_REQUIRE(n_global >= 0 && n_chunk > 0 && origin >= 0 && pool_used >= 0 && pool_used <= pool_capacity,
                  "glove_vocab_merge: bad sizes");
    GLOVE_REQUIRE(n_global == 0 || (g_hash && g_count && g_first && g_off && g_len), "glove_vocab_merge: null global table");
    const int64_t n = n_global + n_chunk;
    GLOVE_REQUIRE(n < (1ll << 31), "glove_vocab_merge: more than 2^31 distinct tokens");
    const VmWs w = vm_ws_view(workspace, n);
    if (workspace_bytes < w.bytes)
        return set_error(GLOVE_EWORKSPACE, "glove_vocab_merge: workspace %zu < required %zu", workspace_bytes, w.bytes);
    GLOVE_CHECK_CUDA(cudaMemsetAsync(w.bad, 0, 4, stream));
    vm_keys_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(text, first, first_len, n_chunk, g_hash, n_global, w.keys[0],
                                                                    w.idx[0]);
    GLOVE_CHECK_LAUNCH();
    size_t tb = w.cub_bytes;
    GLOVE_CHECK_CUDA(cub::DeviceRadixSort::SortPairs(w.cub_temp, tb, w.keys[0], w.keys[1], w.idx[0], w.idx[1], (int)n, 0, 64,
                                                     stream));
    vm_flags_kernel<<<(unsigned)((n + 1 + 255) / 256), 256, 0, stream>>>(w.keys[1], w.idx[1], n, n_global, text, first, first_len,
                                                                         pool, g_off, g_len, w.head, w.new_len, w.bad);
    GLOVE_CHECK_LAUNCH();
    tb = w.cub_bytes;
    GLOVE_CHECK_CUDA(cub::DeviceScan::ExclusiveSum(w.cub_temp, tb, w.head, w.head_off, (int)(n + 1), stream));
    tb = w.cub_bytes;
    GLOVE_CHECK_CUDA(cub::DeviceScan::ExclusiveSum(w.cub_temp, tb, w.new_len, w.new_off, (int)(n + 1), stream));
    int64_t n_out = 0, new_bytes = 0;
    int32_t bad = 0;
    GLOVE_CHECK_CUDA(cudaMemcpyAsync(&n_out, w.head_off + n, 8, cudaMemcpyDeviceToHost, stream));
    GLOVE_CHECK_CUDA(cudaMemcpyAsync(&new_bytes, w.new_off + n, 8, cudaMemcpyDeviceToHost, stream));
    GLOVE_CHECK_CUDA(cudaMemcpyAsync(&bad, w.bad, 4, cudaMemcpyDeviceToHost, stream));
    GLOVE_CHECK_CUDA(cudaStreamSynchronize(stream));
    if (bad) return set_error(GLOVE_EUNSUPPORTED, "glove_vocab_merge: two different tokens share a 64-bit hash");
    *n_out_host = n_out;
    *pool_used_host = pool_used + new_bytes;
    if (n_out > capacity)
        return set_error(GLOVE_EINVAL, "glove_vocab_merge: %lld distinct tokens > capacity %lld", (long long)n_out,
                         (long long)capacity);
    if (pool_used + new_bytes > pool_capacity)
        return set_error(GLOVE_EINVAL, "glove_vocab_merge: token pool needs %lld bytes > capacity %lld",
                         (long long)(pool_used + new_bytes), (long long)pool_capacity);
    vm_write_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(
        w.keys[1], w.idx[1], n, n_global, w.head, w.head_off, w.new_off, text, origin, first, first_len, count, g_count, g_first,
        g_off, g_len, pool, pool_used, o_hash, o_count, o_first, o_off, o_len);
    GLOVE_CHECK_LAUNCH();
    GLOVE_CHECK_CUDA(cudaStreamSynchronize(stream));
    return GLOVE_OK;
}

size_t glove_cooc_csv_workspace_bytes(int64_t n_records) { return csvw_view(nullptr, n_records < 1 ? 1 : n_records).bytes; }

int glove_cooc_csv_size(const int32_t *row, const int32_t *col, const int64_t *count, const double *value,
                        const double *neg_weight, const double *glove_weight, const double *glove_value, int64_t n,
                        const int64_t *token_off, void *workspace, size_t workspace_bytes, int64_t *text_bytes_host,
                        void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GLOVE_REQUIRE(row && col && count && value && neg_weight && glove_weight && glove_value && token_off && workspace &&
                      text_bytes_host, "glove_cooc_csv_size: null pointer");
    GLOVE_REQUIRE(n > 0 && n < (1ll << 31), "glove_cooc_csv_size: n must be 1 .. 2^31-1");
    const CsvWs w = csvw_view(workspace, n);
    if (workspace_bytes < w.bytes)
        return set_error(GLOVE_EWORKSPACE, "glove_cooc_csv_size: workspace %zu < required %zu", workspace_bytes, w.bytes);
    const CsvCols c = {row, col, count, value, neg_weight, glove_weight, glove_value};
    csv_len_kernel<<<(unsigned)((n + 1 + 127) / 128), 128, 0, stream>>>(c, n, token_off, w.len);
    GLOVE_CHECK_LAUNCH();
    size_t tb = w.cub_bytes;
    GLOVE_CHECK_CUDA(cub::DeviceScan::ExclusiveSum(w.cub_temp, tb, w.len, w.offs, (int)(n + 1), stream));
    GLOVE_CHECK_CUDA(cudaMemcpyAsync(text_bytes_host, w.offs + n, 8, cudaMemcpyDeviceToHost, stream));
    GLOVE_CHECK_CUDA(cudaStreamSynchronize(stream));
    return GLOVE_OK;
}

int glove_cooc_csv_format(const int32_t *row, const int32_t *col, const int64_t *count, const double *value,
                          const double *neg_weight, const double *glove_weight, const double *glove_value, int64_t n,
                          const uint8_t *token_bytes, const int64_t *token_off, void *workspace, size_t workspace_bytes,
                          uint8_t *text, int64_t capacity, void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GLOVE_REQUIRE(row && col && count && value && neg_weight && glove_weight && glove_value && token_bytes && token_off &&
                      workspace && text, "glove_cooc_csv_format: null pointer");
    GLOVE_REQUIRE(n > 0 && n < (1ll << 31) && capacity >= 0, "glove_cooc_csv_format: bad sizes");
    const CsvWs w = csvw_view(workspace, n);
    if (workspace_bytes < w.bytes)
        return set_error(GLOVE_EWORKSPACE, "glove_cooc_csv_format: workspace %zu < required %zu", workspace_bytes, w.bytes);
    int64_t need = 0;
    GLOVE_CHECK_CUDA(cudaMemcpyAsync(&need, w.offs + n, 8, cudaMemcpyDeviceToHost, stream));
    GLOVE_CHECK_CUDA(cudaStreamSynchronize(stream));
    if (need > capacity)
        return set_error(GLOVE_EINVAL, "glove_cooc_csv_format: %lld bytes of text > capacity %lld", (long long)need,
                         (long long)capacity);
    const CsvCols c = {row, col, count, value, neg_weight, glove_weight, glove_value};
    csv_write_kernel<<<(unsigned)((n + 127) / 128), 128, 0, stream>>>(c, n, token_bytes, token_off, w.offs, text);
    GLOVE_CHECK_LAUNCH();
    return GLOVE_OK;
}

int glove_format_float64(double value, char *out, int32_t capacity, int32_t *length) {
    GLOVE_REQUIRE(out && length && capacity >= kF64TextMax, "glove_format_float64: out must hold %d bytes", kF64TextMax);
    uint64_t bits;
    memcpy(&bits, &value, 8);
    *length = format_f64(bits, out);
    return GLOVE_OK;
}

// device build of the same formatter, for tests: n bit patterns -> n slots of kF64TextMax bytes, lengths in len.
// Asynchronous.
int glove_format_float64_device(const uint64_t *bits, int64_t n, char *out, int32_t *len, void *stream) {
    GLOVE_REQUIRE(bits && out && len && n > 0, "glove_format_float64_device: bad arguments");
    format_f64_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(bits, n, out, len);
    GLOVE_CHECK_LAUNCH();
    return GLOVE_OK;
}

}  // extern "C"
