// WORD VECTORS: the GloVe text format (``word v_1 ... v_d`` per line, optional word2vec header) <-> device float32 rows.
//
// Import, per chunk of the file (the caller streams the file and carries the unterminated tail of a chunk into the next):
//   nl_count_kernel     one pass over the text: '\n' count per 16 KB tile (no quoting in this format: a plain count)
//   cub ExclusiveSum    tile offsets = index of the first line ending in each tile
//   line_ends_kernel    second pass: position of every '\n'
//   line_flags_kernel   one thread per line: blank (only spaces, tabs, a final '\r') or not
//   cub ExclusiveSum    row id of every non-blank line
//   parse_lines_kernel  one warp per line: the lanes load the line in 16-byte pieces from the right, find field starts
//                       and ends as bit masks (warp shuffles across the pieces), rank them from the right, deal the
//                       last d fields to the lanes (parse_f32 of glove_strtof.cuh: one correct rounding) and write them
//                       to out + row * ld; the word is everything before them (start, length) -- the rsplit rule
// Export, per block of rows:
//   format_len_kernel   one warp per row: byte length of its line (word + d shortest-decimal values, glove_ftoa.cuh)
//   cub ExclusiveSum    line offsets
//   format_write_kernel one warp per row: each lane formats a run of values and writes it at its offset
// Byte work bound by HBM and integer throughput: no tensor cores.  Errors never fall back to the host: the lowest
// offending line of the chunk is reported.
#include <cub/cub.cuh>

#include "glove_common.cuh"
#include "glove_ftoa.cuh"
#include "glove_strtof.cuh"

namespace glove {

constexpr int kNlThreads = 256, kNlThreadBytes = 64, kNlTileBytes = kNlThreads * kNlThreadBytes;
constexpr int kMaxVecDim = 510;
constexpr int kParseWarps = 4;

enum { VEC_OK = 0, VEC_EFIELDS = 1, VEC_ENUMBER = 2, VEC_EDIGITS = 3, VEC_ENONFINITE = 4, VEC_ECOUNT = 5 };
struct VecStatus {
    unsigned long long first_error;   // (line << 8) | code, minimum over all lines; ~0 = none
    long long n_nl;                   // '\n' in the chunk
    long long last_end;               // position of the last '\n' (-1: none)
};

struct VecWs {
    VecStatus *status;
    int64_t *tile_cnt;    // [n_tiles + 1]
    int64_t *tile_off;    // [n_tiles + 1]
    int64_t *ends;        // [n_lines + 1] line ends (parse) / line lengths (format)
    int64_t *flags;       // [n_lines + 1] non-blank lines (parse)
    int64_t *offs;        // [n_lines + 1] row of every line (parse) / line offsets (format)
    void *cub_temp;
    size_t cub_bytes, bytes;
};
static int64_t vec_tiles(int64_t nbytes) { return (nbytes + kNlTileBytes - 1) / kNlTileBytes; }
// the same prefix (status, tile arrays) for every n_lines: glove_vectors_parse reads what glove_vectors_index left there
static VecWs vec_ws_view(void *base, int64_t nbytes, int64_t n_lines) {
    VecWs w;
    char *p = (char *)base;
    size_t off = 0;
    auto take = [&](size_t bytes) { char *r = p ? p + off : nullptr; off += align_up(bytes); return r; };
    const int64_t nt = vec_tiles(nbytes) + 1, nl = n_lines + 1;
    w.status = (VecStatus *)take(sizeof(VecStatus));
    w.tile_cnt = (int64_t *)take(8 * nt);
    w.tile_off = (int64_t *)take(8 * nt);
    w.ends = (int64_t *)take(8 * nl);
    w.flags = (int64_t *)take(8 * nl);
    w.offs = (int64_t *)take(8 * nl);
    size_t a = 0, b = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, a, (int64_t *)nullptr, (int64_t *)nullptr, (int)nt);
    cub::DeviceScan::ExclusiveSum(nullptr, b, (int64_t *)nullptr, (int64_t *)nullptr, (int)nl);
    w.cub_bytes = a > b ? a : b;
    w.cub_temp = take(w.cub_bytes);
    w.bytes = off;
    return w;
}

__device__ __forceinline__ bool is_blank(uint8_t c) { return c == ' ' || c == '\t'; }

// the 16 bytes at an aligned position p (zero outside [0, nbytes): NUL is neither a newline nor a blank)
__device__ __forceinline__ uint4 load16(const uint8_t *text, int64_t nbytes, int64_t p) {
    if (p >= 0 && p + 16 <= nbytes) return __ldg((const uint4 *)(text + p));
    uint8_t b[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) b[k] = p + k >= 0 && p + k < nbytes ? text[p + k] : 0;
    return *(const uint4 *)b;
}
__device__ __forceinline__ int nl_in(uint4 v) {
    return (__popc(__vcmpeq4(v.x, 0x0a0a0a0au)) + __popc(__vcmpeq4(v.y, 0x0a0a0a0au)) + __popc(__vcmpeq4(v.z, 0x0a0a0a0au)) +
            __popc(__vcmpeq4(v.w, 0x0a0a0a0au))) >> 3;
}
__device__ __forceinline__ uint8_t byte_of(const uint4 &v, int i) {
    const uint32_t w = (&v.x)[i >> 2];
    return (uint8_t)(w >> (8 * (i & 3)));
}

__global__ void __launch_bounds__(kNlThreads) nl_count_kernel(const uint8_t *__restrict__ text, int64_t nbytes, int64_t n_tiles,
                                                              int64_t *tile_cnt) {
    const int64_t base = (int64_t)blockIdx.x * kNlTileBytes + (int64_t)threadIdx.x * kNlThreadBytes;
    int c = 0;
#pragma unroll
    for (int u = 0; u < 4; ++u) c += nl_in(load16(text, nbytes, base + 16 * u));
    typedef cub::BlockReduce<int, kNlThreads> Reduce;
    __shared__ typename Reduce::TempStorage tmp;
    const int total = Reduce(tmp).Sum(c);
    if (threadIdx.x == 0) {
        tile_cnt[blockIdx.x] = total;
        if (blockIdx.x == 0) tile_cnt[n_tiles] = 0;
    }
}

__global__ void __launch_bounds__(kNlThreads) line_ends_kernel(const uint8_t *__restrict__ text, int64_t nbytes,
                                                               const int64_t *__restrict__ tile_off, int64_t *ends,
                                                               VecStatus *st) {
    const int64_t base = (int64_t)blockIdx.x * kNlTileBytes + (int64_t)threadIdx.x * kNlThreadBytes;
    uint4 v[4];
    int c = 0;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        v[u] = load16(text, nbytes, base + 16 * u);
        c += nl_in(v[u]);
    }
    typedef cub::BlockScan<int, kNlThreads> Scan;
    __shared__ typename Scan::TempStorage tmp;
    int excl;
    Scan(tmp).ExclusiveSum(c, excl);
    if (!c) return;
    int64_t r = tile_off[blockIdx.x] + excl;
    const int64_t n_nl = st->n_nl;
#pragma unroll
    for (int i = 0; i < kNlThreadBytes; ++i)
        if (byte_of(v[i >> 4], i & 15) == '\n') {
            ends[r] = base + i;
            if (r == n_nl - 1) st->last_end = base + i;
            ++r;
        }
}

// line i = [ends[i-1] + 1, ends[i]); flag = 1 unless it holds nothing but blanks and one final '\r'
__global__ void __launch_bounds__(256) line_flags_kernel(const uint8_t *__restrict__ text, const int64_t *__restrict__ ends,
                                                         int64_t n_lines, int64_t *flags) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n_lines) return;
    if (i == n_lines) { flags[i] = 0; return; }
    const int64_t b = i ? ends[i - 1] + 1 : 0;
    int64_t e = ends[i];
    if (e > b && text[e - 1] == '\r') --e;
    while (e > b && is_blank(text[e - 1])) --e;
    flags[i] = e > b;
}

__device__ __forceinline__ void vec_report(VecStatus *st, int64_t line, int code) {
    atomicMin(&st->first_error, ((unsigned long long)line << 8) | (unsigned)code);
}

// one warp per line.  Windows of 32 x 16 bytes are scanned from the line's end towards its start; in a window lane l holds
// the aligned piece at base + 16 l.  Bytes outside the line count as blanks.  A field START is a non-blank byte after a
// blank, a field END a non-blank byte before one; both are ranked from the right (rank 0 = the last field), and the field
// of rank r < d is value d - 1 - r.  The end of rank d closes the word.
__global__ void __launch_bounds__(kParseWarps * 32) parse_lines_kernel(
    const uint8_t *__restrict__ text, int64_t nbytes, const int64_t *__restrict__ ends, const int64_t *__restrict__ flags,
    const int64_t *__restrict__ row_of, int64_t n_lines, int32_t d, float *out, int64_t ld, int64_t row_cap,
    int64_t *word_start, int32_t *word_len, int64_t first_line, VecStatus *st) {
    __shared__ int32_t fs[kParseWarps][kMaxVecDim], fe[kParseWarps][kMaxVecDim];
    __shared__ int64_t wend_sh[kParseWarps];
    const int wi = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t i = (int64_t)blockIdx.x * kParseWarps + wi;
    if (i >= n_lines || !flags[i]) return;
    const int64_t b = i ? ends[i - 1] + 1 : 0;
    int64_t e = ends[i];
    if (e > b && text[e - 1] == '\r') --e;
    const int64_t row = row_of[i];
    if (row >= row_cap) {
        if (lane == 0) vec_report(st, first_line + i, VEC_ECOUNT);
        return;
    }
    if (lane == 0) wend_sh[wi] = -1;
    __syncwarp();
    int n_starts = 0, n_ends = 0;   // fields seen so far (whole warp, uniform)
    for (int64_t base = ((e - 1) & ~(int64_t)15) - 31 * 16;; base -= 32 * 16) {
        const int64_t p = base + 16 * lane;
        uint32_t nb = 0;   // bit j: byte p + j is inside the line and not blank
        if (p + 16 > b && p < e) {
            const uint4 v = load16(text, nbytes, p);
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const int64_t q = p + j;
                if (q >= b && q < e && !is_blank(byte_of(v, j))) nb |= 1u << j;
            }
        }
        // neighbours across the pieces: byte p - 1 (lane 0: in the next window to the left) and byte p + 16
        uint32_t before = __shfl_up_sync(0xffffffffu, nb >> 15, 1);
        uint32_t after = __shfl_down_sync(0xffffffffu, nb & 1, 1);
        if (lane == 0) before = p - 1 >= b && p - 1 < e && !is_blank(text[p - 1]);
        if (lane == 31) after = p + 16 >= b && p + 16 < e && !is_blank(text[p + 16]);
        const uint32_t starts = nb & ~((nb << 1) | before);
        const uint32_t fends = nb & ~((nb >> 1) | (after << 15));
        // ranks from the right: the fields of the lanes above come first (suffix sums over the lanes)
        const int cs = __popc(starts), ce = __popc(fends);
        int ss = cs, se = ce;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int s2 = __shfl_down_sync(0xffffffffu, ss, o), e2 = __shfl_down_sync(0xffffffffu, se, o);
            if (lane + o < 32) { ss += s2; se += e2; }
        }
        const int above_s = ss - cs, above_e = se - ce;
        for (uint32_t m = starts; m;) {
            const int j = 31 - __clz(m);
            m &= ~(1u << j);
            const int r = n_starts + above_s + __popc(starts >> j >> 1);
            if (r < d) fs[wi][d - 1 - r] = (int32_t)(p + j - b);
        }
        for (uint32_t m = fends; m;) {
            const int j = 31 - __clz(m);
            m &= ~(1u << j);
            const int r = n_ends + above_e + __popc(fends >> j >> 1);
            if (r < d) fe[wi][d - 1 - r] = (int32_t)(p + j + 1 - b);
            else if (r == d) wend_sh[wi] = p + j + 1 - b;
        }
        n_starts += __shfl_sync(0xffffffffu, ss, 0);
        n_ends += __shfl_sync(0xffffffffu, se, 0);
        if (n_ends > d || base <= b) break;
    }
    __syncwarp();
    const int64_t wend = wend_sh[wi];
    if (wend <= 0) {   // fewer than d + 1 fields
        if (lane == 0) vec_report(st, first_line + i, VEC_EFIELDS);
        return;
    }
    const uint8_t *line = text + b;
    float *dst = out + row * ld;
    for (int j = lane; j < d; j += 32) {
        const int s = fs[wi][j], n = fe[wi][j] - s;
        const uint8_t *f = line + s;
        uint32_t bits;
        const int rc = parse_f32([f](int k) { return (int)__ldg(f + k); }, n, bits);
        if (rc != STRTOF_OK) vec_report(st, first_line + i, rc == STRTOF_TOO_LONG ? VEC_EDIGITS : VEC_ENUMBER);
        else if ((bits & 0x7f800000u) == 0x7f800000u) vec_report(st, first_line + i, VEC_ENONFINITE);
        else dst[j] = __uint_as_float(bits);
    }
    if (lane == 0) {
        word_start[row] = b;
        word_len[row] = (int32_t)wend;
    }
}

// ---- export -----------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int f32_len(float x) {
    char buf[kF32TextMax];
    return format_f32(__float_as_uint(x), buf);
}

__global__ void __launch_bounds__(128) format_len_kernel(const float *__restrict__ rows, int64_t ld, int32_t d, int64_t n,
                                                         const int64_t *__restrict__ word_off, int64_t *len) {
    const int64_t r = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (r > n) return;
    if (r == n) {
        if (lane == 0) len[n] = 0;
        return;
    }
    const float *x = rows + r * ld;
    int64_t s = 0;
    for (int j = lane; j < d; j += 32) s += 1 + f32_len(__ldg(x + j));
#pragma unroll
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) len[r] = (word_off[r + 1] - word_off[r]) + s + 1;
}

__global__ void __launch_bounds__(128) format_write_kernel(const float *__restrict__ rows, int64_t ld, int32_t d, int64_t n,
                                                           const uint8_t *__restrict__ words,
                                                           const int64_t *__restrict__ word_off,
                                                           const int64_t *__restrict__ line_off, uint8_t *out) {
    const int64_t r = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (r >= n) return;
    const float *x = rows + r * ld;
    const int64_t w0 = word_off[r], wl = word_off[r + 1] - w0;
    uint8_t *dst = out + line_off[r];
    for (int64_t k = lane; k < wl; k += 32) dst[k] = words[w0 + k];
    // lane l writes the values [l q, (l + 1) q): the run lengths first, then a scan for their positions
    const int q = (d + 31) / 32, j0 = lane * q, j1 = min(d, j0 + q);
    int run = 0;
    for (int j = j0; j < j1; ++j) run += 1 + f32_len(__ldg(x + j));
    int incl = run;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    uint8_t *o = dst + wl + (incl - run);
    for (int j = j0; j < j1; ++j) {
        char buf[kF32TextMax];
        const int m = format_f32(__float_as_uint(__ldg(x + j)), buf);
        *o++ = ' ';
        for (int k = 0; k < m; ++k) *o++ = (uint8_t)buf[k];
    }
    if (lane == 31) dst[wl + incl] = '\n';
}

}  // namespace glove

using namespace glove;

extern "C" {

size_t glove_vectors_workspace_bytes(int64_t nbytes, int64_t n_lines) {
    return vec_ws_view(nullptr, nbytes < 1 ? 1 : nbytes, n_lines < 0 ? 0 : n_lines).bytes;
}

int glove_vectors_index(const uint8_t *text, int64_t nbytes, void *workspace, size_t workspace_bytes, int64_t *n_lines_host,
                        void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GLOVE_REQUIRE(text && workspace && n_lines_host, "glove_vectors_index: null pointer");
    GLOVE_REQUIRE(nbytes > 0 && nbytes < (1ll << 31), "glove_vectors_index: chunk must hold 1 .. 2^31-1 bytes");
    GLOVE_REQUIRE(((uintptr_t)text & 15) == 0, "glove_vectors_index: text must be 16-byte aligned");
    const VecWs w = vec_ws_view(workspace, nbytes, 0);
    if (workspace_bytes < w.bytes)
        return set_error(GLOVE_EWORKSPACE, "glove_vectors_index: workspace %zu < required %zu", workspace_bytes, w.bytes);
    const int64_t nt = vec_tiles(nbytes);
    nl_count_kernel<<<(unsigned)nt, kNlThreads, 0, stream>>>(text, nbytes, nt, w.tile_cnt);
    GLOVE_CHECK_LAUNCH();
    size_t tb = w.cub_bytes;
    GLOVE_CHECK_CUDA(cub::DeviceScan::ExclusiveSum(w.cub_temp, tb, w.tile_cnt, w.tile_off, (int)(nt + 1), stream));
    GLOVE_CHECK_CUDA(cudaMemcpyAsync(n_lines_host, w.tile_off + nt, 8, cudaMemcpyDeviceToHost, stream));
    GLOVE_CHECK_CUDA(cudaStreamSynchronize(stream));
    return GLOVE_OK;
}

int glove_vectors_parse(const uint8_t *text, int64_t nbytes, int32_t final_chunk, int32_t d, int64_t n_lines,
                        void *workspace, size_t workspace_bytes, float *out, int64_t ld, int64_t row_capacity,
                        int64_t *word_start, int32_t *word_len, int64_t first_line, int64_t *n_rows_host,
                        int64_t *consumed_host, void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GLOVE_REQUIRE(text && workspace && word_start && word_len && n_rows_host && consumed_host, "glove_vectors_parse: null pointer");
    GLOVE_REQUIRE(out || row_capacity == 0, "glove_vectors_parse: null output");
    GLOVE_REQUIRE(nbytes > 0 && nbytes < (1ll << 31), "glove_vectors_parse: chunk must hold 1 .. 2^31-1 bytes");
    GLOVE_REQUIRE(((uintptr_t)text & 15) == 0, "glove_vectors_parse: text must be 16-byte aligned");
    GLOVE_REQUIRE(d >= 2 && d <= kMaxVecDim, "glove_vectors_parse: d = %d outside [2, %d]", d, kMaxVecDim);
    GLOVE_REQUIRE(ld >= d && row_capacity >= 0 && n_lines >= 0, "glove_vectors_parse: bad sizes");
    const VecWs w = vec_ws_view(workspace, nbytes, n_lines + 1);
    if (workspace_bytes < w.bytes)
        return set_error(GLOVE_EWORKSPACE, "glove_vectors_parse: workspace %zu < required %zu (n_lines %lld)", workspace_bytes,
                         w.bytes, (long long)n_lines);
    const int64_t nt = vec_tiles(nbytes);
    VecStatus st0 = {~0ull, (long long)n_lines, -1};
    GLOVE_CHECK_CUDA(cudaMemcpyAsync(w.status, &st0, sizeof(st0), cudaMemcpyHostToDevice, stream));
    line_ends_kernel<<<(unsigned)nt, kNlThreads, 0, stream>>>(text, nbytes, w.tile_off, w.ends, w.status);
    GLOVE_CHECK_LAUNCH();
    // final chunk: the unterminated last line ends at nbytes (an empty one is a blank line)
    const int64_t lines = n_lines + (final_chunk ? 1 : 0);
    if (final_chunk) GLOVE_CHECK_CUDA(cudaMemcpyAsync(w.ends + n_lines, &nbytes, 8, cudaMemcpyHostToDevice, stream));
    line_flags_kernel<<<(unsigned)((lines + 1 + 255) / 256), 256, 0, stream>>>(text, w.ends, lines, w.flags);
    GLOVE_CHECK_LAUNCH();
    size_t tb = w.cub_bytes;
    GLOVE_CHECK_CUDA(cub::DeviceScan::ExclusiveSum(w.cub_temp, tb, w.flags, w.offs, (int)(lines + 1), stream));
    if (lines)
        parse_lines_kernel<<<(unsigned)((lines + kParseWarps - 1) / kParseWarps), kParseWarps * 32, 0, stream>>>(
            text, nbytes, w.ends, w.flags, w.offs, lines, d, out, ld, row_capacity, word_start, word_len, first_line, w.status);
    GLOVE_CHECK_LAUNCH();
    VecStatus st;
    int64_t rows = 0;
    GLOVE_CHECK_CUDA(cudaMemcpyAsync(&st, w.status, sizeof(st), cudaMemcpyDeviceToHost, stream));
    GLOVE_CHECK_CUDA(cudaMemcpyAsync(&rows, w.offs + lines, 8, cudaMemcpyDeviceToHost, stream));
    GLOVE_CHECK_CUDA(cudaStreamSynchronize(stream));
    if (st.first_error != ~0ull) {
        static const char *what[] = {"", "fewer than d + 1 fields (a word and d numbers)", "not a number",
                                     "more than 19 significant digits and the tail decides the rounding",
                                     "not a finite number", "more vectors than the output holds"};
        const int code = (int)(st.first_error & 0xff);
        return set_error(GLOVE_EINVAL, "vectors file: line %lld: %s", (long long)(st.first_error >> 8),
                         code >= 1 && code <= 5 ? what[code] : "parse error");
    }
    *n_rows_host = rows;
    *consumed_host = final_chunk ? nbytes : st.last_end + 1;
    return GLOVE_OK;
}

int glove_vectors_format_size(const float *rows, int64_t ld, int32_t d, int64_t n, const int64_t *word_off, void *workspace,
                              size_t workspace_bytes, int64_t *text_bytes_host, void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GLOVE_REQUIRE(rows && word_off && workspace && text_bytes_host, "glove_vectors_format_size: null pointer");
    GLOVE_REQUIRE(d >= 2 && d <= kMaxVecDim && ld >= d && n > 0, "glove_vectors_format_size: bad sizes");
    const VecWs w = vec_ws_view(workspace, 1, n);
    if (workspace_bytes < w.bytes)
        return set_error(GLOVE_EWORKSPACE, "glove_vectors_format_size: workspace %zu < required %zu", workspace_bytes, w.bytes);
    format_len_kernel<<<(unsigned)((n + 1 + 3) / 4), 128, 0, stream>>>(rows, ld, d, n, word_off, w.ends);
    GLOVE_CHECK_LAUNCH();
    size_t tb = w.cub_bytes;
    GLOVE_CHECK_CUDA(cub::DeviceScan::ExclusiveSum(w.cub_temp, tb, w.ends, w.offs, (int)(n + 1), stream));
    GLOVE_CHECK_CUDA(cudaMemcpyAsync(text_bytes_host, w.offs + n, 8, cudaMemcpyDeviceToHost, stream));
    GLOVE_CHECK_CUDA(cudaStreamSynchronize(stream));
    return GLOVE_OK;
}

int glove_vectors_format(const float *rows, int64_t ld, int32_t d, int64_t n, const uint8_t *words, const int64_t *word_off,
                         void *workspace, size_t workspace_bytes, uint8_t *text, int64_t capacity, void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GLOVE_REQUIRE(rows && words && word_off && workspace && text, "glove_vectors_format: null pointer");
    GLOVE_REQUIRE(d >= 2 && d <= kMaxVecDim && ld >= d && n > 0 && capacity >= 0, "glove_vectors_format: bad sizes");
    const VecWs w = vec_ws_view(workspace, 1, n);
    if (workspace_bytes < w.bytes)
        return set_error(GLOVE_EWORKSPACE, "glove_vectors_format: workspace %zu < required %zu", workspace_bytes, w.bytes);
    int64_t need = 0;
    GLOVE_CHECK_CUDA(cudaMemcpyAsync(&need, w.offs + n, 8, cudaMemcpyDeviceToHost, stream));
    GLOVE_CHECK_CUDA(cudaStreamSynchronize(stream));
    if (need > capacity)
        return set_error(GLOVE_EINVAL, "glove_vectors_format: %lld bytes of text > capacity %lld", (long long)need, (long long)capacity);
    format_write_kernel<<<(unsigned)((n + 3) / 4), 128, 0, stream>>>(rows, ld, d, n, words, word_off, w.offs, text);
    GLOVE_CHECK_LAUNCH();
    return GLOVE_OK;
}

int glove_format_float32(float value, char *out, int32_t capacity, int32_t *length) {
    GLOVE_REQUIRE(out && length && capacity >= kF32TextMax, "glove_format_float32: out must hold %d bytes", kF32TextMax);
    uint32_t bits;
    memcpy(&bits, &value, 4);
    *length = format_f32(bits, out);
    return GLOVE_OK;
}

}  // extern "C"
