// INGEST: interaction.csv text -> device-resident COO, the wire format of the drop-in (SURVEY §8 f.1).
//
// Replaces tf.data make_csv_dataset(select_columns=[row, col, weight, target]) [ref src/models/data_utils.py:4-26] and the
// per-step StaticHashTable string -> id lookup with default 0 [ref src/models/model_utils.py:121-127,
// src/models/estimator.py:26-28]: the file bytes are parsed ONCE on the GPU, token strings are resolved against
// vocab.txt once, and the result is the (row, col, colA, colB) triple buffer that glove_prepare_batches reads.
//
//   tile_stats_kernel   one pass over the text: per 16 KB tile, the quote-parity flip and the number of record
//                       terminators under both hypotheses (tile starts outside / inside a quoted field)
//   cub InclusiveScan   composes the tile summaries (associative, non-commutative) -> parity and record index at every
//                       tile start
//   row_ends_kernel     second pass: position of the terminating '\n' of every non-empty record
//   parse_rows_kernel   one thread per record: split the fields (RFC-4180 quoting, "" escapes, \r\n), resolve the two
//                       token columns through the device hash table (or parse *_id columns), convert the two value
//                       columns with the correctly rounded decimal -> float32 routine of glove_strtof.cuh
//   vocab_build_kernel  open-addressing table of vocab line numbers keyed by the token bytes (first line wins)
//
// HBM-bound byte work: no tensor cores.  Errors never fall back to the host: the lowest offending record is reported.
#include <cub/cub.cuh>
#include <thrust/iterator/counting_iterator.h>

#include "glove_common.cuh"
#include "glove_strtof.cuh"

namespace glove {

constexpr int kTileThreads = 256, kThreadBytes = 64, kTileBytes = kTileThreads * kThreadBytes;

// summary of a byte range: does it flip the quote parity; records terminated inside it if it starts outside / inside quotes
struct QState { uint32_t flip, n_out, n_in; };
struct QCombine {
    __host__ __device__ __forceinline__ QState operator()(const QState &a, const QState &b) const {
        QState r;
        r.flip = a.flip ^ b.flip;
        r.n_out = a.n_out + (a.flip ? b.n_in : b.n_out);
        r.n_in = a.n_in + (a.flip ? b.n_out : b.n_in);
        return r;
    }
};

enum { CSV_OK = 0, CSV_EFIELDS = 1, CSV_EQUOTE = 2, CSV_EFLOAT = 3, CSV_EDIGITS = 4, CSV_EINT = 5, CSV_ERANGE = 6 };
struct CsvStatus {
    unsigned long long first_error;   // (record << 8) | code, minimum over all records; ~0 = none
    long long n_terms;                // non-empty terminated records of the chunk
    long long tail_valid;             // final chunk: 1 when an unterminated last record exists
    long long last_end;               // position of the last terminator (-1: none)
    long long open_quote;             // parity at the end of the chunk
};

struct CsvWs {
    QState *tile;       // [n_tiles] inclusive scan of the tile summaries
    QState *tile_raw;   // [n_tiles]
    CsvStatus *status;
    void *cub_temp;
    size_t cub_bytes;
    size_t bytes;
};
static int64_t n_tiles_of(int64_t nbytes) { return (nbytes + kTileBytes - 1) / kTileBytes; }
static CsvWs csv_ws_view(void *base, int64_t nbytes) {
    CsvWs w;
    char *p = (char *)base;
    size_t off = 0;
    auto take = [&](size_t bytes) { char *r = p ? p + off : nullptr; off += align_up(bytes); return r; };
    const int64_t nt = n_tiles_of(nbytes) + 1;
    w.status = (CsvStatus *)take(sizeof(CsvStatus));
    w.tile = (QState *)take(sizeof(QState) * nt);
    w.tile_raw = (QState *)take(sizeof(QState) * nt);
    w.cub_bytes = 0;
    cub::DeviceScan::InclusiveScan(nullptr, w.cub_bytes, (QState *)nullptr, (QState *)nullptr, QCombine(), (int)nt);
    w.cub_temp = take(w.cub_bytes);
    w.bytes = off;
    return w;
}

// a '\n' outside quotes at `pos` terminates an EMPTY record when nothing but an optional '\r' lies between it and the
// previous terminator (or the start of the chunk); empty records are skipped like tf.data's CsvDataset does
__device__ __forceinline__ bool empty_record(const uint8_t *text, int64_t pos) {
    if (pos == 0) return true;
    uint8_t p1 = text[pos - 1];
    if (p1 == '\r') {
        if (pos == 1) return true;
        p1 = text[pos - 2];
    }
    return p1 == '\n';
}

// the thread's 64 bytes as 4 x 16 (zero beyond the end: NUL is neither a quote nor a newline)
__device__ __forceinline__ void load_span(const uint8_t *text, int64_t nbytes, int64_t base, uint4 (&v)[4]) {
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        const int64_t o = base + 16 * u;
        if (o + 16 <= nbytes) v[u] = __ldg((const uint4 *)(text + o));
        else {
            uint8_t b[16];
#pragma unroll
            for (int k = 0; k < 16; ++k) b[k] = o + k < nbytes ? text[o + k] : 0;
            v[u] = *(const uint4 *)b;
        }
    }
}
__device__ __forceinline__ uint8_t span_byte(const uint4 (&v)[4], int i) {
    const uint32_t w = ((const uint32_t *)v)[i >> 2];
    return (uint8_t)(w >> (8 * (i & 3)));
}

__global__ void __launch_bounds__(kTileThreads) tile_stats_kernel(const uint8_t *__restrict__ text, int64_t nbytes,
                                                                  QState *tile_raw) {
    const int64_t base = (int64_t)blockIdx.x * kTileBytes + (int64_t)threadIdx.x * kThreadBytes;
    QState s = {0u, 0u, 0u};
    if (base < nbytes) {
        uint4 v[4];
        load_span(text, nbytes, base, v);
        uint32_t par = 0, c[2] = {0u, 0u};
#pragma unroll
        for (int i = 0; i < kThreadBytes; ++i) {
            const uint8_t b = span_byte(v, i);
            if (b == '"') par ^= 1u;
            else if (b == '\n' && !empty_record(text, base + i)) ++c[par];
        }
        s.flip = par; s.n_out = c[0]; s.n_in = c[1];
    }
    typedef cub::BlockScan<QState, kTileThreads> Scan;
    __shared__ typename Scan::TempStorage tmp;
    QState incl;
    Scan(tmp).InclusiveScan(s, incl, QCombine());
    if (threadIdx.x == kTileThreads - 1) tile_raw[blockIdx.x] = incl;
}

__global__ void __launch_bounds__(kTileThreads) row_ends_kernel(const uint8_t *__restrict__ text, int64_t nbytes,
                                                                const QState *__restrict__ tile, int64_t n_tiles,
                                                                int64_t *row_ends, int64_t capacity, CsvStatus *status) {
    const int64_t base = (int64_t)blockIdx.x * kTileBytes + (int64_t)threadIdx.x * kThreadBytes;
    QState s = {0u, 0u, 0u};
    uint4 v[4];
    if (base < nbytes) {
        load_span(text, nbytes, base, v);
        uint32_t par = 0, c[2] = {0u, 0u};
#pragma unroll
        for (int i = 0; i < kThreadBytes; ++i) {
            const uint8_t b = span_byte(v, i);
            if (b == '"') par ^= 1u;
            else if (b == '\n' && !empty_record(text, base + i)) ++c[par];
        }
        s.flip = par; s.n_out = c[0]; s.n_in = c[1];
    }
    typedef cub::BlockScan<QState, kTileThreads> Scan;
    __shared__ typename Scan::TempStorage tmp;
    QState excl;
    const QState ident = {0u, 0u, 0u};
    Scan(tmp).ExclusiveScan(s, excl, ident, QCombine());
    const QState before = blockIdx.x ? QCombine()(tile[blockIdx.x - 1], excl) : excl;   // the chunk starts outside quotes
    if (base >= nbytes) return;
    uint32_t par = before.flip;
    int64_t r = before.n_out;
#pragma unroll
    for (int i = 0; i < kThreadBytes; ++i) {
        const uint8_t b = span_byte(v, i);
        if (b == '"') par ^= 1u;
        else if (b == '\n' && !par && !empty_record(text, base + i)) {
            if (r < capacity) row_ends[r] = base + i;
            ++r;
        }
    }
    if (base + kThreadBytes >= nbytes) status->open_quote = par;
}

__global__ void init_status_kernel(CsvStatus *st, const QState *tile, int64_t n_tiles) {
    st->first_error = ~0ull;
    st->n_terms = n_tiles ? tile[n_tiles - 1].n_out : 0;
    st->tail_valid = 0;
    st->last_end = -1;
    st->open_quote = 0;
}

// ---- vocab hash table ----------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t fnv1a(uint64_t h, uint8_t b) { return (h ^ b) * 0x100000001b3ull; }
constexpr uint64_t kFnvSeed = 0xcbf29ce484222325ull;
__device__ __forceinline__ uint32_t slot_of(uint64_t h, int64_t slots) {
    h ^= h >> 29;
    h *= 0xbf58476d1ce4e5b9ull;
    h ^= h >> 32;
    return (uint32_t)(h & (uint64_t)(slots - 1));
}

// vocab line v = vocab_bytes[vocab_off[v] .. vocab_off[v+1] - 1)   (every line is followed by one '\n')
__global__ void __launch_bounds__(256) vocab_build_kernel(int32_t *table, int64_t slots, const uint8_t *__restrict__ vb,
                                                          const int64_t *__restrict__ voff, int64_t n_vocab) {
    const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n_vocab) return;
    const int64_t b0 = voff[v], len = voff[v + 1] - 1 - b0;
    uint64_t h = kFnvSeed;
    for (int64_t i = 0; i < len; ++i) h = fnv1a(h, vb[b0 + i]);
    uint32_t s = slot_of(h, slots);
    for (;;) {
        const int32_t old = atomicCAS(&table[s], -1, (int32_t)v);
        if (old == -1) return;
        // occupied: the same token (duplicate vocab line) keeps the LOWEST line number; another token -> next slot
        const int64_t o0 = voff[old], olen = voff[old + 1] - 1 - o0;
        bool same = olen == len;
        for (int64_t i = 0; same && i < len; ++i) same = vb[o0 + i] == vb[b0 + i];
        if (same) { atomicMin(&table[s], (int32_t)v); return; }
        s = (s + 1) & (uint32_t)(slots - 1);
    }
}

struct Schema {
    int32_t n_cols;
    int32_t sel[4];    // column index of row, col, colA, colB
    int32_t kind[4];   // GLOVE_CSV_TOKEN / _INT / _FLOAT
};
struct Field { int32_t b, e, esc; };   // content bytes [b, e); esc: contains "" escapes

// the bytes of one record, addressed relative to its first byte (32-bit offsets keep the address arithmetic short)
struct Bytes {
    const uint8_t *p;
    __device__ __forceinline__ uint8_t operator[](int i) const { return __ldg(p + i); }
};

// logical bytes of a field (collapses "" to ")
struct FieldBytes {
    const Bytes &text;
    int i, e;
    bool esc;
    __device__ __forceinline__ bool next(uint8_t &c) {
        if (i >= e) return false;
        c = text[i++];
        if (esc && c == '"') ++i;
        return true;
    }
};

__device__ int32_t lookup_token(const Bytes &text, const Field &f, const int32_t *__restrict__ table,
                                int64_t slots, const uint8_t *__restrict__ vb, const int64_t *__restrict__ voff,
                                int32_t missing = 0) {
    uint64_t h = kFnvSeed;
    int len = 0;
    {
        FieldBytes it = {text, f.b, f.e, f.esc != 0};
        uint8_t c;
        while (it.next(c)) { h = fnv1a(h, c); ++len; }
    }
    uint32_t s = slot_of(h, slots);
    for (;;) {
        const int32_t v = table[s];
        if (v < 0) return missing;                 // StaticHashTable default_value = 0
        const int64_t o0 = voff[v];
        if (voff[v + 1] - 1 - o0 == len) {
            FieldBytes it = {text, f.b, f.e, f.esc != 0};
            uint8_t c;
            int k = 0;
            bool same = true;
            while (same && it.next(c)) same = vb[o0 + k++] == c;
            if (same) return v;
        }
        s = (s + 1) & (uint32_t)(slots - 1);
    }
}

__device__ __forceinline__ void report(CsvStatus *st, int64_t record, int code) {
    atomicMin(&st->first_error, ((unsigned long long)record << 8) | (unsigned)code);
}

__global__ void __launch_bounds__(128) parse_rows_kernel(const uint8_t *__restrict__ text_bytes, int64_t nbytes, int32_t final_chunk,
                                                         const int64_t *__restrict__ row_ends, CsvStatus *st, Schema sc,
                                                         const int32_t *__restrict__ table, int64_t slots,
                                                         const uint8_t *__restrict__ vb, const int64_t *__restrict__ voff,
                                                         int64_t n_vocab, int32_t *out_row, int32_t *out_col, float *out_a,
                                                         float *out_b, int64_t capacity, int64_t record0) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t n_terms = st->n_terms;
    if (r > n_terms || r >= capacity || (r == n_terms && !final_chunk)) return;
    int64_t pos0 = r ? row_ends[r - 1] + 1 : 0;
    int64_t end0 = r < n_terms ? row_ends[r] : nbytes;
    if (r == n_terms - 1) st->last_end = end0;
    // skipped empty records in front of this one
    while (pos0 < end0 && (text_bytes[pos0] == '\n' || (text_bytes[pos0] == '\r' && pos0 + 1 < end0 && text_bytes[pos0 + 1] == '\n')))
        ++pos0;
    if (end0 > pos0 && text_bytes[end0 - 1] == '\r') --end0;
    if (r == n_terms) {              // unterminated last record of the file
        if (pos0 >= end0) return;
        if (st->open_quote) { report(st, record0 + r, CSV_EQUOTE); return; }
        st->tail_valid = 1;
    }
    if (end0 - pos0 > 0x3fffffff) { report(st, record0 + r, CSV_EFIELDS); return; }
    const Bytes text = {text_bytes + pos0};
    int pos = 0;
    const int end = (int)(end0 - pos0);
    Field sel[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) sel[c] = Field{0, 0, 0};
    int32_t field = 0;
    bool bad_quote = false;
    for (;;) {
        Field f;
        f.esc = 0;
        if (pos < end && text[pos] == '"') {
            f.b = ++pos;
            for (;;) {
                if (pos >= end) { bad_quote = true; break; }
                if (text[pos] == '"') {
                    if (pos + 1 < end && text[pos + 1] == '"') { pos += 2; f.esc = 1; continue; }
                    break;
                }
                ++pos;
            }
            f.e = pos;
            if (!bad_quote) {
                ++pos;
                if (pos < end && text[pos] != ',') bad_quote = true;
            }
        } else {
            f.b = pos;
            while (pos < end && text[pos] != ',') ++pos;
            f.e = pos;
        }
        if (bad_quote) break;
#pragma unroll
        for (int c = 0; c < 4; ++c)
            if (sc.sel[c] == field) sel[c] = f;
        ++field;
        if (pos >= end) break;
        ++pos;   // the comma
    }
    if (bad_quote) { report(st, record0 + r, CSV_EQUOTE); return; }
    if (field != sc.n_cols) { report(st, record0 + r, CSV_EFIELDS); return; }
    int32_t ids[2];
    float vals[2];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        const Field f = sel[c];
        if (sc.kind[c] == GLOVE_CSV_TOKEN) {
            ids[c & 1] = lookup_token(text, f, table, slots, vb, voff);
        } else if (sc.kind[c] == GLOVE_CSV_INT) {
            int i = f.b;
            int64_t v = 0;
            bool neg = false, ok = f.e > f.b && !f.esc;
            if (ok && (text[i] == '-' || text[i] == '+')) { neg = text[i] == '-'; ++i; ok = i < f.e; }
            for (; ok && i < f.e; ++i) {
                const unsigned dgt = (unsigned)(text[i] - '0');
                ok = dgt <= 9 && v < (1ll << 40);
                v = v * 10 + dgt;
            }
            if (!ok) { report(st, record0 + r, CSV_EINT); return; }
            if (neg) v = -v;
            if (v < 0 || v >= n_vocab) { report(st, record0 + r, CSV_ERANGE); return; }
            ids[c & 1] = (int32_t)v;
        } else {
            uint32_t bits;
            const Bytes fb = {text.p + f.b};
            const int rc = f.esc ? (int)STRTOF_BAD : parse_f32([fb](int i) { return (int)fb[i]; }, f.e - f.b, bits);
            if (rc != STRTOF_OK) { report(st, record0 + r, rc == STRTOF_TOO_LONG ? CSV_EDIGITS : CSV_EFLOAT); return; }
            vals[c & 1] = __uint_as_float(bits);
        }
    }
    out_row[r] = ids[0];
    out_col[r] = ids[1];
    out_a[r] = vals[0];
    out_b[r] = vals[1];
}


// ---- corpus text -> token stream (front half of the preprocessor, SURVEY §8 f.4) -------------------------------------
// str.split() of the reference [ref src/data/text8.py:47]: tokens are maximal runs of non-whitespace.  ASCII whitespace
// only (space, \t \n \v \f \r, 0x1c-0x1f); the UTF-8 encodings of the other Unicode separators str.split() knows are
// detected and refused, never mis-split.
__device__ __forceinline__ bool is_space(uint8_t b) { return b == 0x20 || (b >= 0x09 && b <= 0x0d) || (b >= 0x1c && b <= 0x1f); }
__device__ __forceinline__ bool unicode_space_at(const uint8_t *t, int64_t i, int64_t n) {
    const uint8_t b = t[i];
    if (b == 0xc2) return i + 1 < n && (t[i + 1] == 0x85 || t[i + 1] == 0xa0);
    if (i + 2 >= n) return false;
    const uint8_t c = t[i + 1], d = t[i + 2];
    if (b == 0xe1) return c == 0x9a && d == 0x80;
    if (b == 0xe2) return (c == 0x80 && ((d >= 0x80 && d <= 0x8a) || d == 0xa8 || d == 0xa9 || d == 0xaf)) || (c == 0x81 && d == 0x9f);
    if (b == 0xe3) return c == 0x80 && d == 0x80;
    return false;
}
__global__ void __launch_bounds__(256) token_flags_kernel(const uint8_t *__restrict__ text, int64_t nbytes, uint8_t *flags,
                                                          int32_t *bad) {
    const int64_t i0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 16;
    if (i0 >= nbytes) return;
    uint8_t b[17];
    b[0] = i0 ? text[i0 - 1] : (uint8_t)' ';
#pragma unroll
    for (int k = 0; k < 16; ++k) b[k + 1] = i0 + k < nbytes ? text[i0 + k] : (uint8_t)' ';
    uint8_t f[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        f[k] = (i0 + k < nbytes) && !is_space(b[k + 1]) && is_space(b[k]);
        if (b[k + 1] >= 0xc2 && i0 + k < nbytes && unicode_space_at(text, i0 + k, nbytes)) *bad = 1;
    }
    if (i0 + 16 <= nbytes) *(uint4 *)(flags + i0) = *(const uint4 *)f;
    else
        for (int k = 0; i0 + k < nbytes; ++k) flags[i0 + k] = f[k];
}
// length and 64-bit hash of the token that starts at starts[i]
__global__ void __launch_bounds__(256) token_hash_kernel(const uint8_t *__restrict__ text, int64_t nbytes,
                                                         const int64_t *__restrict__ starts, int64_t n, int32_t *lens,
                                                         uint64_t *hash, uint32_t *idx) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t s = starts[i];
    uint64_t h = kFnvSeed;
    int64_t e = s;
    while (e < nbytes && !is_space(text[e])) h = fnv1a(h, text[e++]);
    lens[i] = (int32_t)(e - s);
    if (hash) {
        h ^= h >> 29; h *= 0xbf58476d1ce4e5b9ull; h ^= h >> 32;
        hash[i] = h;
        idx[i] = (uint32_t)i;
    }
}
// equal hashes must be equal tokens (adjacent elements of the sorted order are compared: equality is transitive)
__global__ void __launch_bounds__(256) token_verify_kernel(const uint8_t *__restrict__ text, const int64_t *__restrict__ starts,
                                                           const int32_t *__restrict__ lens, const uint64_t *__restrict__ hash,
                                                           const uint32_t *__restrict__ idx, int64_t n, int32_t *bad) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < 1 || i >= n || hash[i] != hash[i - 1]) return;
    const uint32_t a = idx[i], b = idx[i - 1];
    bool same = lens[a] == lens[b];
    for (int k = 0; same && k < lens[a]; ++k) same = text[starts[a] + k] == text[starts[b] + k];
    if (!same) *bad = 1;
}
__global__ void __launch_bounds__(256) token_runs_kernel(const uint32_t *__restrict__ idx, const int64_t *__restrict__ starts,
                                                         const int32_t *__restrict__ lens, const int32_t *__restrict__ run_len,
                                                         const int32_t *__restrict__ run_off, int64_t n_runs,
                                                         int64_t *first_start, int32_t *first_len, int64_t *count) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_runs) return;
    const uint32_t head = idx[run_off[r]];      // stable sort: the first element of a run is the first occurrence
    first_start[r] = starts[head];
    first_len[r] = lens[head];
    count[r] = run_len[r];
}
template <int32_t kMissing>
__global__ void __launch_bounds__(256) token_lookup_kernel(const uint8_t *__restrict__ text, const int64_t *__restrict__ starts,
                                                           const int32_t *__restrict__ lens, int64_t n,
                                                           const int32_t *__restrict__ table, int64_t slots,
                                                           const uint8_t *__restrict__ vb, const int64_t *__restrict__ voff,
                                                           int32_t *ids) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const Bytes t = {text + starts[i]};
    const Field f = {0, lens[i], 0};
    ids[i] = lookup_token(t, f, table, slots, vb, voff, kMissing);
}

// ---- Stanford GloVe's token stream (vocab_count / cooccur semantics, corpus.py scheme "stanford") ----------------------
// Bytes that Stanford's get_word glues into tokens (it splits on ' ', '\t', '\n' only and drops every '\r') but that this
// project's vocabulary readers would split: \v, \f, 0x1c-0x1f, and a \r that is not directly before a \n.  With these
// refused, the token boundaries of Stanford's tokenizer are those of glove_tokens_scan.  next_byte: the byte after the
// chunk (-1 at the end of the file).  The lowest offending offset wins.
__device__ __forceinline__ bool refused_byte(uint8_t b, int32_t next) {
    return b == 0x0b || b == 0x0c || (b >= 0x1c && b <= 0x1f) || (b == 0x0d && next != 0x0a);
}
__global__ void __launch_bounds__(256) text_refused_kernel(const uint8_t *__restrict__ text, int64_t nbytes, int32_t next_byte,
                                                           unsigned long long *first) {
    const int64_t i0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 16;
    if (i0 >= nbytes) return;
    alignas(16) uint8_t b[16];
    if (i0 + 16 <= nbytes) *(uint4 *)b = __ldg((const uint4 *)(text + i0));
    else
        for (int k = 0; k < 16; ++k) b[k] = i0 + k < nbytes ? text[i0 + k] : (uint8_t)' ';
    const int32_t after = i0 + 16 < nbytes ? (int32_t)text[i0 + 16] : i0 + 16 == nbytes ? next_byte : -1;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        if (refused_byte(b[k], k < 15 ? (int32_t)b[k + 1] : after)) {
            atomicMin(first, (unsigned long long)(i0 + k));
            return;
        }
    }
}
// brk[i] = 1 when a '\n' lies between token i - 1 and token i (token 0: between text_begin and its start, or
// newline_before, a '\n' after the last token of the previous chunk)
__global__ void __launch_bounds__(256) token_breaks_kernel(const uint8_t *__restrict__ text, int64_t text_begin,
                                                           const int64_t *__restrict__ starts, const int32_t *__restrict__ lens,
                                                           int64_t n, int32_t newline_before, uint32_t *brk) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t lo = i ? starts[i - 1] + lens[i - 1] : text_begin;
    bool nl = i == 0 && newline_before;
    for (int64_t e = starts[i] - 1; !nl && e >= lo; --e) nl = text[e] == '\n';
    brk[i] = nl;
}
// in-vocabulary tokens as (segment << 32) | id, segment = segment_base + number of line breaks up to the token
__global__ void __launch_bounds__(256) token_pack_kernel(const int32_t *__restrict__ ids, const uint32_t *__restrict__ seg,
                                                         int64_t n, uint32_t segment_base, uint64_t *packed, uint8_t *keep) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    packed[i] = ((uint64_t)(segment_base + seg[i]) << 32) | (uint32_t)ids[i];
    keep[i] = ids[i] >= 0;
}

struct TokWs {
    uint8_t *flags;
    uint64_t *hash[2];
    uint32_t *idx[2];
    int32_t *run_len, *run_off;
    long long *n_out;
    int32_t *bad;
    void *cub_temp;
    size_t cub_bytes, bytes;
};
static TokWs tok_ws_view(void *base, int64_t nbytes, int64_t n_tokens) {
    TokWs w;
    char *p = (char *)base;
    size_t off = 0;
    auto take = [&](size_t bytes) { char *r = p ? p + off : nullptr; off += align_up(bytes); return r; };
    const int64_t n = n_tokens < 1 ? 1 : n_tokens;
    w.flags = (uint8_t *)take(nbytes + 16);
    for (int i = 0; i < 2; ++i) w.hash[i] = (uint64_t *)take(8 * n);
    for (int i = 0; i < 2; ++i) w.idx[i] = (uint32_t *)take(4 * n);
    w.run_len = (int32_t *)take(4 * n);
    w.run_off = (int32_t *)take(4 * n);
    w.n_out = (long long *)take(8);
    w.bad = (int32_t *)take(4);
    size_t a = 0, b = 0, c = 0, d = 0, e = 0;
    cub::DeviceReduce::Sum(nullptr, e, (uint8_t *)nullptr, (long long *)nullptr, (int)(nbytes < 1 ? 1 : nbytes));
    cub::DeviceSelect::Flagged(nullptr, a, thrust::counting_iterator<int64_t>(0), (uint8_t *)nullptr, (int64_t *)nullptr,
                               (long long *)nullptr, (int)(nbytes < 1 ? 1 : nbytes));
    cub::DeviceRadixSort::SortPairs(nullptr, b, (uint64_t *)nullptr, (uint64_t *)nullptr, (uint32_t *)nullptr, (uint32_t *)nullptr, (int)n);
    cub::DeviceRunLengthEncode::Encode(nullptr, c, (uint64_t *)nullptr, (uint64_t *)nullptr, (int32_t *)nullptr, (long long *)nullptr, (int)n);
    cub::DeviceScan::ExclusiveSum(nullptr, d, (int32_t *)nullptr, (int32_t *)nullptr, (int)n);
    w.cub_bytes = a > b ? a : b;
    if (c > w.cub_bytes) w.cub_bytes = c;
    if (d > w.cub_bytes) w.cub_bytes = d;
    if (e > w.cub_bytes) w.cub_bytes = e;
    w.cub_temp = take(w.cub_bytes);
    w.bytes = off;
    return w;
}

struct StreamWs {
    int32_t *ids;
    uint32_t *brk, *seg;
    uint64_t *packed;
    uint8_t *keep;
    long long *n_out;
    void *cub_temp;
    size_t cub_bytes, bytes;
};
static StreamWs stream_ws_view(void *base, int64_t n) {
    StreamWs w;
    char *p = (char *)base;
    size_t off = 0;
    auto take = [&](size_t bytes) { char *r = p ? p + off : nullptr; off += align_up(bytes); return r; };
    w.ids = (int32_t *)take(4 * n);
    w.brk = (uint32_t *)take(4 * n);
    w.seg = (uint32_t *)take(4 * n);
    w.packed = (uint64_t *)take(8 * n);
    w.keep = (uint8_t *)take(n);
    w.n_out = (long long *)take(8);
    size_t a = 0, b = 0;
    cub::DeviceScan::InclusiveSum(nullptr, a, (uint32_t *)nullptr, (uint32_t *)nullptr, (int)n);
    cub::DeviceSelect::Flagged(nullptr, b, (uint64_t *)nullptr, (uint8_t *)nullptr, (uint64_t *)nullptr, (long long *)nullptr,
                               (int)n);
    w.cub_bytes = a > b ? a : b;
    w.cub_temp = take(w.cub_bytes);
    w.bytes = off;
    return w;
}

}  // namespace glove

using namespace glove;

extern "C" {

int64_t glove_vocab_slots(int64_t n_vocab) {
    int64_t s = 1024;
    while (s < 2 * n_vocab) s <<= 1;
    return s;
}

int glove_vocab_build(int32_t *table, int64_t slots, const uint8_t *vocab_bytes, const int64_t *vocab_off,
                      int64_t n_vocab, void *stream) {
    GLOVE_REQUIRE(table && vocab_bytes && vocab_off && n_vocab > 0, "glove_vocab_build: bad arguments");
    GLOVE_REQUIRE(slots >= 2 * n_vocab && (slots & (slots - 1)) == 0 && n_vocab < (1ll << 31),
                  "glove_vocab_build: slots must be a power of two >= 2 * n_vocab");
    GLOVE_CHECK_CUDA(cudaMemsetAsync(table, 0xff, sizeof(int32_t) * slots, (cudaStream_t)stream));
    vocab_build_kernel<<<(unsigned)((n_vocab + 255) / 256), 256, 0, (cudaStream_t)stream>>>(table, slots, vocab_bytes,
                                                                                            vocab_off, n_vocab);
    GLOVE_CHECK_LAUNCH();
    return GLOVE_OK;
}

size_t glove_csv_workspace_bytes(int64_t nbytes) { return csv_ws_view(nullptr, nbytes < 1 ? 1 : nbytes).bytes; }

int glove_csv_index(const uint8_t *text, int64_t nbytes, void *workspace, size_t workspace_bytes, int64_t *n_records_host,
                    void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GLOVE_REQUIRE(text && workspace && n_records_host && nbytes > 0, "glove_csv_index: bad arguments");
    GLOVE_REQUIRE(((uintptr_t)text & 15) == 0, "glove_csv_index: text must be 16-byte aligned");
    GLOVE_REQUIRE(nbytes < (1ll << 40), "glove_csv_index: chunk too large");
    const CsvWs w = csv_ws_view(workspace, nbytes);
    if (workspace_bytes < w.bytes)
        return set_error(GLOVE_EWORKSPACE, "glove_csv_index: workspace %zu < required %zu", workspace_bytes, w.bytes);
    const int64_t nt = n_tiles_of(nbytes);
    tile_stats_kernel<<<(unsigned)nt, kTileThreads, 0, stream>>>(text, nbytes, w.tile_raw);
    GLOVE_CHECK_LAUNCH();
    size_t tb = w.cub_bytes;
    GLOVE_CHECK_CUDA(cub::DeviceScan::InclusiveScan(w.cub_temp, tb, w.tile_raw, w.tile, QCombine(), (int)nt, stream));
    init_status_kernel<<<1, 1, 0, stream>>>(w.status, w.tile, nt);
    GLOVE_CHECK_LAUNCH();
    CsvStatus st;
    GLOVE_CHECK_CUDA(cudaMemcpyAsync(&st, w.status, sizeof(st), cudaMemcpyDeviceToHost, stream));
    GLOVE_CHECK_CUDA(cudaStreamSynchronize(stream));
    *n_records_host = st.n_terms;
    return GLOVE_OK;
}

int glove_csv_parse(const uint8_t *text, int64_t nbytes, int32_t final_chunk, void *workspace, size_t workspace_bytes,
                    const glove_csv_schema *schema, const int32_t *vocab_table, int64_t vocab_slots,
                    const uint8_t *vocab_bytes, const int64_t *vocab_off, int64_t n_vocab, int64_t *row_ends,
                    int32_t *row, int32_t *col, float *colA, float *colB, int64_t capacity, int64_t first_record,
                    int64_t *n_rows_host, int64_t *consumed_host, void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GLOVE_REQUIRE(text && workspace && schema && row_ends && row && col && colA && colB && n_rows_host && consumed_host,
                  "glove_csv_parse: null pointer");
    GLOVE_REQUIRE(nbytes > 0 && capacity > 0 && n_vocab > 0, "glove_csv_parse: bad sizes");
    Schema sc;
    sc.n_cols = schema->n_cols;
    bool need_vocab = false;
    for (int c = 0; c < 4; ++c) {
        sc.sel[c] = schema->column[c];
        sc.kind[c] = schema->kind[c];
        GLOVE_REQUIRE(sc.sel[c] >= 0 && sc.sel[c] < sc.n_cols, "glove_csv_parse: selected column %d out of range", sc.sel[c]);
        if (c < 2) GLOVE_REQUIRE(sc.kind[c] == GLOVE_CSV_TOKEN || sc.kind[c] == GLOVE_CSV_INT, "glove_csv_parse: id column kind");
        else GLOVE_REQUIRE(sc.kind[c] == GLOVE_CSV_FLOAT, "glove_csv_parse: value column kind");
        need_vocab |= sc.kind[c] == GLOVE_CSV_TOKEN;
    }
    if (need_vocab) GLOVE_REQUIRE(vocab_table && vocab_bytes && vocab_off && vocab_slots > 0, "glove_csv_parse: vocab table missing");
    const CsvWs w = csv_ws_view(workspace, nbytes);
    if (workspace_bytes < w.bytes)
        return set_error(GLOVE_EWORKSPACE, "glove_csv_parse: workspace %zu < required %zu", workspace_bytes, w.bytes);
    const int64_t nt = n_tiles_of(nbytes);
    row_ends_kernel<<<(unsigned)nt, kTileThreads, 0, stream>>>(text, nbytes, w.tile, nt, row_ends, capacity, w.status);
    GLOVE_CHECK_LAUNCH();
    parse_rows_kernel<<<(unsigned)((capacity + 127) / 128), 128, 0, stream>>>(
        text, nbytes, final_chunk, row_ends, w.status, sc, vocab_table, vocab_slots, vocab_bytes, vocab_off, n_vocab, row,
        col, colA, colB, capacity, first_record);
    GLOVE_CHECK_LAUNCH();
    CsvStatus st;
    GLOVE_CHECK_CUDA(cudaMemcpyAsync(&st, w.status, sizeof(st), cudaMemcpyDeviceToHost, stream));
    GLOVE_CHECK_CUDA(cudaStreamSynchronize(stream));
    if (st.n_terms + (final_chunk ? 1 : 0) > capacity)
        return set_error(GLOVE_EINVAL, "glove_csv_parse: capacity %lld < %lld records (+1 for a final chunk)",
                         (long long)capacity, (long long)st.n_terms);
    if (st.first_error != ~0ull) {
        static const char *what[] = {"", "wrong number of fields", "malformed quoting", "not a number",
                                     "more than 19 significant digits and the tail decides the rounding", "not an integer id",
                                     "id outside [0, vocab size)"};
        const int code = (int)(st.first_error & 0xff);
        return set_error(GLOVE_EINVAL, "interaction csv: record %lld: %s", (long long)(st.first_error >> 8),
                         code >= 1 && code <= 6 ? what[code] : "parse error");
    }
    if (final_chunk && st.open_quote)
        return set_error(GLOVE_EINVAL, "interaction csv: unterminated quoted field at end of file");
    *n_rows_host = st.n_terms + st.tail_valid;
    *consumed_host = final_chunk ? nbytes : st.last_end + 1;
    return GLOVE_OK;
}

size_t glove_tokens_workspace_bytes(int64_t nbytes, int64_t n_tokens) {
    return tok_ws_view(nullptr, nbytes < 1 ? 1 : nbytes, n_tokens).bytes;
}

int glove_tokens_scan(const uint8_t *text, int64_t nbytes, void *workspace, size_t workspace_bytes, int64_t *starts,
                      int32_t *lens, int64_t capacity, int64_t *n_tokens_host, void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GLOVE_REQUIRE(text && workspace && starts && lens && n_tokens_host, "glove_tokens_scan: null pointer");
    GLOVE_REQUIRE(nbytes > 0 && nbytes < (1ll << 31), "glove_tokens_scan: chunk must hold 1 .. 2^31-1 bytes");
    const TokWs w = tok_ws_view(workspace, nbytes, 0);
    if (workspace_bytes < w.bytes)
        return set_error(GLOVE_EWORKSPACE, "glove_tokens_scan: workspace %zu < required %zu", workspace_bytes, w.bytes);
    GLOVE_CHECK_CUDA(cudaMemsetAsync(w.bad, 0, 4, stream));
    token_flags_kernel<<<(unsigned)((nbytes + 4095) / 4096), 256, 0, stream>>>(text, nbytes, w.flags, w.bad);
    GLOVE_CHECK_LAUNCH();
    size_t tb = w.cub_bytes;
    // capacity is checked after the count is known: select into the caller's buffer only if it fits
    long long n = 0;
    {
        // first pass: count (sum of the flags) -- cheap, and it lets us refuse before writing past `capacity`
        size_t rb = w.cub_bytes;
        GLOVE_CHECK_CUDA(cub::DeviceReduce::Sum(w.cub_temp, rb, w.flags, w.n_out, (int)nbytes, stream));
        int32_t bad = 0;
        GLOVE_CHECK_CUDA(cudaMemcpyAsync(&bad, w.bad, 4, cudaMemcpyDeviceToHost, stream));
        GLOVE_CHECK_CUDA(cudaMemcpyAsync(&n, w.n_out, 8, cudaMemcpyDeviceToHost, stream));
        GLOVE_CHECK_CUDA(cudaStreamSynchronize(stream));
        if (bad) return set_error(GLOVE_EUNSUPPORTED, "corpus holds non-ASCII Unicode whitespace, which str.split() would split on");
    }
    *n_tokens_host = n;
    if (n > capacity) return set_error(GLOVE_EINVAL, "glove_tokens_scan: %lld tokens > capacity %lld", n, (long long)capacity);
    if (n == 0) return GLOVE_OK;
    GLOVE_CHECK_CUDA(cub::DeviceSelect::Flagged(w.cub_temp, tb, thrust::counting_iterator<int64_t>(0), w.flags, starts, w.n_out,
                                                (int)nbytes, stream));
    token_hash_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(text, nbytes, starts, n, lens, nullptr, nullptr);
    GLOVE_CHECK_LAUNCH();
    GLOVE_CHECK_CUDA(cudaStreamSynchronize(stream));
    return GLOVE_OK;
}

int glove_tokens_count(const uint8_t *text, int64_t nbytes, const int64_t *starts, int64_t n_tokens, void *workspace,
                       size_t workspace_bytes, int64_t *first_start, int32_t *first_len, int64_t *count, int64_t capacity,
                       int64_t *n_distinct_host, void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GLOVE_REQUIRE(text && starts && workspace && first_start && first_len && count && n_distinct_host,
                  "glove_tokens_count: null pointer");
    GLOVE_REQUIRE(n_tokens > 0 && n_tokens < (1ll << 31) && nbytes > 0, "glove_tokens_count: bad sizes");
    const TokWs w = tok_ws_view(workspace, nbytes, n_tokens);
    if (workspace_bytes < w.bytes)
        return set_error(GLOVE_EWORKSPACE, "glove_tokens_count: workspace %zu < required %zu", workspace_bytes, w.bytes);
    const unsigned g = (unsigned)((n_tokens + 255) / 256);
    int32_t *lens = w.run_off;   // token lengths live here until the run offsets are needed
    GLOVE_CHECK_CUDA(cudaMemsetAsync(w.bad, 0, 4, stream));
    token_hash_kernel<<<g, 256, 0, stream>>>(text, nbytes, starts, n_tokens, lens, w.hash[0], w.idx[0]);
    GLOVE_CHECK_LAUNCH();
    size_t tb = w.cub_bytes;
    GLOVE_CHECK_CUDA(cub::DeviceRadixSort::SortPairs(w.cub_temp, tb, w.hash[0], w.hash[1], w.idx[0], w.idx[1], (int)n_tokens, 0, 64,
                                                     stream));
    token_verify_kernel<<<g, 256, 0, stream>>>(text, starts, lens, w.hash[1], w.idx[1], n_tokens, w.bad);
    GLOVE_CHECK_LAUNCH();
    tb = w.cub_bytes;
    GLOVE_CHECK_CUDA(cub::DeviceRunLengthEncode::Encode(w.cub_temp, tb, w.hash[1], w.hash[0], w.run_len, w.n_out, (int)n_tokens,
                                                        stream));
    long long runs = 0;
    int32_t bad = 0;
    GLOVE_CHECK_CUDA(cudaMemcpyAsync(&bad, w.bad, 4, cudaMemcpyDeviceToHost, stream));
    GLOVE_CHECK_CUDA(cudaMemcpyAsync(&runs, w.n_out, 8, cudaMemcpyDeviceToHost, stream));
    GLOVE_CHECK_CUDA(cudaStreamSynchronize(stream));
    if (bad) return set_error(GLOVE_EUNSUPPORTED, "glove_tokens_count: two different tokens share a 64-bit hash");
    *n_distinct_host = runs;
    if (runs > capacity)
        return set_error(GLOVE_EINVAL, "glove_tokens_count: %lld distinct tokens > capacity %lld", runs, (long long)capacity);
    // first occurrence of every run: the lengths move to idx[0] (free now) so that run_off can hold the offsets
    int32_t *lens2 = (int32_t *)w.idx[0];
    GLOVE_CHECK_CUDA(cudaMemcpyAsync(lens2, lens, 4 * n_tokens, cudaMemcpyDeviceToDevice, stream));
    tb = w.cub_bytes;
    GLOVE_CHECK_CUDA(cub::DeviceScan::ExclusiveSum(w.cub_temp, tb, w.run_len, w.run_off, (int)runs, stream));
    token_runs_kernel<<<(unsigned)((runs + 255) / 256), 256, 0, stream>>>(w.idx[1], starts, lens2, w.run_len, w.run_off, runs,
                                                                           first_start, first_len, count);
    GLOVE_CHECK_LAUNCH();
    GLOVE_CHECK_CUDA(cudaStreamSynchronize(stream));
    return GLOVE_OK;
}

int glove_tokens_lookup(const uint8_t *text, const int64_t *starts, const int32_t *lens, int64_t n_tokens,
                        const int32_t *vocab_table, int64_t vocab_slots, const uint8_t *vocab_bytes, const int64_t *vocab_off,
                        int32_t *ids, void *stream) {
    GLOVE_REQUIRE(text && starts && lens && vocab_table && vocab_bytes && vocab_off && ids && n_tokens > 0 && vocab_slots > 0,
                  "glove_tokens_lookup: bad arguments");
    token_lookup_kernel<0><<<(unsigned)((n_tokens + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        text, starts, lens, n_tokens, vocab_table, vocab_slots, vocab_bytes, vocab_off, ids);
    GLOVE_CHECK_LAUNCH();
    return GLOVE_OK;
}

int glove_text_refused(const uint8_t *text, int64_t nbytes, int32_t next_byte, uint64_t *scratch, int64_t *first_host,
                       void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GLOVE_REQUIRE(text && scratch && first_host, "glove_text_refused: null pointer");
    GLOVE_REQUIRE(nbytes > 0 && nbytes < (1ll << 40) && next_byte >= -1 && next_byte <= 255, "glove_text_refused: bad sizes");
    GLOVE_REQUIRE(((uintptr_t)text & 15) == 0, "glove_text_refused: text must be 16-byte aligned");
    GLOVE_CHECK_CUDA(cudaMemsetAsync(scratch, 0xff, 8, stream));
    const int64_t threads = (nbytes + 15) / 16;
    text_refused_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, stream>>>(text, nbytes, next_byte,
                                                                              (unsigned long long *)scratch);
    GLOVE_CHECK_LAUNCH();
    uint64_t first = 0;
    GLOVE_CHECK_CUDA(cudaMemcpyAsync(&first, scratch, 8, cudaMemcpyDeviceToHost, stream));
    GLOVE_CHECK_CUDA(cudaStreamSynchronize(stream));
    *first_host = first == ~0ull ? -1 : (int64_t)first;
    return GLOVE_OK;
}

size_t glove_tokens_stream_workspace_bytes(int64_t n_tokens) { return stream_ws_view(nullptr, n_tokens < 1 ? 1 : n_tokens).bytes; }

int glove_tokens_stream(const uint8_t *text, int64_t text_begin, const int64_t *starts, const int32_t *lens, int64_t n_tokens,
                        int32_t newline_before, uint32_t segment_base, const int32_t *vocab_table, int64_t vocab_slots,
                        const uint8_t *vocab_bytes, const int64_t *vocab_off, void *workspace, size_t workspace_bytes,
                        uint64_t *out, int64_t capacity, int64_t *n_out_host, uint32_t *last_segment_host, void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GLOVE_REQUIRE(text && starts && lens && vocab_table && vocab_bytes && vocab_off && workspace && out && n_out_host &&
                      last_segment_host,
                  "glove_tokens_stream: null pointer");
    GLOVE_REQUIRE(n_tokens > 0 && n_tokens < (1ll << 31) && text_begin >= 0 && vocab_slots > 0,
                  "glove_tokens_stream: bad sizes");
    GLOVE_REQUIRE(capacity >= n_tokens, "glove_tokens_stream: capacity %lld < n_tokens %lld", (long long)capacity,
                  (long long)n_tokens);
    const StreamWs w = stream_ws_view(workspace, n_tokens);
    if (workspace_bytes < w.bytes)
        return set_error(GLOVE_EWORKSPACE, "glove_tokens_stream: workspace %zu < required %zu", workspace_bytes, w.bytes);
    const unsigned g = (unsigned)((n_tokens + 255) / 256);
    token_lookup_kernel<-1><<<g, 256, 0, stream>>>(text, starts, lens, n_tokens, vocab_table, vocab_slots, vocab_bytes, vocab_off,
                                                   w.ids);
    GLOVE_CHECK_LAUNCH();
    token_breaks_kernel<<<g, 256, 0, stream>>>(text, text_begin, starts, lens, n_tokens, newline_before, w.brk);
    GLOVE_CHECK_LAUNCH();
    size_t tb = w.cub_bytes;
    GLOVE_CHECK_CUDA(cub::DeviceScan::InclusiveSum(w.cub_temp, tb, w.brk, w.seg, (int)n_tokens, stream));
    token_pack_kernel<<<g, 256, 0, stream>>>(w.ids, w.seg, n_tokens, segment_base, w.packed, w.keep);
    GLOVE_CHECK_LAUNCH();
    tb = w.cub_bytes;
    GLOVE_CHECK_CUDA(cub::DeviceSelect::Flagged(w.cub_temp, tb, w.packed, w.keep, out, w.n_out, (int)n_tokens, stream));
    long long n = 0;
    uint32_t last = 0;
    GLOVE_CHECK_CUDA(cudaMemcpyAsync(&n, w.n_out, 8, cudaMemcpyDeviceToHost, stream));
    GLOVE_CHECK_CUDA(cudaMemcpyAsync(&last, w.seg + n_tokens - 1, 4, cudaMemcpyDeviceToHost, stream));
    GLOVE_CHECK_CUDA(cudaStreamSynchronize(stream));
    *n_out_host = n;
    *last_segment_host = segment_base + last;
    return GLOVE_OK;
}

// host-side entry to the SAME decimal -> float32 routine the kernels use (CPU tests check it against exact rounding)
int glove_parse_float32(const char *text, int32_t n, float *out) {
    GLOVE_REQUIRE(text && out && n >= 0, "glove_parse_float32: bad arguments");
    uint32_t bits;
    const int rc = parse_f32([text](int i) { return (int)(uint8_t)text[i]; }, n, bits);
    if (rc != STRTOF_OK) return set_error(GLOVE_EINVAL, "glove_parse_float32: %s", rc == STRTOF_TOO_LONG ? "too many digits" : "not a number");
    memcpy(out, &bits, 4);
    return GLOVE_OK;
}

}  // extern "C"
