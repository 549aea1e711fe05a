// Stanford GloVe co-occurrence records (cooccurrence.bin / cooccurrence.shuf.bin of cooccur.c and shuffle.c, default
// build with real = double): struct { int32 word1; int32 word2; float64 val; }, little-endian, 16 bytes, no header.
// Ids are 1-based vocabulary line numbers.
//
//   bin_parse    one chunk of records -> the engine's COO columns: row = word1 - 1, col = word2 - 1,
//                target = (float)log(val), weight = (float)(val >= x_max ? 1 : pow(val / x_max, alpha)), both in float64
//                and rounded once (glove.c's objective with the weight taken from X).  An id outside 1..V or a val that
//                is not finite and > 0 is recorded in one device word by atomicMin(record * 4 + kind): the lowest bad
//                record of the chunk wins and its kind comes along.
//   bin_format   finished records (row, col, value of glove_cooc_finish_sorted) -> 16-byte records with ids + 1.
//
// One 128-bit load or store per record; memory bound, no shared memory.
#include "glove_common.cuh"

namespace glove {

constexpr int kCrecThreads = 256;
constexpr int kCrecPerThread = 4;      // records per thread of a full grid (grid-stride loop)

__global__ void __launch_bounds__(kCrecThreads) crec_parse_kernel(const int4 *__restrict__ rec, int64_t n, int64_t first,
                                                                  int64_t V, double x_max, double alpha,
                                                                  int32_t *__restrict__ row, int32_t *__restrict__ col,
                                                                  float *__restrict__ target, float *__restrict__ weight,
                                                                  unsigned long long *error) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    unsigned long long bad = ~0ull;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int4 r = __ldcs(rec + i);
        const double val = __hiloint2double(r.w, r.z);
        GLOVE_CREC_KIND(kind, r, val, V);
        if (kind >= 0 && bad == ~0ull) bad = (unsigned long long)(first + i) * 4 + kind;   // i ascends: first bad is lowest
        row[i] = r.x - 1;
        col[i] = r.y - 1;
        target[i] = (float)log(val);
        weight[i] = val >= x_max ? 1.0f : (float)pow(val / x_max, alpha);
    }
    if (bad != ~0ull) atomicMin(error, bad);
}

__global__ void __launch_bounds__(kCrecThreads) crec_format_kernel(const int32_t *__restrict__ row, const int32_t *__restrict__ col,
                                                                   const double *__restrict__ value, int64_t n,
                                                                   int4 *__restrict__ rec) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const double v = value[i];
        __stcs(rec + i, make_int4(row[i] + 1, col[i] + 1, __double2loint(v), __double2hiint(v)));
    }
}

static unsigned crec_blocks(int64_t n) {
    const int64_t per_block = (int64_t)kCrecThreads * kCrecPerThread;
    const int64_t b = (n + per_block - 1) / per_block;
    return (unsigned)(b < (1 << 30) ? b : (1 << 30));
}

}  // namespace glove

using namespace glove;

extern "C" {

int glove_cooc_bin_parse(const void *records, int64_t n, int64_t first_record, int64_t V, double x_max, double alpha,
                         int32_t *row, int32_t *col, float *target, float *weight, unsigned long long *error, void *stream) {
    GLOVE_REQUIRE(records && row && col && target && weight && error, "glove_cooc_bin_parse: null pointer");
    GLOVE_REQUIRE(((uintptr_t)records & 15) == 0, "glove_cooc_bin_parse: records must be 16-byte aligned");
    GLOVE_REQUIRE(n > 0 && first_record >= 0 && first_record <= (INT64_MAX >> 2) - n, "glove_cooc_bin_parse: bad record range");
    GLOVE_REQUIRE(V >= 1 && V < (1ll << 31), "glove_cooc_bin_parse: V must be 1 .. 2^31-1");
    GLOVE_REQUIRE(x_max > 0 && x_max <= 1.7976931348623157e308 && alpha == alpha, "glove_cooc_bin_parse: bad x_max or alpha");
    crec_parse_kernel<<<crec_blocks(n), kCrecThreads, 0, (cudaStream_t)stream>>>((const int4 *)records, n, first_record, V,
                                                                                   x_max, alpha, row, col, target, weight, error);
    GLOVE_CHECK_LAUNCH();
    return GLOVE_OK;
}

int glove_cooc_bin_format(const int32_t *row, const int32_t *col, const double *value, int64_t n, void *records,
                          void *stream) {
    GLOVE_REQUIRE(row && col && value && records, "glove_cooc_bin_format: null pointer");
    GLOVE_REQUIRE(((uintptr_t)records & 15) == 0, "glove_cooc_bin_format: records must be 16-byte aligned");
    GLOVE_REQUIRE(n > 0, "glove_cooc_bin_format: n must be > 0");
    crec_format_kernel<<<crec_blocks(n), kCrecThreads, 0, (cudaStream_t)stream>>>(row, col, value, n, (int4 *)records);
    GLOVE_CHECK_LAUNCH();
    return GLOVE_OK;
}

}  // extern "C"
