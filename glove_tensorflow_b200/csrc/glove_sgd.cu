// Stanford GloVe's trainer (glove.c with -threads 1): per-record AdaGrad over the co-occurrence file in file order, run
// exactly on the GPU along the records' dependencies (DESIGN.md section 3, "Stanford GloVe's trainer").
//
// State in glove.c's layout: W and gradsq are 2V rows of d + 1 doubles (rows 0..V-1 word vectors, V..2V-1 context
// vectors, last element the bias).  Records are {a = word1 - 1, c = word2 - 1} plus {L = log(val), f} (glove_sgd_parse).
// Two records conflict only through a shared word1 (row a) or word2 (row V + c), so record j waits for prev[j].x, the
// last earlier record with the same word1, and prev[j].y, the same for word2 (-1: none); every schedule that respects
// those links computes the sequential recurrence.
//
//   parse_kernel   cooccurrence.bin records -> the above, with glove_cooc_bin_parse's validation and error word
//   links_kernel   stable radix sort of (word, index) per side, then adjacent difference -> prev
//   init_kernel    W[i] = (u(seed, i) - 0.5) / d, u a uniform double of splitmix64 (restated in oracle/)
//   epoch_kernel   persistent grid, one warp per record.  Records are claimed in increasing index from a ticket, so a
//                  warp only ever waits on records that running warps hold and progress does not depend on residency.
//                  done[j] = epoch number (never cleared).  Waits use ld.acquire.gpu with __nanosleep backoff and are
//                  bounded by clock64; rows are read with L1-bypassing loads, written, fenced, and published by a
//                  release store.  A link that does not point backwards or a wait past the bound sets the error word.
//   sum_kernel     fixed-shape reduction of the per-record costs: the epoch cost is bit-identical for any grid
//   rows_kernel    W -> float32 rows of the text file (model 0/1/2) and the <unk> row
//
// Arithmetic order (so that no schedule and no contraction changes a bit): lane l sums fma(W[a][b], W[c][b], acc) over
// b = l (mod 32) in ascending b from 0.0, then a __shfl_xor butterfly over 16, 8, 4, 2, 1 (the same bits in every lane);
// the AdaGrad steps are explicit __d*_rn operations in glove.c's order; the two update sums use the same lane/butterfly
// order as the dot.
#include <cub/cub.cuh>

#include "glove_common.cuh"

namespace glove {

constexpr int kSgdThreads = 256;
constexpr int kSgdMaxK = 16;                 // elements per lane: d <= 32 * kSgdMaxK
constexpr int kSumThreads = 256;
constexpr int kSumChunk = kSumThreads * 32;  // values per CTA of one reduction level
constexpr long long kSgdWaitCycles = 1ll << 31;   // about a second at the B200's clocks
constexpr int kSgdBadLink = 1, kSgdTimeout = 2;

__device__ __forceinline__ int ld_acquire_gpu(const int *p) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_gpu(int *p, int v) {
    asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

__host__ __device__ inline uint64_t splitmix64(uint64_t z) {
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

// glove_cooc_bin_parse's records with its validation (GLOVE_CREC_KIND) as the trainer's records: words[i] =
// {word1 - 1, word2 - 1}, lf[i] = {log(val), val > x_max ? 1 : pow(val / x_max, alpha)} in float64, never rounded.
__global__ void __launch_bounds__(256) sgd_parse_kernel(const int4 *__restrict__ rec, int64_t n, int64_t first, int64_t V,
                                                        double x_max, double alpha, int2 *__restrict__ words,
                                                        double2 *__restrict__ lf, unsigned long long *error) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    unsigned long long bad = ~0ull;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int4 r = __ldcs(rec + i);
        const double val = __hiloint2double(r.w, r.z);
        GLOVE_CREC_KIND(kind, r, val, V);
        if (kind >= 0 && bad == ~0ull) bad = (unsigned long long)(first + i) * 4 + kind;
        words[i] = make_int2(r.x - 1, r.y - 1);
        lf[i] = make_double2(log(val), val > x_max ? 1.0 : pow(val / x_max, alpha));
    }
    if (bad != ~0ull) atomicMin(error, bad);
}

__global__ void sgd_keys_kernel(const int2 *__restrict__ words, int64_t n, int side, int32_t *__restrict__ key,
                                int32_t *__restrict__ idx) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int2 w = words[i];
        key[i] = side ? w.y : w.x;
        idx[i] = (int32_t)i;
    }
}

__global__ void sgd_prev_kernel(const int32_t *__restrict__ key, const int32_t *__restrict__ idx, int64_t n, int side,
                                int32_t *__restrict__ prev) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        prev[2 * (int64_t)idx[i] + side] = (i > 0 && key[i - 1] == key[i]) ? idx[i - 1] : -1;
}

__global__ void sgd_init_kernel(double *__restrict__ W, int64_t n, int d, uint64_t seed) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const uint64_t z = splitmix64(seed * 0xD1B54A32D192ED03ull + (uint64_t)i * 0x9E3779B97F4A7C15ull);
        const double u = (double)(z >> 11) * 0x1p-53;
        W[i] = __ddiv_rn(u - 0.5, (double)d);   // u - 0.5 is exact
    }
}

struct SgdEpoch {
    double *W, *G;
    const int2 *words;
    const double2 *lf;
    const int2 *prev;
    int *done;
    double *cost;        // [n] per-record cost (0 for a skipped record)
    int *ctrl;           // [0] ticket, [1] error word; zeroed before the launch
    int64_t V;
    int n, d, epoch;
    double eta, clip;
};

// true once done[q] >= epoch (q < 0: no link); false when the error word is set or the wait passes the bound
__device__ __forceinline__ bool sgd_wait(const SgdEpoch &p, int q) {
    if (q < 0 || ld_acquire_gpu(p.done + q) >= p.epoch) return true;
    const long long t0 = clock64();
    unsigned ns = 32;
    for (;;) {
        __nanosleep(ns);
        ns = min(ns * 2, 256u);
        if (ld_acquire_gpu(p.done + q) >= p.epoch) return true;
        if (*(volatile int *)(p.ctrl + 1)) return false;
        if (clock64() - t0 > kSgdWaitCycles) {
            atomicOr(p.ctrl + 1, kSgdTimeout);
            return false;
        }
    }
}

__device__ __forceinline__ double butterfly_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = __dadd_rn(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ double check_nan(double v) { return isfinite(v) ? v : 0.0; }

template <int K>
__global__ void __launch_bounds__(kSgdThreads) sgd_epoch_kernel(const SgdEpoch p) {
    const int lane = threadIdx.x & 31, d = p.d;
    const int64_t ld = d + 1;
    int next = 0;
    if (lane == 0) next = atomicAdd(p.ctrl, 1);
    next = __shfl_sync(0xffffffffu, next, 0);
    while (next < p.n) {
        const int j = next;
        if (lane == 0) next = atomicAdd(p.ctrl, 1);   // claim the next record now: the atomic overlaps this one
        const int2 w = p.words[j];
        const double2 lf = p.lf[j];
        const int2 pv = p.prev[j];
        if (pv.x >= j || pv.y >= j) {
            if (lane == 0) atomicOr(p.ctrl + 1, kSgdBadLink);
            return;
        }
        const bool ready = sgd_wait(p, pv.x) && sgd_wait(p, pv.y);
        if (!__all_sync(0xffffffffu, ready)) return;
        next = __shfl_sync(0xffffffffu, next, 0);

        double *Wa = p.W + (int64_t)w.x * ld, *Wc = p.W + (p.V + w.y) * ld;
        double *Ga = p.G + (int64_t)w.x * ld, *Gc = p.G + (p.V + w.y) * ld;
        double wa[K], wc[K], ga[K], gc[K];
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const int b = lane + 32 * k;
            if (b < d) { wa[k] = __ldcg(Wa + b); wc[k] = __ldcg(Wc + b); ga[k] = __ldcg(Ga + b); gc[k] = __ldcg(Gc + b); }
        }
        const double ba = __ldcg(Wa + d), bc = __ldcg(Wc + d);
        double acc = 0.0;
#pragma unroll
        for (int k = 0; k < K; ++k)
            if (lane + 32 * k < d) acc = __fma_rn(wa[k], wc[k], acc);
        const double diff = __dadd_rn(butterfly_sum(acc), __dsub_rn(__dadd_rn(ba, bc), lf.x));
        const double fdiff = __dmul_rn(lf.y, diff);
        const bool skip = !isfinite(diff) || !isfinite(fdiff);
        if (lane == 0) p.cost[j] = skip ? 0.0 : __dmul_rn(__dmul_rn(0.5, fdiff), diff);
        if (!skip) {
            double s1 = 0.0, s2 = 0.0;
#pragma unroll
            for (int k = 0; k < K; ++k) {
                if (lane + 32 * k < d) {
                    const double t1 = __dmul_rn(fmin(fmax(__dmul_rn(fdiff, wc[k]), -p.clip), p.clip), p.eta);
                    const double t2 = __dmul_rn(fmin(fmax(__dmul_rn(fdiff, wa[k]), -p.clip), p.clip), p.eta);
                    const double u1 = __ddiv_rn(t1, __dsqrt_rn(ga[k]));
                    const double u2 = __ddiv_rn(t2, __dsqrt_rn(gc[k]));
                    s1 = __dadd_rn(s1, u1);
                    s2 = __dadd_rn(s2, u2);
                    ga[k] = __dadd_rn(ga[k], __dmul_rn(t1, t1));
                    gc[k] = __dadd_rn(gc[k], __dmul_rn(t2, t2));
                    wa[k] = __dsub_rn(wa[k], u1);   // both from the old rows: t1, t2 are taken first
                    wc[k] = __dsub_rn(wc[k], u2);
                }
            }
            const bool update = isfinite(butterfly_sum(s1)) && isfinite(butterfly_sum(s2));
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const int b = lane + 32 * k;
                if (b < d) {
                    if (update) { __stcg(Wa + b, wa[k]); __stcg(Wc + b, wc[k]); }
                    __stcg(Ga + b, ga[k]);
                    __stcg(Gc + b, gc[k]);
                }
            }
            if (lane == 0) {
                const double gba = __ldcg(Ga + d), gbc = __ldcg(Gc + d);
                __stcg(Wa + d, __dsub_rn(ba, check_nan(__ddiv_rn(fdiff, __dsqrt_rn(gba)))));
                __stcg(Wc + d, __dsub_rn(bc, check_nan(__ddiv_rn(fdiff, __dsqrt_rn(gbc)))));
                const double f2 = __dmul_rn(fdiff, fdiff);
                __stcg(Ga + d, __dadd_rn(gba, f2));
                __stcg(Gc + d, __dadd_rn(gbc, f2));
            }
        }
        __threadfence();
        __syncwarp();
        if (lane == 0) st_release_gpu(p.done + j, p.epoch);
    }
}

// out[blockIdx.x] = the sum of x[blockIdx.x * kSumChunk ..) in a fixed shape: thread t adds x[t], x[t + 256], ... of its
// chunk in ascending order from 0.0, then a shared-memory tree halves 256 -> 1.  The last level divides by `divide`.
__global__ void __launch_bounds__(kSumThreads) sgd_sum_kernel(const double *__restrict__ x, int64_t n, double *out,
                                                              double divide) {
    __shared__ double s[kSumThreads];
    const int64_t base = (int64_t)blockIdx.x * kSumChunk;
    double acc = 0.0;
    for (int i = threadIdx.x; i < kSumChunk && base + i < n; i += kSumThreads) acc = __dadd_rn(acc, x[base + i]);
    s[threadIdx.x] = acc;
    __syncthreads();
    for (int h = kSumThreads / 2; h > 0; h >>= 1) {
        if (threadIdx.x < h) s[threadIdx.x] = __dadd_rn(s[threadIdx.x], s[threadIdx.x + h]);
        __syncthreads();
    }
    if (threadIdx.x == 0) out[blockIdx.x] = divide > 0 ? __ddiv_rn(s[0], divide) : s[0];
}

// one thread per (row, column) of the output; row V is the <unk> row: per element the sum over the last m rows of
// W / m in ascending order from 0.0, for both halves, then the model's rule
__global__ void sgd_rows_kernel(const double *__restrict__ W, int64_t V, int d, int model, int64_t rows, float *out) {
    const int ncol = model == 0 ? 2 * d + 2 : d;
    const int64_t ld = d + 1;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < rows * ncol; t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = t / ncol;
        const int col = (int)(t % ncol);
        const int half = (model == 0 && col > d) ? 1 : 0;
        const int b = model == 0 ? col - half * (d + 1) : col;
        double x, y = 0.0;
        if (i < V) {
            x = W[(half * V + i) * ld + b];
            if (model == 2) y = W[(V + i) * ld + b];
        } else {
            const int64_t m = V < 100 ? V : 100;
            x = 0.0;
            for (int64_t a = V - m; a < V; ++a) {
                x = __dadd_rn(x, __ddiv_rn(W[(half * V + a) * ld + b], (double)m));
                if (model == 2) y = __dadd_rn(y, __ddiv_rn(W[(V + a) * ld + b], (double)m));
            }
        }
        out[t] = (float)(model == 2 ? __dadd_rn(x, y) : x);
    }
}

static unsigned sgd_blocks(int64_t n, int threads = 256) {
    const int64_t b = (n + threads - 1) / threads;
    return (unsigned)(b < 4096 ? (b > 0 ? b : 1) : 4096);
}

template <int K>
static int sgd_launch(const SgdEpoch &p, int grid, cudaStream_t st) {
    if (grid <= 0) {
        int per_sm = 0, dev = 0, sms = 0;
        GLOVE_CHECK_CUDA(cudaGetDevice(&dev));
        GLOVE_CHECK_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        GLOVE_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sgd_epoch_kernel<K>, kSgdThreads, 0));
        grid = per_sm * sms;
    }
    sgd_epoch_kernel<K><<<grid, kSgdThreads, 0, st>>>(p);
    GLOVE_CHECK_LAUNCH();
    return GLOVE_OK;
}

}  // namespace glove

using namespace glove;

extern "C" {

int glove_sgd_parse(const void *records, int64_t n, int64_t first_record, int64_t V, double x_max, double alpha,
                    int32_t *words, double *lf, unsigned long long *error, void *stream) {
    GLOVE_REQUIRE(records && words && lf && error, "glove_sgd_parse: null pointer");
    GLOVE_REQUIRE(((uintptr_t)records & 15) == 0 && ((uintptr_t)lf & 15) == 0 && ((uintptr_t)words & 7) == 0,
                  "glove_sgd_parse: records and lf must be 16-byte aligned, words 8-byte aligned");
    GLOVE_REQUIRE(n > 0 && first_record >= 0 && first_record <= (INT64_MAX >> 2) - n, "glove_sgd_parse: bad record range");
    GLOVE_REQUIRE(V >= 1 && V < (1ll << 31), "glove_sgd_parse: V must be 1 .. 2^31-1");
    GLOVE_REQUIRE(x_max > 0 && x_max <= 1.7976931348623157e308 && alpha == alpha, "glove_sgd_parse: bad x_max or alpha");
    sgd_parse_kernel<<<sgd_blocks(n), 256, 0, (cudaStream_t)stream>>>((const int4 *)records, n, first_record, V, x_max,
                                                                       alpha, (int2 *)words, (double2 *)lf, error);
    GLOVE_CHECK_LAUNCH();
    return GLOVE_OK;
}

size_t glove_sgd_links_workspace_bytes(int64_t n) {
    if (n < 1 || n >= (1ll << 31)) return 0;
    size_t temp = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, temp, (const int32_t *)nullptr, (int32_t *)nullptr, (const int32_t *)nullptr,
                                    (int32_t *)nullptr, (int)n);
    return 4 * align_up(4 * (size_t)n) + align_up(temp);
}

int glove_sgd_links(const int32_t *words, int64_t n, int64_t V, int32_t *prev, void *workspace, size_t workspace_bytes,
                    void *stream) {
    GLOVE_REQUIRE(words && prev && workspace, "glove_sgd_links: null pointer");
    GLOVE_REQUIRE(n >= 1 && n < (1ll << 31), "glove_sgd_links: n must be 1 .. 2^31-1");
    GLOVE_REQUIRE(V >= 1 && V < (1ll << 31), "glove_sgd_links: V must be 1 .. 2^31-1");
    GLOVE_REQUIRE(workspace_bytes >= glove_sgd_links_workspace_bytes(n), "glove_sgd_links: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    char *w = (char *)workspace;
    const size_t a = align_up(4 * (size_t)n);
    int32_t *key_in = (int32_t *)w, *key_out = (int32_t *)(w + a), *idx_in = (int32_t *)(w + 2 * a),
            *idx_out = (int32_t *)(w + 3 * a);
    size_t temp = workspace_bytes - 4 * a;
    int bits = 1;
    while (bits < 31 && (1ll << bits) < V) ++bits;
    for (int side = 0; side < 2; ++side) {
        sgd_keys_kernel<<<sgd_blocks(n), 256, 0, st>>>((const int2 *)words, n, side, key_in, idx_in);
        GLOVE_CHECK_LAUNCH();
        GLOVE_CHECK_CUDA(cub::DeviceRadixSort::SortPairs(w + 4 * a, temp, key_in, key_out, idx_in, idx_out, (int)n, 0, bits,
                                                         st));
        sgd_prev_kernel<<<sgd_blocks(n), 256, 0, st>>>(key_out, idx_out, n, side, prev);
        GLOVE_CHECK_LAUNCH();
    }
    return GLOVE_OK;
}

int glove_sgd_init(double *W, int64_t V, int32_t d, uint64_t seed, void *stream) {
    GLOVE_REQUIRE(W, "glove_sgd_init: null pointer");
    GLOVE_REQUIRE(V >= 1 && V < (1ll << 31) && d >= 1, "glove_sgd_init: need V in 1 .. 2^31-1 and d >= 1");
    const int64_t n = 2 * V * (d + 1);
    sgd_init_kernel<<<sgd_blocks(n), 256, 0, (cudaStream_t)stream>>>(W, n, d, seed);
    GLOVE_CHECK_LAUNCH();
    return GLOVE_OK;
}

size_t glove_sgd_epoch_workspace_bytes(int64_t n) {
    if (n < 1 || n >= (1ll << 31)) return 0;
    const int64_t p1 = (n + kSumChunk - 1) / kSumChunk;
    return align_up(8 * (size_t)n) + 2 * align_up(8 * (size_t)p1) + 256;
}

int glove_sgd_epoch(double *W, double *gradsq, int64_t V, int32_t d, const int32_t *words, const double *lf,
                    const int32_t *prev, int64_t n, double eta, double grad_clip, int32_t epoch, int32_t *done,
                    int32_t grid, void *workspace, size_t workspace_bytes, double *cost, void *stream) {
    GLOVE_REQUIRE(W && gradsq && words && lf && prev && done && workspace && cost, "glove_sgd_epoch: null pointer");
    GLOVE_REQUIRE(V >= 1 && V < (1ll << 31), "glove_sgd_epoch: V must be 1 .. 2^31-1");
    GLOVE_REQUIRE(d >= 1 && d <= 32 * kSgdMaxK, "glove_sgd_epoch: d must be 1 .. %d", 32 * kSgdMaxK);
    GLOVE_REQUIRE(n >= 1 && n < (1ll << 31), "glove_sgd_epoch: n must be 1 .. 2^31-1");
    GLOVE_REQUIRE(epoch >= 1 && grid >= 0, "glove_sgd_epoch: epoch must be >= 1 and grid >= 0");
    GLOVE_REQUIRE(eta == eta && grad_clip == grad_clip, "glove_sgd_epoch: eta and grad_clip must not be NaN");
    GLOVE_REQUIRE(((uintptr_t)lf & 15) == 0 && ((uintptr_t)words & 7) == 0 && ((uintptr_t)prev & 7) == 0,
                  "glove_sgd_epoch: lf must be 16-byte aligned, words and prev 8-byte aligned");
    GLOVE_REQUIRE(workspace_bytes >= glove_sgd_epoch_workspace_bytes(n), "glove_sgd_epoch: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    char *w = (char *)workspace;
    const int64_t p1 = (n + kSumChunk - 1) / kSumChunk;
    double *rec_cost = (double *)w, *part[2] = {(double *)(w + align_up(8 * (size_t)n)),
                                                (double *)(w + align_up(8 * (size_t)n) + align_up(8 * (size_t)p1))};
    int *ctrl = (int *)(w + align_up(8 * (size_t)n) + 2 * align_up(8 * (size_t)p1));
    GLOVE_CHECK_CUDA(cudaMemsetAsync(ctrl, 0, 2 * sizeof(int), st));
    SgdEpoch p{W, gradsq, (const int2 *)words, (const double2 *)lf, (const int2 *)prev, done, rec_cost, ctrl, V, (int)n, d,
               epoch, eta, grad_clip};
    int rc;
    switch ((d + 31) / 32) {
#define GLOVE_SGD_CASE(k) case k: rc = sgd_launch<k>(p, grid, st); break;
        GLOVE_SGD_CASE(1) GLOVE_SGD_CASE(2) GLOVE_SGD_CASE(3) GLOVE_SGD_CASE(4) GLOVE_SGD_CASE(5) GLOVE_SGD_CASE(6)
        GLOVE_SGD_CASE(7) GLOVE_SGD_CASE(8) GLOVE_SGD_CASE(9) GLOVE_SGD_CASE(10) GLOVE_SGD_CASE(11) GLOVE_SGD_CASE(12)
        GLOVE_SGD_CASE(13) GLOVE_SGD_CASE(14) GLOVE_SGD_CASE(15) GLOVE_SGD_CASE(16)
#undef GLOVE_SGD_CASE
        default: rc = GLOVE_EINVAL;
    }
    if (rc != GLOVE_OK) return rc;
    // fixed-shape reduction of the per-record costs; the last level divides by n
    const double *x = rec_cost;
    int64_t m = n;
    for (int level = 0;; ++level) {
        const int64_t blocks = (m + kSumChunk - 1) / kSumChunk;
        double *y = blocks == 1 ? cost : part[level & 1];
        sgd_sum_kernel<<<(unsigned)blocks, kSumThreads, 0, st>>>(x, m, y, blocks == 1 ? (double)n : 0.0);
        GLOVE_CHECK_LAUNCH();
        if (blocks == 1) break;
        x = y;
        m = blocks;
    }
    int err = 0;
    GLOVE_CHECK_CUDA(cudaMemcpyAsync(&err, ctrl + 1, sizeof(int), cudaMemcpyDeviceToHost, st));
    GLOVE_CHECK_CUDA(cudaStreamSynchronize(st));
    if (err & kSgdBadLink) return set_error(GLOVE_EINVAL, "glove_sgd_epoch: a dependency link does not point to an earlier record");
    if (err & kSgdTimeout)
        return set_error(GLOVE_ECUDA, "glove_sgd_epoch: a record waited more than %lld cycles for its dependencies", kSgdWaitCycles);
    return GLOVE_OK;
}

int glove_sgd_rows(const double *W, int64_t V, int32_t d, int32_t model, int32_t unk, float *out, void *stream) {
    GLOVE_REQUIRE(W && out, "glove_sgd_rows: null pointer");
    GLOVE_REQUIRE(V >= 1 && V < (1ll << 31) && d >= 1, "glove_sgd_rows: need V in 1 .. 2^31-1 and d >= 1");
    GLOVE_REQUIRE(model >= 0 && model <= 2 && (unk == 0 || unk == 1), "glove_sgd_rows: model must be 0, 1 or 2, unk 0 or 1");
    const int64_t rows = V + unk;
    sgd_rows_kernel<<<sgd_blocks(rows * (model == 0 ? 2 * d + 2 : d)), 256, 0, (cudaStream_t)stream>>>(W, V, d, model, rows,
                                                                                                       out);
    GLOVE_CHECK_LAUNCH();
    return GLOVE_OK;
}

}  // extern "C"
