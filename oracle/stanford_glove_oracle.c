/* The sequential recurrence of Stanford GloVe's glove.c (one thread) over the trainer's 24-byte records, in plain C
 * compiled with -ffp-contract=off by oracle/stanford_glove_oracle.py (DESIGN.md section 3, "Stanford GloVe's trainer").
 * TEST / BENCHMARK INFRASTRUCTURE ONLY.
 *
 * order 0: glove.c's order (the dot and the two update sums ascend over b with separate multiply and add).
 * order 1: the GPU kernel's order: lane l = b mod 32 sums fma(W[a][b], W[c][b], acc) over its b ascending from 0.0, and
 *          the 32 partial sums are combined by the butterfly v[l] += v[l ^ o], o = 16, 8, 4, 2, 1; the update sums the
 *          same way with plain additions. */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

static double butterfly(double *v) {
    double t[32];
    for (int o = 16; o > 0; o >>= 1) {
        for (int l = 0; l < 32; ++l) t[l] = v[l] + v[l ^ o];
        for (int l = 0; l < 32; ++l) v[l] = t[l];
    }
    return v[0];
}

static double check_nan(double v) { return (isnan(v) || isinf(v)) ? 0.0 : v; }

/* One epoch over n records: W, G are 2V rows of d + 1 doubles; words[2j], words[2j+1] = word1 - 1, word2 - 1;
 * lf[2j], lf[2j+1] = log(val), f.  cost[j] receives the record's cost (0 for a skipped record).  Returns 0. */
int sg_oracle_epoch(int64_t V, int32_t d, double *W, double *G, const int32_t *words, const double *lf, int64_t n,
                    double eta, double clip, int32_t order, double *cost) {
    const int64_t ld = d + 1;
    double *u1 = malloc(sizeof(double) * d), *u2 = malloc(sizeof(double) * d);
    if (!u1 || !u2) return -1;
    for (int64_t j = 0; j < n; ++j) {
        double *wa = W + (int64_t)words[2 * j] * ld, *wc = W + (V + words[2 * j + 1]) * ld;
        double *ga = G + (int64_t)words[2 * j] * ld, *gc = G + (V + words[2 * j + 1]) * ld;
        double diff = 0.0;
        if (order == 0) {
            for (int b = 0; b < d; ++b) diff += wa[b] * wc[b];
        } else {
            double acc[32] = {0};
            for (int b = 0; b < d; ++b) acc[b & 31] = fma(wa[b], wc[b], acc[b & 31]);
            diff = butterfly(acc);
        }
        diff = diff + ((wa[d] + wc[d]) - lf[2 * j]);
        double fdiff = lf[2 * j + 1] * diff;
        cost[j] = 0.0;
        if (isnan(diff) || isnan(fdiff) || isinf(diff) || isinf(fdiff)) continue;
        cost[j] = (0.5 * fdiff) * diff;
        double s1[32] = {0}, s2[32] = {0};
        for (int b = 0; b < d; ++b) {
            const double t1 = fmin(fmax(fdiff * wc[b], -clip), clip) * eta;
            const double t2 = fmin(fmax(fdiff * wa[b], -clip), clip) * eta;
            u1[b] = t1 / sqrt(ga[b]);
            u2[b] = t2 / sqrt(gc[b]);
            const int l = order == 0 ? 0 : (b & 31);
            s1[l] += u1[b];
            s2[l] += u2[b];
            ga[b] += t1 * t1;
            gc[b] += t2 * t2;
        }
        const double sum1 = order == 0 ? s1[0] : butterfly(s1), sum2 = order == 0 ? s2[0] : butterfly(s2);
        if (!isnan(sum1) && !isinf(sum1) && !isnan(sum2) && !isinf(sum2)) {
            for (int b = 0; b < d; ++b) {
                wa[b] -= u1[b];
                wc[b] -= u2[b];
            }
        }
        wa[d] -= check_nan(fdiff / sqrt(ga[d]));
        wc[d] -= check_nan(fdiff / sqrt(gc[d]));
        fdiff *= fdiff;
        ga[d] += fdiff;
        gc[d] += fdiff;
    }
    free(u1);
    free(u2);
    return 0;
}

/* Longest dependency chain (in records) over the links prev[2j], prev[2j+1] (-1: none); -1 if a link does not point to
 * an earlier record. */
int64_t sg_oracle_chain(const int32_t *prev, int64_t n) {
    int32_t *depth = malloc(sizeof(int32_t) * (n > 0 ? n : 1));
    if (!depth) return -1;
    int64_t best = 0;
    for (int64_t j = 0; j < n; ++j) {
        int32_t dj = 1;
        for (int s = 0; s < 2; ++s) {
            const int32_t p = prev[2 * j + s];
            if (p >= j) { free(depth); return -1; }
            if (p >= 0 && depth[p] + 1 > dj) dj = depth[p] + 1;
        }
        depth[j] = dj;
        if (dj > best) best = dj;
    }
    free(depth);
    return best;
}
