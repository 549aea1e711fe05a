// float32 -> shortest decimal text, for the word-vector export (glove_vectors.cu) and the host entry glove_format_float32.
//
// Contract (DESIGN.md §3, "Word vectors in the GloVe text format"): the digits are the SHORTEST decimal that parses back to
// the same float32 under one correct rounding (decimal_to_f32_bits of glove_strtof.cuh, round-half-even); when two digit
// strings of that length both parse back, the one closer to the exact value, and the even one when x lies exactly halfway
// (343126.125 -> 343126.12).  This is the digit string of Dragon4 "unique" mode
// (numpy.format_float_scientific(np.float32(x), unique=True)).
//
// Algorithm.  For p significant digits the candidates are floor(x / 10^k) and that + 1, k = E - p + 1 (E = floor(log10 x),
// exact).  Whether some p-digit decimal parses back is monotone in p (c 10^k parses back => 10c 10^(k-1) does), so the
// shortest p is found by a binary search over p in [1, 9] (9 digits always suffice for float32).  Everything that
// decides the output is exact:
//   - round trip: decimal_to_f32_bits, the parser's own rounding, which reads the 128-bit power-of-five table;
//   - floor(x / 10^k), E, and "which candidate is closer": the sign of m 2^e - c 10^k, evaluated in 192-bit integers
//     (m < 2^24, c < 2^31, |k| <= 53: no product exceeds 2^182).  A double estimate only picks the first floor candidate.
//
// Layout: with E the decimal exponent of the scientific form, -5 <= E <= 8 prints positionally ("0.00001", "-0.05123",
// "123456790"), otherwise "d[.ddd]e+XX" with at least two exponent digits.  0 -> "0", -0 -> "-0", NaN -> "nan",
// +-inf -> "inf" / "-inf".  At most kF32TextMax = 16 bytes.
#pragma once
#include <math.h>
#include <stdint.h>

#include "glove_strtof.cuh"

namespace glove {

constexpr int kF32TextMax = 16;

struct U192 { uint64_t w[3]; };   // little-endian limbs

GLOVE_HD void u192_mul(U192 &a, uint64_t b) {
    uint64_t carry = 0;
    for (int i = 0; i < 3; ++i) {
        uint64_t hi, lo;
        mul64(a.w[i], b, hi, lo);
        lo += carry;
        hi += lo < carry;
        a.w[i] = lo;
        carry = hi;
    }
}
GLOVE_HD void u192_shl(U192 &a, int s) {   // 0 <= s < 192
    const int q = s >> 6, r = s & 63;
    uint64_t o[3];
    for (int i = 2; i >= 0; --i) {
        const int j = i - q;
        uint64_t v = j >= 0 ? a.w[j] << r : 0;
        if (r && j >= 1) v |= a.w[j - 1] >> (64 - r);
        o[i] = v;
    }
    for (int i = 0; i < 3; ++i) a.w[i] = o[i];
}
GLOVE_HD int u192_cmp(const U192 &a, const U192 &b) {
    for (int i = 2; i >= 0; --i)
        if (a.w[i] != b.w[i]) return a.w[i] < b.w[i] ? -1 : 1;
    return 0;
}
GLOVE_HD uint64_t pow5_u64(int n) {   // n <= 27
    uint64_t r = 1, b = 5;
    for (; n; n >>= 1, b *= b)
        if (n & 1) r *= b;
    return r;
}

// sign of m 2^e - c 10^k
GLOVE_HD int cmp_scaled(uint64_t m, int e, uint64_t c, int k) {
    U192 L = {{m, 0, 0}}, R = {{c, 0, 0}};
    U192 &F = k >= 0 ? R : L;
    for (int n = k >= 0 ? k : -k; n > 0; n -= 27) u192_mul(F, pow5_u64(n > 27 ? 27 : n));
    const int s = e - k;
    if (s >= 0) u192_shl(L, s);
    else u192_shl(R, -s);
    return u192_cmp(L, R);
}

// floor(m 2^e / 10^k) for a value whose quotient lies in [1, 2^31)
GLOVE_HD uint64_t floor_scaled(uint64_t m, int e, int k) {
#if defined(__CUDA_ARCH__)
    const Pow5 t = kPow5Dev[k - kPow5Min];
#else
    const Pow5 t = kPow5Host[k - kPow5Min];
#endif
    // 10^k = t.hi 2^(floor(log2 10^k) - 63) to 2^-63
    const int b = (int)(((int64_t)217706 * k) >> 16);
    double y = ldexp((double)m / (double)t.hi, e - b + 63);
    uint64_t c = y < 1.0 ? 1 : (uint64_t)y;
    while (c > 1 && cmp_scaled(m, e, c, k) < 0) --c;
    while (cmp_scaled(m, e, c + 1, k) >= 0) ++c;
    return c;
}

// the closer of the candidates floor(x / 10^k), + 1 that parse back to `bits`; 0 when neither does
GLOVE_HD uint64_t shortest_at(uint32_t bits, uint64_t m, int e, int k) {
    const uint64_t c = floor_scaled(m, e, k);
    const bool lo = decimal_to_f32_bits(c, k) == bits, hi = decimal_to_f32_bits(c + 1, k) == bits;
    if (lo && hi) {   // the closer one; x exactly halfway (e.g. 343126.125 at 8 digits): the even one
        const int s = cmp_scaled(m, e + 1, 2 * c + 1, k);
        return s < 0 || (s == 0 && c % 2 == 0) ? c : c + 1;
    }
    return lo ? c : hi ? c + 1 : 0;
}

// writes the text of the float32 with bit pattern `bits` to out[0 .. kF32TextMax) and returns its length
GLOVE_HD int format_f32(uint32_t bits, char *out) {
    int n = 0;
    const uint32_t mag = bits & 0x7fffffffu;
    if (mag > 0x7f800000u) {
        out[0] = 'n'; out[1] = 'a'; out[2] = 'n';
        return 3;
    }
    if (bits >> 31) out[n++] = '-';
    if (mag == 0x7f800000u) {
        out[n] = 'i'; out[n + 1] = 'n'; out[n + 2] = 'f';
        return n + 3;
    }
    if (mag == 0) {
        out[n] = '0';
        return n + 1;
    }
    const uint32_t bexp = mag >> 23;
    const uint64_t m = bexp ? (mag & 0x7fffffu) | 0x800000u : mag;
    const int e = bexp ? (int)bexp - 150 : -149;
    // E = floor(log10 x): x in [2^t, 2^(t+1)) gives floor(t log10 2) or one more
    const int t = 63 - clz64(m) + e;
    int E = (int)(((int64_t)t * 78913) >> 18);
    if (cmp_scaled(m, e, 1, E + 1) >= 0) ++E;
    int lo = 1, hi = 9;
    while (lo < hi) {
        const int p = (lo + hi) >> 1;
        if (shortest_at(mag, m, e, E - p + 1)) hi = p;
        else lo = p + 1;
    }
    int k = E - lo + 1;
    uint64_t c = shortest_at(mag, m, e, k);
    while (c % 10 == 0) { c /= 10; ++k; }
    char dig[10];
    int nd = 0;
    for (uint64_t v = c; v; v /= 10) dig[nd++] = (char)('0' + v % 10);   // reversed
    const int X = k + nd - 1;                                              // scientific exponent
    if (X >= -5 && X <= 8) {
        if (X < 0) {
            out[n++] = '0'; out[n++] = '.';
            for (int i = 0; i < -X - 1; ++i) out[n++] = '0';
            for (int i = nd - 1; i >= 0; --i) out[n++] = dig[i];
        } else {
            for (int i = 0; i <= X; ++i) out[n++] = i < nd ? dig[nd - 1 - i] : '0';
            if (nd > X + 1) {
                out[n++] = '.';
                for (int i = X + 1; i < nd; ++i) out[n++] = dig[nd - 1 - i];
            }
        }
        return n;
    }
    out[n++] = dig[nd - 1];
    if (nd > 1) {
        out[n++] = '.';
        for (int i = nd - 2; i >= 0; --i) out[n++] = dig[i];
    }
    out[n++] = 'e';
    out[n++] = X < 0 ? '-' : '+';
    const int ax = X < 0 ? -X : X;
    out[n++] = (char)('0' + ax / 10);
    out[n++] = (char)('0' + ax % 10);
    return n;
}

}  // namespace glove
