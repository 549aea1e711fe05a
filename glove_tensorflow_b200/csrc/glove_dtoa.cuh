// float64 -> text exactly as Python's repr(float) prints it, for the interaction.csv writer (glove_corpus.cu) and the
// host entry glove_format_float64.  pandas' to_csv writes float64 columns with repr, so this is what makes the streamed
// preprocessor's csv byte-identical to save_data's.
//
// Digits: the shortest decimal that parses back to the same double, and of those the one closest to the exact value
// (ties to even) -- the Ryu algorithm (U. Adams, "Ryu: fast float-to-string conversion", PLDI 2018), which yields the
// same digits as the shortest mode of David Gay's dtoa that CPython uses.  The 125-bit multipliers come from
// tools/gen_ryu_table.py (glove_ryu_table.inc).
//
// Layout (CPython's float_repr_style 'short', format code 'r'): with X the exponent of the scientific form,
// -4 <= X <= 15 prints positionally with at least one digit after the point ("2.0", "0.0001", "1234567890123456.0"),
// otherwise "d[.ddd]e+XX" / "d[.ddd]e-XX" with at least two exponent digits ("1e-05", "1e+16", "5e-324").
// 0 -> "0.0", -0 -> "-0.0", NaN -> "nan" (either sign), +-inf -> "inf" / "-inf".  At most kF64TextMax = 24 bytes.
#pragma once
#include <stdint.h>

#include "glove_strtof.cuh"   // GLOVE_HD, mul64

namespace glove {

constexpr int kF64TextMax = 24;

#define GLOVE_RYU_QUAL static const
#define GLOVE_RYU_NAME(x) kRyu##x##Host
#include "glove_ryu_table.inc"
#undef GLOVE_RYU_QUAL
#undef GLOVE_RYU_NAME
#if defined(__CUDACC__)
#define GLOVE_RYU_QUAL static __device__ const
#define GLOVE_RYU_NAME(x) kRyu##x##Dev
#include "glove_ryu_table.inc"
#undef GLOVE_RYU_QUAL
#undef GLOVE_RYU_NAME
#endif

GLOVE_HD int ryu_pow5bits(int e) { return (int)(((uint32_t)e * 1217359u) >> 19) + 1; }   // bit length of 5^e
GLOVE_HD int ryu_log10pow2(int e) { return (int)(((uint32_t)e * 78913u) >> 18); }       // floor(e log10 2)
GLOVE_HD int ryu_log10pow5(int e) { return (int)(((uint32_t)e * 732923u) >> 20); }      // floor(e log10 5)
GLOVE_HD bool ryu_multiple_of_pow5(uint64_t v, int p) {
    int c = 0;
    while (v % 5 == 0) { v /= 5; ++c; }
    return c >= p;
}
// (m * mul) >> j for a 128-bit mul = {low, high} and j >= 64
GLOVE_HD uint64_t ryu_mul_shift(uint64_t m, const uint64_t *mul, int j) {
    uint64_t h0, l0, h1, l1;
    mul64(m, mul[0], h0, l0);
    mul64(m, mul[1], h1, l1);
    const uint64_t lo = l1 + h0, hi = h1 + (lo < l1);
    const int s = j - 64;
    if (s >= 64) return hi >> (s - 64);
    return s == 0 ? lo : (hi << (64 - s)) | (lo >> s);
}

// shortest digits `out_digits` 10^`out_exp` of a finite nonzero double given by its mantissa and biased exponent fields
GLOVE_HD void ryu_d2d(uint64_t ieee_m, uint32_t ieee_e, uint64_t &out_digits, int &out_exp) {
    int e2;
    uint64_t m2;
    if (ieee_e == 0) { e2 = 1 - 1023 - 52 - 2; m2 = ieee_m; }
    else { e2 = (int)ieee_e - 1023 - 52 - 2; m2 = (1ull << 52) | ieee_m; }
    const bool accept_bounds = (m2 & 1) == 0;
    const uint64_t mv = 4 * m2;
    const uint32_t mm_shift = ieee_m != 0 || ieee_e <= 1;
    uint64_t vr, vp, vm;
    int e10;
    bool vm_tz = false, vr_tz = false;
    if (e2 >= 0) {
        const int q = ryu_log10pow2(e2) - (e2 > 3);
        e10 = q;
        const int k = 125 + ryu_pow5bits(q) - 1;
        const int i = -e2 + q + k;
#if defined(__CUDA_ARCH__)
        const uint64_t *mul = kRyuInvDev[q];
#else
        const uint64_t *mul = kRyuInvHost[q];
#endif
        vr = ryu_mul_shift(4 * m2, mul, i);
        vp = ryu_mul_shift(4 * m2 + 2, mul, i);
        vm = ryu_mul_shift(4 * m2 - 1 - mm_shift, mul, i);
        if (q <= 21) {
            if (mv % 5 == 0) vr_tz = ryu_multiple_of_pow5(mv, q);
            else if (accept_bounds) vm_tz = ryu_multiple_of_pow5(mv - 1 - mm_shift, q);
            else vp -= ryu_multiple_of_pow5(mv + 2, q);
        }
    } else {
        const int q = ryu_log10pow5(-e2) - (-e2 > 1);
        e10 = q + e2;
        const int i = -e2 - q;
        const int k = ryu_pow5bits(i) - 125;
        const int j = q - k;
#if defined(__CUDA_ARCH__)
        const uint64_t *mul = kRyuPowDev[i];
#else
        const uint64_t *mul = kRyuPowHost[i];
#endif
        vr = ryu_mul_shift(4 * m2, mul, j);
        vp = ryu_mul_shift(4 * m2 + 2, mul, j);
        vm = ryu_mul_shift(4 * m2 - 1 - mm_shift, mul, j);
        if (q <= 1) {
            vr_tz = true;
            if (accept_bounds) vm_tz = mm_shift == 1;
            else --vp;
        } else if (q < 63) {
            vr_tz = (mv & ((1ull << q) - 1)) == 0;
        }
    }
    int removed = 0;
    uint64_t output;
    if (vm_tz || vr_tz) {
        int last = 0;
        while (vp / 10 > vm / 10) {
            vm_tz &= vm % 10 == 0;
            vr_tz &= last == 0;
            last = (int)(vr % 10);
            vr /= 10; vp /= 10; vm /= 10; ++removed;
        }
        if (vm_tz)
            while (vm % 10 == 0) {
                vr_tz &= last == 0;
                last = (int)(vr % 10);
                vr /= 10; vp /= 10; vm /= 10; ++removed;
            }
        if (vr_tz && last == 5 && vr % 2 == 0) last = 4;   // exactly halfway: round to even
        output = vr + ((vr == vm && (!accept_bounds || !vm_tz)) || last >= 5);
    } else {
        bool round_up = false;
        if (vp / 100 > vm / 100) {
            round_up = vr % 100 >= 50;
            vr /= 100; vp /= 100; vm /= 100; removed += 2;
        }
        while (vp / 10 > vm / 10) {
            round_up = vr % 10 >= 5;
            vr /= 10; vp /= 10; vm /= 10; ++removed;
        }
        output = vr + (vr == vm || round_up);
    }
    out_digits = output;
    out_exp = e10 + removed;
}

// writes repr(x) for the double with bit pattern `bits` to out[0 .. kF64TextMax) and returns its length
GLOVE_HD int format_f64(uint64_t bits, char *out) {
    int n = 0;
    const uint64_t ieee_m = bits & ((1ull << 52) - 1);
    const uint32_t ieee_e = (uint32_t)(bits >> 52) & 0x7ffu;
    if (ieee_e == 0x7ffu && ieee_m) {
        out[0] = 'n'; out[1] = 'a'; out[2] = 'n';
        return 3;
    }
    if (bits >> 63) out[n++] = '-';
    if (ieee_e == 0x7ffu) {
        out[n] = 'i'; out[n + 1] = 'n'; out[n + 2] = 'f';
        return n + 3;
    }
    if (ieee_e == 0 && ieee_m == 0) {
        out[n] = '0'; out[n + 1] = '.'; out[n + 2] = '0';
        return n + 3;
    }
    uint64_t c;
    int k;
    ryu_d2d(ieee_m, ieee_e, c, k);
    while (c % 10 == 0) { c /= 10; ++k; }
    char dig[20];
    int nd = 0;
    for (uint64_t v = c; v; v /= 10) dig[nd++] = (char)('0' + v % 10);   // reversed
    const int X = k + nd - 1;                                              // scientific exponent
    if (X >= -4 && X <= 15) {
        if (X < 0) {
            out[n++] = '0'; out[n++] = '.';
            for (int i = 0; i < -X - 1; ++i) out[n++] = '0';
            for (int i = nd - 1; i >= 0; --i) out[n++] = dig[i];
        } else {
            for (int i = 0; i <= X; ++i) out[n++] = i < nd ? dig[nd - 1 - i] : '0';
            out[n++] = '.';
            if (nd > X + 1)
                for (int i = X + 1; i < nd; ++i) out[n++] = dig[nd - 1 - i];
            else
                out[n++] = '0';
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
    if (ax >= 100) out[n++] = (char)('0' + ax / 100);
    out[n++] = (char)('0' + ax / 10 % 10);
    out[n++] = (char)('0' + ax % 10);
    return n;
}

}  // namespace glove
