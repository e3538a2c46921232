// Edge-list line formatting, written once for the device writer (edgefmt.cu) and for a plain C++ build on the host
// (tests/native/edgefmt_check.cpp; tests/test_edgefmt_cpu.py compares it with Python and with the host writer).
//
// The specification is the host writer (io_edges.cpp): a line is "u<sep>v<sep>weight\n", ids as std::to_chars prints
// an int32, the weight in one of two styles (include/bin3c_io.h), laid out by CPython's format_float_short rules
// (io_edges.cpp: layout()):
//   B3C_FLOAT_REPR   the shortest decimal that reads back to the same double, the closest to the exact value among
//                    the shortest (ties to even): what std::to_chars(chars_format::scientific) gives.  Computed with
//                    the Ryu algorithm (Adams, PLDI 2018): 64 x 128-bit products against the tables of
//                    edgefmt_pow5.h, exact by construction.
//   B3C_FLOAT_STR12  the exact binary value correctly rounded to 12 significant digits, ties to even: what glibc's
//                    "%.11e" gives.  The same 128-bit products give the scaled value with ~80 fraction bits and an
//                    error under 2 units of the last bit; only when the fraction lies within that bound of one half
//                    (exact ties such as 13-digit integers ending in 5, and near-ties) is it decided exactly, with
//                    multi-word integers (Big).
#pragma once

#include <stdint.h>
#include <string.h>

#include "../../include/bin3c_io.h"

#ifdef __CUDACC__
#define B3C_SHD __host__ __device__ __forceinline__
#define B3C_EDGEFMT_TABLE static __device__ const
#else
#define B3C_SHD inline
#define B3C_EDGEFMT_TABLE static const
#endif

#include "edgefmt_pow5.h"

namespace b3c_edgefmt {

typedef unsigned __int128 u128;

constexpr int MAX_ID_CHARS = 11;                  // "-2147483648"
constexpr int MAX_WEIGHT_CHARS = 24;              // "-d.dddddddddddddddde-308"
constexpr int MAX_LINE_BYTES = MAX_ID_CHARS + 1 + MAX_ID_CHARS + 1 + MAX_WEIGHT_CHARS + 1;
static_assert(MAX_LINE_BYTES == 49, "line bound of include/bin3c_b200.h: B3C_EDGES_MAX_LINE_BYTES");

// the two tables, passed by pointer: device code points at its global-memory copy, host code at the static arrays
struct Pow5 {
    const uint64_t (*pos)[2];
    const uint64_t (*inv)[2];
};

B3C_SHD uint64_t tab_ld(const uint64_t *p) {
#ifdef __CUDA_ARCH__
    return __ldg((const unsigned long long *)p);      // read-only path: lanes read different rows
#else
    return *p;
#endif
}

B3C_SHD int clz64(uint64_t x) {
#ifdef __CUDA_ARCH__
    return __clzll((long long)x);
#else
    return __builtin_clzll(x);
#endif
}

// Ryu's exact integer logarithms (valid far beyond the exponent range of a double)
B3C_SHD int pow5bits(int e) { return (int)(((uint32_t)e * 1217359u) >> 19) + 1; }   // bit length of 5^e
B3C_SHD int log10_pow2(int e) { return (int)(((uint32_t)e * 78913u) >> 18); }        // floor(e log10 2)
B3C_SHD int log10_pow5(int e) { return (int)(((uint32_t)e * 732923u) >> 20); }       // floor(e log10 5)

// (m * mul) >> 64 as a 128-bit value (the low 64 bits of the 192-bit product dropped)
B3C_SHD u128 mul_hi(uint64_t m, const uint64_t *mul) {
    const u128 b0 = (u128)m * tab_ld(mul), b2 = (u128)m * tab_ld(mul + 1);
    return (b0 >> 64) + b2;
}
B3C_SHD uint64_t mul_shift(uint64_t m, const uint64_t *mul, int j) { return (uint64_t)(mul_hi(m, mul) >> (j - 64)); }

B3C_SHD int pow5_factor(uint64_t v) {
    int c = 0;
    while (v % 5 == 0) {
        v /= 5;
        ++c;
    }
    return c;
}

B3C_SHD int decimal_length(uint64_t v) {
    int n = 1;
    while (v >= 10) {
        v /= 10;
        ++n;
    }
    return n;
}

// A finite weight as digits: the value is 0.d_1 d_2 ... d_n * 10^decpt with d = d_1 ... d_n, no trailing zeros
// (the Digits of io_edges.cpp).  kind 1 nan, 2 inf.
struct Weight {
    uint64_t d;
    int n, decpt;
    int kind;
    bool neg;
};

B3C_SHD void strip_zeros(Weight &g) {
    while (g.n > 1 && g.d % 10 == 0) {
        g.d /= 10;
        --g.n;
    }
}

// ---- B3C_FLOAT_REPR: Ryu's d2d, the shortest round-trip digits -------------------------------------------------
B3C_SHD void shortest_digits(uint64_t ieee_m, int ieee_e, const Pow5 &T, uint64_t *out, int *e10_out) {
    int e2;
    uint64_t m2;
    if (ieee_e == 0) {
        e2 = 1 - 1023 - 52 - 2;
        m2 = ieee_m;
    } else {
        e2 = ieee_e - 1023 - 52 - 2;
        m2 = (1ull << 52) | ieee_m;
    }
    const bool accept_bounds = (m2 & 1) == 0;
    const uint64_t mv = 4 * m2;
    const uint64_t mm_shift = (ieee_m != 0 || ieee_e <= 1) ? 1 : 0;
    uint64_t vr, vp, vm;
    int e10;
    bool vm_tz = false, vr_tz = false;
    if (e2 >= 0) {
        const int q = log10_pow2(e2) - (e2 > 3);
        e10 = q;
        const int k = POW5_INV_BITCOUNT + pow5bits(q) - 1;
        const int i = -e2 + q + k;
        const uint64_t *mul = T.inv[q];
        vr = mul_shift(4 * m2, mul, i);
        vp = mul_shift(4 * m2 + 2, mul, i);
        vm = mul_shift(4 * m2 - 1 - mm_shift, mul, i);
        if (q <= 21) {
            if (mv % 5 == 0)
                vr_tz = pow5_factor(mv) >= q;
            else if (accept_bounds)
                vm_tz = pow5_factor(mv - 1 - mm_shift) >= q;
            else
                vp -= pow5_factor(mv + 2) >= q ? 1 : 0;
        }
    } else {
        const int q = log10_pow5(-e2) - (-e2 > 1);
        e10 = q + e2;
        const int i = -e2 - q;
        const int k = pow5bits(i) - POW5_BITCOUNT;
        const int j = q - k;
        const uint64_t *mul = T.pos[i];
        vr = mul_shift(4 * m2, mul, j);
        vp = mul_shift(4 * m2 + 2, mul, j);
        vm = mul_shift(4 * m2 - 1 - mm_shift, mul, j);
        if (q <= 1) {
            vr_tz = true;
            if (accept_bounds)
                vm_tz = mm_shift == 1;
            else
                --vp;
        } else if (q < 63) {
            vr_tz = (mv & ((1ull << q) - 1)) == 0;
        }
    }
    int removed = 0;
    int last = 0;
    uint64_t output;
    if (vm_tz || vr_tz) {
        while (vp / 10 > vm / 10) {
            vm_tz &= vm % 10 == 0;
            vr_tz &= last == 0;
            last = (int)(vr % 10);
            vr /= 10;
            vp /= 10;
            vm /= 10;
            ++removed;
        }
        if (vm_tz) {
            while (vm % 10 == 0) {
                vr_tz &= last == 0;
                last = (int)(vr % 10);
                vr /= 10;
                vp /= 10;
                vm /= 10;
                ++removed;
            }
        }
        if (vr_tz && last == 5 && vr % 2 == 0) last = 4;           // exactly half way: round to even
        output = vr + (((vr == vm && (!accept_bounds || !vm_tz)) || last >= 5) ? 1 : 0);
    } else {
        bool round_up = false;
        if (vp / 100 > vm / 100) {
            round_up = vr % 100 >= 50;
            vr /= 100;
            vp /= 100;
            vm /= 100;
            removed += 2;
        }
        while (vp / 10 > vm / 10) {
            round_up = vr % 10 >= 5;
            vr /= 10;
            vp /= 10;
            vm /= 10;
            ++removed;
        }
        output = vr + ((vr == vm || round_up) ? 1 : 0);
    }
    *out = output;
    *e10_out = e10 + removed;
}

// ---- B3C_FLOAT_STR12: 12 significant digits, correctly rounded --------------------------------------------------
// A non-negative integer of up to BIG_WORDS 32-bit words: enough for m * 5^341 and for m * 2^1024.
constexpr int BIG_WORDS = 36;
struct Big {
    uint32_t w[BIG_WORDS];
};

B3C_SHD void big_set(Big &b, uint64_t v) {
    for (int i = 0; i < BIG_WORDS; ++i) b.w[i] = 0;
    b.w[0] = (uint32_t)v;
    b.w[1] = (uint32_t)(v >> 32);
}
B3C_SHD void big_mul_small(Big &b, uint32_t f) {
    uint64_t carry = 0;
    for (int i = 0; i < BIG_WORDS; ++i) {
        const uint64_t t = (uint64_t)b.w[i] * f + carry;
        b.w[i] = (uint32_t)t;
        carry = t >> 32;
    }
}
B3C_SHD void big_mul_pow5(Big &b, int e) {
    for (; e >= 13; e -= 13) big_mul_small(b, 1220703125u);   // 5^13
    uint32_t f = 1;
    for (; e > 0; --e) f *= 5;
    big_mul_small(b, f);
}
B3C_SHD void big_shl(Big &b, int s) {
    const int ws = s >> 5, bs = s & 31;
    for (int i = BIG_WORDS - 1; i >= 0; --i) {
        const int a = i - ws;
        uint32_t hi = a >= 0 ? b.w[a] : 0u, lo = a >= 1 ? b.w[a - 1] : 0u;
        b.w[i] = bs ? (hi << bs) | (lo >> (32 - bs)) : hi;
    }
}
B3C_SHD int big_cmp(const Big &a, const Big &b) {
    for (int i = BIG_WORDS - 1; i >= 0; --i)
        if (a.w[i] != b.w[i]) return a.w[i] < b.w[i] ? -1 : 1;
    return 0;
}
// sign of a * 5^a5 * 2^a2 - b * 5^b5 * 2^b2 (all exponents >= 0)
B3C_SHD int exact_cmp(uint64_t a, int a5, int a2, uint64_t b, int b5, int b2) {
    Big x, y;
    big_set(x, a);
    big_mul_pow5(x, a5);
    big_shl(x, a2);
    big_set(y, b);
    big_mul_pow5(y, b5);
    big_shl(y, b2);
    return big_cmp(x, y);
}

// round_half_even(m * 2^e2 * 10^k) for 2^63 <= m < 2^64, where the result lies in [10^10, 2 10^12]
B3C_SHD uint64_t scaled_round(uint64_t m, int e2, int k, const Pow5 &T) {
    u128 R;
    int sh;                                       // R / 2^sh estimates the value, under by less than 2 units of R
    if (k >= 0) {
        R = mul_hi(m, T.pos[k]);                  // pos[k] = floor(5^k / 2^t), t = pow5bits(k) - 125
        sh = -(pow5bits(k) - POW5_BITCOUNT + e2 + k + 64);
    } else {
        R = mul_hi(m, T.inv[-k]);                 // inv[j] = floor(2^u / 5^j) + 1, u = pow5bits(j) - 1 + 125
        sh = -(e2 + k - (pow5bits(-k) - 1 + POW5_INV_BITCOUNT) + 64);
    }
    const uint64_t n0 = (uint64_t)(R >> sh);
    const u128 fr = R & (((u128)1 << sh) - 1), half = (u128)1 << (sh - 1);
    if (fr + 2 < half) return n0;
    if (fr > half + 2) return n0 + 1;
    // within the error bound of one half: the sign of 2 * value - (2 n0 + 1), exactly
    int c;
    if (k >= 0) {
        const int s = e2 + k + 1;
        c = exact_cmp(m, k, s > 0 ? s : 0, 2 * n0 + 1, 0, s < 0 ? -s : 0);
    } else {
        const int s = e2 + 1 + k;                 // multiply both sides by 10^-k
        c = exact_cmp(m, 0, s > 0 ? s : 0, 2 * n0 + 1, -k, s < 0 ? -s : 0);
    }
    if (c < 0) return n0;
    if (c > 0) return n0 + 1;
    return n0 + (n0 & 1);
}

constexpr uint64_t E11 = 100000000000ull, E12 = 1000000000000ull;

// 12 correctly rounded significant digits of m2 * 2^e2 (m2 != 0): *d in [10^11, 10^12), value ~ d * 10^(*q - 11)
B3C_SHD void digits12(uint64_t m2, int e2, const Pow5 &T, uint64_t *d, int *q_out) {
    const int lz = clz64(m2);
    const uint64_t m = m2 << lz;
    e2 -= lz;
    const int b = e2 + 64;                        // 2^(b-1) <= value < 2^b
    // q0 = floor((b - 1) log10 2) <= log10(value): the scaled value is >= 10^11 and below 2 10^12
    const int q0 = b - 1 >= 0 ? log10_pow2(b - 1) : -log10_pow2(-(b - 1)) - 1;
    int q = q0;
    uint64_t r = scaled_round(m, e2, 11 - q, T);
    if (r >= E12) {                               // value >= 10^(q0 + 1) - half a unit: one digit fewer of scale
        ++q;
        r = scaled_round(m, e2, 11 - q, T);
    }
    if (r == E12) {                               // rounding carried into a new decade
        r = E11;
        ++q;
    }
    *d = r;
    *q_out = q;
}

// ---- weights ------------------------------------------------------------------------------------------------------
B3C_SHD Weight weight_digits(double w, int style, const Pow5 &T) {
#ifdef __CUDA_ARCH__
    const uint64_t bits = (uint64_t)__double_as_longlong(w);
#else
    uint64_t bits;
    memcpy(&bits, &w, 8);
#endif
    Weight g;
    g.neg = (bits >> 63) != 0;
    g.kind = 0;
    const uint64_t ieee_m = bits & ((1ull << 52) - 1);
    const int ieee_e = (int)((bits >> 52) & 0x7ff);
    if (ieee_e == 0x7ff) {
        g.kind = ieee_m ? 1 : 2;
        g.d = 0;
        g.n = g.decpt = 0;
        return g;
    }
    if (ieee_e == 0 && ieee_m == 0) {
        g.d = 0;
        g.n = 1;
        g.decpt = 1;
        return g;
    }
    if (style == B3C_FLOAT_STR12) {
        const uint64_t m2 = ieee_e ? ((1ull << 52) | ieee_m) : ieee_m;
        const int e2 = (ieee_e ? ieee_e : 1) - 1023 - 52;
        int q;
        digits12(m2, e2, T, &g.d, &q);
        g.n = 12;
        g.decpt = q + 1;
    } else {
        int e10;
        shortest_digits(ieee_m, ieee_e, T, &g.d, &e10);
        g.n = decimal_length(g.d);
        g.decpt = e10 + g.n;
    }
    strip_zeros(g);
    return g;
}

// exponent form when decpt <= -4 or decpt > max_fixed (16 for repr, 12 for str12)
B3C_SHD int max_fixed(int style) { return style == B3C_FLOAT_STR12 ? 12 : 16; }

B3C_SHD int weight_len(const Weight &g, int style) {
    if (g.kind) return g.kind == 1 ? 3 : (g.neg ? 4 : 3);
    const int s = g.neg ? 1 : 0;
    if (g.decpt <= -4 || g.decpt > max_fixed(style)) {
        const int ex = g.decpt - 1;
        return s + 1 + (g.n > 1 ? g.n : 0) + 2 + ((ex >= 100 || ex <= -100) ? 3 : 2);
    }
    if (g.decpt <= 0) return s + 2 - g.decpt + g.n;
    if (g.decpt >= g.n) return s + g.decpt + 2;
    return s + g.n + 1;
}

// the n digits of d to o[0 .. n)
B3C_SHD void put_digits(uint64_t d, int n, char *o) {
    for (int i = n - 1; i >= 0; --i) {
        o[i] = (char)('0' + d % 10);
        d /= 10;
    }
}

// writes weight_len(g, style) bytes
B3C_SHD void weight_put(const Weight &g, int style, char *o) {
    if (g.kind == 1) {
        o[0] = 'n', o[1] = 'a', o[2] = 'n';
        return;
    }
    if (g.kind == 2) {
        if (g.neg) *o++ = '-';
        o[0] = 'i', o[1] = 'n', o[2] = 'f';
        return;
    }
    if (g.neg) *o++ = '-';
    if (g.decpt <= -4 || g.decpt > max_fixed(style)) {
        uint64_t d = g.d;
        for (int i = g.n; i >= 2; --i) {          // d_1 '.' d_2 ... d_n, or d_1 alone
            o[i] = (char)('0' + d % 10);
            d /= 10;
        }
        o[0] = (char)('0' + d);
        if (g.n > 1) o[1] = '.';
        o += g.n > 1 ? g.n + 1 : 1;
        int ex = g.decpt - 1;
        *o++ = 'e';
        *o++ = ex < 0 ? '-' : '+';
        if (ex < 0) ex = -ex;
        if (ex >= 100) *o++ = (char)('0' + ex / 100);
        *o++ = (char)('0' + ex / 10 % 10);
        *o++ = (char)('0' + ex % 10);
    } else if (g.decpt <= 0) {
        *o++ = '0';
        *o++ = '.';
        for (int i = 0; i < -g.decpt; ++i) *o++ = '0';
        put_digits(g.d, g.n, o);
    } else if (g.decpt >= g.n) {
        put_digits(g.d, g.n, o);
        o += g.n;
        for (int i = g.n; i < g.decpt; ++i) *o++ = '0';
        o[0] = '.', o[1] = '0';
    } else {
        uint64_t d = g.d;
        for (int i = g.n; i > g.decpt; --i) {     // the digits after the point, then the point, then the rest
            o[i] = (char)('0' + d % 10);
            d /= 10;
        }
        o[g.decpt] = '.';
        put_digits(d, g.decpt, o);
    }
}

// ---- ids and lines --------------------------------------------------------------------------------------------------
B3C_SHD int id_len(int32_t v) {
    const uint32_t a = v < 0 ? 0u - (uint32_t)v : (uint32_t)v;
    return (v < 0 ? 1 : 0) + decimal_length(a);
}
B3C_SHD void id_put(int32_t v, int len, char *o) {
    uint32_t a = v < 0 ? 0u - (uint32_t)v : (uint32_t)v;
    if (v < 0) *o = '-';
    for (int i = len - 1; i >= (v < 0 ? 1 : 0); --i) {
        o[i] = (char)('0' + a % 10);
        a /= 10;
    }
}

// One line, measured first and then written: the digits of the weight are computed once.
struct Line {
    Weight g;
    int lu, lv, lw;
    B3C_SHD int bytes() const { return lu + lv + lw + 3; }
};

B3C_SHD Line line_measure(int32_t u, int32_t v, double w, int style, const Pow5 &T) {
    Line L;
    L.g = weight_digits(w, style, T);
    L.lu = id_len(u);
    L.lv = id_len(v);
    L.lw = weight_len(L.g, style);
    return L;
}

B3C_SHD void line_put(const Line &L, int32_t u, int32_t v, char sep, int style, char *o) {
    id_put(u, L.lu, o);
    o += L.lu;
    *o++ = sep;
    id_put(v, L.lv, o);
    o += L.lv;
    *o++ = sep;
    weight_put(L.g, style, o);
    o[L.lw] = '\n';
}

}  // namespace b3c_edgefmt
