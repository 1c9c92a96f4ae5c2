// f32_fmt.cuh — Rust's `Display` for f32 (bamstats.rs:262-265 prints the three identities with `{}`): the shortest decimal
// digits that round-trip, closest to the value, printed positionally ("99.89702", "100", "0.000012", "NaN", "inf").
//
// Free-format algorithm of Steele & White / Burger & Dybvig over a small fixed-width big integer — the same algorithm Rust's
// core::num::flt2dec::strategy::dragon::format_shortest implements (its Grisu fast path falls back to it and is defined to
// agree with it): exact rounding interval (asymmetric at exact powers of two), even mantissas own their interval ends, a
// final-digit tie rounds up.  Integer arithmetic only, no tables, no libc: __host__ __device__.
//
// Status: equal to the oracle's independent fmt_f32 (printf trial + exact-expansion tie test) on every f32 in [0, 100]
// (1 120 403 457 values) and on strided sweeps of the rest; equal to std::to_chars except at 2 048 exact ties in [0, 100], which
// Ryu rounds to even (tests/native/f32_fmt_check.cpp, profiles/r01z_f32_fmt.txt).  The tie rule is stated from knowledge of the
// std sources (std is not present in this image): "parity unpinned", switchable with -DRB_F32_TIE_EVEN.  Used by the C++ host
// (rbh::fmt_f32) today; it is also the core of the GPU-side `rb stats` row formatter that DESIGN.md §8 lists as next.
#pragma once
#include <stdint.h>
#include <string.h>

#include "rb_common.cuh"

namespace rb {

constexpr int F32_LIMBS = 8;  // 256 bits: the largest intermediate is ~2^160 (subnormals scaled by 10^45; 2^128-sized values)
struct Big { uint32_t w[F32_LIMBS]; };

RB_HD void big_zero(Big& a) { for (int i = 0; i < F32_LIMBS; i++) a.w[i] = 0; }
RB_HD void big_set_pow2(Big& a, uint32_t e) { big_zero(a); a.w[e >> 5] = 1u << (e & 31); }
RB_HD void big_set_u32_shl(Big& a, uint32_t v, uint32_t e) {  // a = v * 2^e
    big_zero(a);
    const uint32_t i = e >> 5, b = e & 31;
    a.w[i] = v << b;
    if (b && i + 1 < F32_LIMBS) a.w[i + 1] = v >> (32 - b);
}
RB_HD void big_mul_small(Big& a, uint32_t m) {
    uint64_t c = 0;
    for (int i = 0; i < F32_LIMBS; i++) { c += (uint64_t)a.w[i] * m; a.w[i] = (uint32_t)c; c >>= 32; }
}
RB_HD void big_add(Big& a, const Big& b) {
    uint64_t c = 0;
    for (int i = 0; i < F32_LIMBS; i++) { c += (uint64_t)a.w[i] + b.w[i]; a.w[i] = (uint32_t)c; c >>= 32; }
}
RB_HD void big_sub(Big& a, const Big& b) {  // a >= b
    int64_t c = 0;
    for (int i = 0; i < F32_LIMBS; i++) { c += (int64_t)a.w[i] - (int64_t)b.w[i]; a.w[i] = (uint32_t)c; c >>= 32; }
}
RB_HD int big_cmp(const Big& a, const Big& b) {
    for (int i = F32_LIMBS - 1; i >= 0; i--)
        if (a.w[i] != b.w[i]) return a.w[i] < b.w[i] ? -1 : 1;
    return 0;
}

// Shortest digits of a positive finite f32 given by its bit pattern: value = 0.d1 d2 ... dn x 10^k.  Returns n (1..9).
RB_HD int f32_shortest_digits(uint32_t bits, uint8_t* digits, int& k_out) {
    const uint32_t be = (bits >> 23) & 0xFFu, frac = bits & 0x7FFFFFu;
    const uint32_t f = be ? (frac | 0x800000u) : frac;  // value = f * 2^e
    const int e = be ? (int)be - 150 : -149;
    const bool even = (f & 1u) == 0;                     // round-to-even: an even mantissa owns both ends of its interval
    const bool pow2 = be > 1 && frac == 0;               // the gap below is half the gap above
    Big r, s, mp, mm;
    if (e >= 0) {
        if (!pow2) { big_set_u32_shl(r, f, (uint32_t)e + 1); big_set_pow2(s, 1); big_set_pow2(mp, (uint32_t)e); big_set_pow2(mm, (uint32_t)e); }
        else { big_set_u32_shl(r, f, (uint32_t)e + 2); big_set_pow2(s, 2); big_set_pow2(mp, (uint32_t)e + 1); big_set_pow2(mm, (uint32_t)e); }
    } else {
        if (!pow2) { big_set_u32_shl(r, f, 1); big_set_pow2(s, (uint32_t)(-e) + 1); big_set_pow2(mp, 0); big_set_pow2(mm, 0); }
        else { big_set_u32_shl(r, f, 2); big_set_pow2(s, (uint32_t)(-e) + 2); big_set_pow2(mp, 1); big_set_pow2(mm, 0); }
    }
    int k = 0;
    for (;;) {  // scale s up while (r + m+) / s >= 1
        Big t = r;
        big_add(t, mp);
        const int c = big_cmp(t, s);
        if (even ? c >= 0 : c > 0) { big_mul_small(s, 10); k++; } else break;
    }
    for (;;) {  // scale r up while (r + m+) * 10 / s < 1
        Big t = r;
        big_add(t, mp);
        big_mul_small(t, 10);
        const int c = big_cmp(t, s);
        if (even ? c < 0 : c <= 0) { big_mul_small(r, 10); big_mul_small(mp, 10); big_mul_small(mm, 10); k--; } else break;
    }
    int n = 0;
    for (;;) {
        big_mul_small(r, 10); big_mul_small(mp, 10); big_mul_small(mm, 10);
        uint32_t d = 0;
        while (big_cmp(r, s) >= 0) { big_sub(r, s); d++; }
        const int c1 = big_cmp(r, mm);
        const bool low = even ? c1 <= 0 : c1 < 0;     // the digits so far, cut here, are inside the interval
        Big t = r;
        big_add(t, mp);
        const int c2 = big_cmp(t, s);
        const bool high = even ? c2 >= 0 : c2 > 0;    // ... and so are they with the last digit bumped
        if (!low && !high && n < 16) { digits[n++] = (uint8_t)d; continue; }
        bool up = high;
        if (low && high) {  // both: the closer one; a tie rounds up (dragon.rs format_shortest: `*mant.mul_pow2(1) >= scale`)
            Big t2 = r;
            big_mul_small(t2, 2);
            const int c3 = big_cmp(t2, s);
#ifdef RB_F32_TIE_EVEN  // what printf / Ryu / std::to_chars do with an exact tie (2 048 of the 1.12 G f32 in [0, 100] differ)
            up = c3 > 0 || (c3 == 0 && (d & 1u));
#else
            up = c3 >= 0;
#endif
        }
        digits[n++] = (uint8_t)d;
        if (up) {  // +1 in the last place, carrying through nines
            int i = n - 1;
            while (i >= 0 && digits[i] == 9) { digits[i] = 0; i--; }
            if (i >= 0) digits[i]++;
            else { digits[0] = 1; n = 1; k++; }
            while (n > 1 && digits[n - 1] == 0) n--;
        }
        break;
    }
    k_out = k;
    return n;
}

// ---- fast path for the identities `rb stats` prints (k_emit's RB_WANT_STATS_TEXT rows) ------------------------------------
// The same answer as f32_shortest_digits without big integers, for the values the path produces (0 < v < 2^24 with a binary
// exponent not below 2^-60: 100 * equal / total over u32 counters is 0, NaN or >= 1.1e-8): for n = 1, 2, ... significant
// digits, floor(v * 10^q) and that + 1 are the only n-digit decimals that can lie in v's rounding interval; the first n at
// which one of them does is the shortest length (the free-format algorithm stops at exactly that digit), both -> the closer
// one, an exact tie rounds up.  v * 10^q is a 96-bit integer over a power of two: two 64-bit limbs, shifts and masks.
// Outside that domain: the big-integer core.  Equal to the core on every f32 in [0, 100] (tests/native/f32_fmt_check.cpp).
struct F32Dec {        // value = 0.d1..dn x 10^k with D = d1..dn as an integer ; n == 0: not a positive finite number
    uint32_t D;
    int n, k;
};
RB_HD uint64_t f32_pow10_u64(int q) {  // 10^q, 0 <= q <= 19
    uint64_t p = 1;
    for (int i = 0; i < q; i++) p *= 10ull;
    return p;
}
RB_HD void f32_mul_64x32(uint64_t a, uint32_t b, uint64_t& hi, uint64_t& lo) {  // a * b as 96 bits
    const uint64_t l = (a & 0xFFFFFFFFull) * b, h = (a >> 32) * b;
    lo = l + (h << 32);
    hi = (h >> 32) + (lo < l ? 1ull : 0ull);
}
// the big-integer core as a call of its own (its 256-bit temporaries live on the stack: kept out of the caller's frame); static: one
// copy in every translation unit that uses it
#if defined(__CUDACC__)
static __host__ __device__ __noinline__
#else
inline
#endif
F32Dec f32_shortest_core(uint32_t bits) {
    F32Dec r;
    uint8_t dg[20];
    int k;
    const int n = f32_shortest_digits(bits, dg, k);
    uint32_t D = 0;
    for (int i = 0; i < n; i++) D = D * 10u + dg[i];
    r.D = D; r.n = n; r.k = k;
    return r;
}
RB_HD F32Dec f32_shortest_fast(uint32_t bits) {
    F32Dec r;
    r.D = 0; r.n = 0; r.k = 0;
    const uint32_t be = (bits >> 23) & 0xFFu, frac = bits & 0x7FFFFFu;
    if ((bits >> 31) || be == 0xFFu || (bits & 0x7FFFFFFFu) == 0) return r;
    const uint32_t f = be ? (frac | 0x800000u) : frac;
    const int e = be ? (int)be - 150 : -149;  // v = f * 2^e
    const bool pow2 = be > 1 && frac == 0;    // the gap below is half the gap above
    // v = V * 2^-s with the interval (V - mm, V + mp) in the same unit
    const uint32_t V = pow2 ? 4u * f : 2u * f, mm = 1u, mp = pow2 ? 2u : 1u;
    const int s = pow2 ? 2 - e : 1 - e;
    if (s < 1 || s > 62 || e > 0) return f32_shortest_core(bits);  // outside the fast domain
    const bool even = (f & 1u) == 0;
    // k with 10^(k-1) <= v < 10^k : from the integer part (v < 2^24 here), or by scaling a fraction up
    int k = -99;
    {
        const uint64_t ip = (uint64_t)V >> s;  // floor(v)
        if (ip) { k = 1; for (uint64_t t = ip; t >= 10; t /= 10) k++; }
        else {
            for (int j = 1; j <= 18; j++) {  // the first j with v * 10^j >= 1, i.e. (V * 10^j) >> s != 0 (a 96-bit product)
                uint64_t hi, lo;
                f32_mul_64x32(f32_pow10_u64(j), V, hi, lo);
                if (hi != 0 || (lo >> s) != 0) { k = 1 - j; break; }
            }
        }
    }
    if (k == -99) k = -40;  // smaller than 1e-18: the loop below finds nothing within reach and hands over to the core
    for (int n = 1; n <= 9; n++) {
        const int q = n - k;  // v * 10^q has n digits in front of the point
        uint64_t Dfl, rem_lo, den_lo, m_lo;  // floor(v * 10^q), its remainder, the denominator, one unit of V in the remainder's scale
        if (q >= 0) {
            if (q > 18) break;
            uint64_t nh, nl;
            const uint64_t p10 = f32_pow10_u64(q);
            f32_mul_64x32(p10, V, nh, nl);              // N = V * 10^q ; den = 2^s
            Dfl = (nh << (64 - s)) | (nl >> s);          // N >> s (1 <= s <= 62; the quotient is below 10^9, so the low limb holds it)
            rem_lo = nl & ((1ull << s) - 1ull);
            den_lo = 1ull << s;
            m_lo = p10;                                  // one unit of V scaled like N
        } else {
            const uint64_t p10 = f32_pow10_u64(-q);      // den = 2^s * 10^-q  (v >= 10 here: s <= 21, fits 64 bits)
            if (s > 40) break;
            den_lo = p10 << s;
            Dfl = (uint64_t)V / den_lo;
            rem_lo = (uint64_t)V % den_lo;
            m_lo = 1;
        }
        // low: floor candidate inside the interval  <=>  rem < mm * m   (<= when the mantissa is even)
        // high: floor + 1 inside                    <=>  den - rem < mp * m  (<=)
        const uint64_t lo_w = (uint64_t)mm * m_lo, hi_w = (uint64_t)mp * m_lo, up_gap = den_lo - rem_lo;
        const bool low = even ? rem_lo <= lo_w : rem_lo < lo_w;
        const bool high = even ? up_gap <= hi_w : up_gap < hi_w;
        if (!low && !high) continue;
        bool up = high;
        if (low && high) {
#ifdef RB_F32_TIE_EVEN
            up = 2 * rem_lo > den_lo || (2 * rem_lo == den_lo && (Dfl & 1ull));
#else
            up = 2 * rem_lo >= den_lo;  // the closer one; a tie rounds up
#endif
        }
        uint64_t D = Dfl + (up ? 1ull : 0ull);
        int nn = n, kk = k;
        uint64_t lim = 1;
        for (int i = 0; i < n; i++) lim *= 10ull;
        if (D >= lim) { D /= 10ull; kk++; }  // 9.99.. rounded up to 10.0..: one digit "1", one decade higher
        while (nn > 1 && D % 10ull == 0) { D /= 10ull; nn--; }  // trailing zeros are not digits
        if (D == 0) break;  // (not reachable: v > 0)
        r.D = (uint32_t)D; r.n = nn; r.k = kk;
        return r;
    }
    return f32_shortest_core(bits);  // outside the reach of 64-bit limbs (or, never for an f32, nothing within 9 digits)
}
// bytes `{}` prints for v (F32Dec from f32_shortest_fast; the special values by their bit pattern)
RB_HD uint32_t f32_display_len(uint32_t bits, const F32Dec& d) {
    if (d.n == 0) {
        if ((bits & 0x7F800000u) == 0x7F800000u) return (bits & 0x7FFFFFu) ? 3u : ((bits >> 31) ? 4u : 3u);  // NaN / -inf / inf
        return (bits >> 31) ? 2u : 1u;                                                                        // -0 / 0
    }
    if (d.k <= 0) return 2u + (uint32_t)(-d.k) + (uint32_t)d.n;
    if (d.k >= d.n) return (uint32_t)d.k;
    return (uint32_t)d.n + 1u;
}
RB_HD uint8_t* f32_display_put(uint8_t* p, uint32_t bits, const F32Dec& d) {
    if (d.n == 0) {
        if ((bits & 0x7F800000u) == 0x7F800000u) {
            if (bits & 0x7FFFFFu) { p[0] = 'N'; p[1] = 'a'; p[2] = 'N'; return p + 3; }
            if (bits >> 31) *p++ = '-';
            p[0] = 'i'; p[1] = 'n'; p[2] = 'f';
            return p + 3;
        }
        if (bits >> 31) *p++ = '-';
        *p++ = '0';
        return p;
    }
    uint8_t dg[10];
    uint32_t D = d.D;
    for (int i = d.n - 1; i >= 0; i--) { dg[i] = (uint8_t)('0' + D % 10u); D /= 10u; }
    if (d.k <= 0) {
        *p++ = '0'; *p++ = '.';
        for (int i = 0; i < -d.k; i++) *p++ = '0';
        for (int i = 0; i < d.n; i++) *p++ = dg[i];
    } else if (d.k >= d.n) {
        for (int i = 0; i < d.n; i++) *p++ = dg[i];
        for (int i = d.n; i < d.k; i++) *p++ = '0';
    } else {
        for (int i = 0; i < d.k; i++) *p++ = dg[i];
        *p++ = '.';
        for (int i = d.k; i < d.n; i++) *p++ = dg[i];
    }
    return p;
}

// `format!("{}", v)`: returns the number of bytes written to out (at most 64).
RB_HD int f32_display(float v, uint8_t* out) {
    uint32_t bits;
    memcpy(&bits, &v, 4);
    int p = 0;
    if ((bits & 0x7F800000u) == 0x7F800000u) {
        if (bits & 0x7FFFFFu) { out[0] = 'N'; out[1] = 'a'; out[2] = 'N'; return 3; }
        if (bits >> 31) out[p++] = '-';
        out[p++] = 'i'; out[p++] = 'n'; out[p++] = 'f';
        return p;
    }
    if (bits >> 31) out[p++] = '-';
    if ((bits & 0x7FFFFFFFu) == 0) { out[p++] = '0'; return p; }
    uint8_t dg[20];
    int k;
    const int n = f32_shortest_digits(bits & 0x7FFFFFFFu, dg, k);
    if (k <= 0) {
        out[p++] = '0'; out[p++] = '.';
        for (int i = 0; i < -k; i++) out[p++] = '0';
        for (int i = 0; i < n; i++) out[p++] = (uint8_t)('0' + dg[i]);
    } else if (k >= n) {
        for (int i = 0; i < n; i++) out[p++] = (uint8_t)('0' + dg[i]);
        for (int i = n; i < k; i++) out[p++] = '0';
    } else {
        for (int i = 0; i < k; i++) out[p++] = (uint8_t)('0' + dg[i]);
        out[p++] = '.';
        for (int i = k; i < n; i++) out[p++] = (uint8_t)('0' + dg[i]);
    }
    return p;
}

}  // namespace rb
