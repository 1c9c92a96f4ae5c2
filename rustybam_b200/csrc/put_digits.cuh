// put_digits.cuh — the byte and decimal writers of the row serialisers (k_emit, k_serialise, k_stats_rows), __host__ __device__ so
// that the CPU tests run the same code.  P is a byte pointer into shared or global memory; each returns the position after what it wrote.
#pragma once
#include <stdint.h>

#include "rb_common.cuh"

namespace rb {

template <class P>
RB_HD P put_u32(P p, uint32_t v) {
    if (v < 1000u) {  // CIGAR lengths are mostly 1-3 digits: straight-line code, no loop
        if (v < 10u) { p[0] = (uint8_t)('0' + v); return p + 1; }
        const uint32_t h = (v * 41u) >> 12;    // v / 100 for v < 1000
        const uint32_t r = v - h * 100u;
        const uint32_t t = (r * 103u) >> 10;   // r / 10 for r < 100
        if (v < 100u) { p[0] = (uint8_t)('0' + t); p[1] = (uint8_t)('0' + (r - t * 10u)); return p + 2; }
        p[0] = (uint8_t)('0' + h); p[1] = (uint8_t)('0' + t); p[2] = (uint8_t)('0' + (r - t * 10u));
        return p + 3;
    }
    const uint32_t nd = ndigits32(v);
    int i = (int)nd;
    while (v >= 100u) {  // two digits per division
        const uint32_t q = v / 100u, r = v - q * 100u;
        const uint32_t d1 = (r * 103u) >> 10;  // r / 10 for r < 100
        p[i - 1] = (uint8_t)('0' + (r - d1 * 10u));
        p[i - 2] = (uint8_t)('0' + d1);
        i -= 2;
        v = q;
    }
    if (v >= 10u) {
        const uint32_t d1 = (v * 103u) >> 10;
        p[i - 1] = (uint8_t)('0' + (v - d1 * 10u));
        p[i - 2] = (uint8_t)('0' + d1);
    } else {
        p[i - 1] = (uint8_t)('0' + v);
    }
    return p + nd;
}
template <class P>
RB_HD P put_u64(P p, uint64_t v) {
    if (v < 4294967296ull) return put_u32(p, (uint32_t)v);
    const uint32_t nd = ndigits64(v);
    for (int i = (int)nd - 1; i >= 0; i--) {
        p[i] = (uint8_t)('0' + (uint32_t)(v % 10ull));
        v /= 10ull;
    }
    return p + nd;
}
template <class P>
RB_HD P put_bytes(P p, const uint8_t* __restrict__ src, uint32_t n) {
    for (uint32_t i = 0; i < n; i++) p[i] = src[i];
    return p + n;
}

}  // namespace rb
