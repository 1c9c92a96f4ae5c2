// rb_kernels.cu — hand-written sm_100a kernels of the PAF liftover + stats path.
//
//   K1 k_tokenise     CIGAR text -> packed ops, single pass, decoupled look-back on op counts
//                     (replaces rust-htslib CigarString::try_from via paf.rs:398-399)
//   K1b k_rec_ops     per-record op offsets + record-head bitmap + boundary validation
//   K2 k_samples      segmented exclusive scan (decoupled look-back) of 11 prefix counters, sampled
//                     every 32 ops (replaces the per-base arrays of aligned_pairs, paf.rs:501-538)
//   K3 k_rec_prep     indel strip + integrity + window join bounds per record
//                     (paf.rs:656-783, 825-857, 622-627; liftover.rs:123-127)
//      k_pair_scan    pair offsets in emission order (liftover.rs:151-164)
//   K4 k_lift         one thread per (window, record) pair: closed-form lift/trim + fused stats
//                     (liftover.rs:17-105, paf.rs:541-620, bamstats.rs:107-142) — lift_core.cuh
//      k_scan_lines   exclusive scan of line sizes / valid rows (decoupled look-back)
//   K5 k_serialise    PAF text + numeric mirror + stats rows (paf.rs:923-943, bamstats.rs:138-142)
//
// All of it is HBM-bound integer/byte work: no tensor cores on purpose.
#include <algorithm>
#include <cstdio>

#include "f32_fmt.cuh"
#include "lift_core.cuh"
#include "put_digits.cuh"
#include "rb_kernels.cuh"
#include "rec_core.cuh"
#include "stream_core.cuh"

namespace rb {

// ------------------------------------------------------------------------------------------------
// small device helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 ld_nc_v4(const void* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ unsigned long long ld_volatile_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ uint32_t ld_volatile_u32(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ uint4 ld_cg_v4(const void* p) {
    uint4 r;
    asm volatile("ld.global.cg.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ void report(unsigned long long* slot, uint64_t key, uint32_t code) {
    atomicMin(slot, (unsigned long long)((key << 8) | code));
}
// per-byte "is not an ASCII digit": bit 7 of each byte lane set for a non-digit (exact for all 256 byte values)
__device__ __forceinline__ uint32_t nondigit_bytes(uint32_t x) {
    const uint32_t t = x ^ 0x30303030u;  // digits -> 0x00..0x09
    return (((t & 0x7F7F7F7Fu) + 0x76767676u) | t) & 0x80808080u;
}
__device__ __forceinline__ uint32_t nondigit_count(uint4 c) {
    return __popc(nondigit_bytes(c.x)) + __popc(nondigit_bytes(c.y)) + __popc(nondigit_bytes(c.z)) + __popc(nondigit_bytes(c.w));
}
// op character -> BAM code (15 = not one of MIDNSHP=X).  (c & 31) is a perfect hash of the alphabet:
// D=4 H=8 I=9 M=13 N=14 P=16 S=19 X=24 '='=29 ; two 16-nibble tables, then an exact compare.
constexpr unsigned long long make_code_table(int half) {
    unsigned long long t = ~0ull;
    const char alphabet[10] = "MIDNSHP=X";
    for (int c = 0; c < 9; c++) {
        const int k = alphabet[c] & 31;
        if ((k >> 4) == half) {
            t &= ~(15ull << ((k & 15) * 4));
            t |= ((unsigned long long)c) << ((k & 15) * 4);
        }
    }
    return t;
}
constexpr unsigned long long CODE_TBL_LO = make_code_table(0), CODE_TBL_HI = make_code_table(1);
constexpr unsigned long long CODE_CHARS = 0x3D5048534E44494Dull;  // bytes "MIDNSHP=" little-endian, code 8 = 'X'
__device__ __forceinline__ uint32_t char_of_code(uint32_t code) {
    return (code < 8u) ? (uint32_t)((CODE_CHARS >> (code * 8)) & 0xFFu) : 0x58u;
}
__device__ __forceinline__ uint32_t code_of_char(uint32_t ch) {
    const uint32_t k = ch & 31u;
    const uint32_t code = (uint32_t)(((k & 16u) ? CODE_TBL_HI : CODE_TBL_LO) >> ((k & 15u) * 4)) & 15u;
    return (code <= 8u && char_of_code(code) == ch) ? code : 15u;
}

__constant__ uint32_t c_pow10[10] = {1u, 10u, 100u, 1000u, 10000u, 100000u, 1000000u, 10000000u, 100000000u, 1000000000u};

// ------------------------------------------------------------------------------------------------
// decoupled look-back, one 64-bit word per tile: [63:62] = 0 invalid / 1 aggregate / 2 inclusive prefix
// ------------------------------------------------------------------------------------------------
constexpr unsigned long long LB_AGG = 1ull << 62, LB_PRE = 2ull << 62, LB_VAL = (1ull << 62) - 1;

// executed by one full warp; returns the exclusive prefix of `tile` and publishes its inclusive prefix
__device__ __forceinline__ unsigned long long lookback_u64(unsigned long long* state, uint64_t tile, unsigned long long agg) {
    const int lane = threadIdx.x & 31;
    if (tile == 0) {
        if (lane == 0) atomicExch(&state[0], LB_PRE | agg);
        return 0;
    }
    if (lane == 0) atomicExch(&state[tile], LB_AGG | agg);
    unsigned long long excl = 0;
    long long look = (long long)tile - 1;
    for (;;) {
        const long long idx = look - lane;
        unsigned long long s = LB_PRE;  // before tile 0: prefix 0
        if (idx >= 0) {
            do { s = ld_volatile_u64(&state[idx]); } while ((s >> 62) == 0);
        }
        const unsigned pm = __ballot_sync(0xffffffffu, (s >> 62) == 2);
        const int first = pm ? (__ffs(pm) - 1) : 32;
        unsigned long long v = (lane <= first) ? (s & LB_VAL) : 0ull;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
        excl += v;
        if (pm) break;
        look -= 32;
    }
    if (lane == 0) atomicExch(&state[tile], LB_PRE | (excl + agg));
    return excl;
}

// The same look-back in two steps, for blocks that have work to do between knowing their aggregate and needing their
// prefix (k_emit composes its lines in between, which gives the blocks in front time to publish theirs):
// lb_publish by one lane as early as possible, lb_walk by one full warp when the prefix is needed.
__device__ __forceinline__ void lb_publish(unsigned long long* state, uint64_t tile, unsigned long long agg) {
    atomicExch(&state[tile], (tile == 0 ? LB_PRE : LB_AGG) | agg);
}
__device__ __forceinline__ unsigned long long lb_walk(unsigned long long* state, uint64_t tile, unsigned long long agg) {
    const int lane = threadIdx.x & 31;
    if (tile == 0) return 0;
    unsigned long long excl = 0;
    long long look = (long long)tile - 1;
    for (;;) {
        const long long idx = look - lane;
        unsigned long long s = LB_PRE;  // before tile 0: prefix 0
        if (idx >= 0) {
            s = ld_volatile_u64(&state[idx]);
            while ((s >> 62) == 0) { __nanosleep(64); s = ld_volatile_u64(&state[idx]); }  // (sleeping frees the issue slots)
        }
        const unsigned pm = __ballot_sync(0xffffffffu, (s >> 62) == 2);
        const int first = pm ? (__ffs(pm) - 1) : 32;
        unsigned long long v = (lane <= first) ? (s & LB_VAL) : 0ull;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
        excl += v;
        if (pm) break;
        look -= 32;
    }
    if (lane == 0) atomicExch(&state[tile], LB_PRE | (excl + agg));
    return excl;
}

// ------------------------------------------------------------------------------------------------
// K1  tokeniser
// ------------------------------------------------------------------------------------------------
// exact re-parse of the number that ends right before the op character at byte `pos` (rare path:
// >= 9 digits, numbers that span more than one 16-byte chunk).  Returns false on error.
__device__ __noinline__ bool exact_len(const uint8_t* text, uint64_t pos, uint32_t& len, uint32_t& err) {
    long long s = (long long)pos;
    while (text[s - 1] >= '0' && text[s - 1] <= '9') s--;  // text[-1..-16] is 0xFF
    if (s == (long long)pos) { err = RE_CIGAR_PARSE; return false; }
    unsigned long long v = 0;
    for (long long k = s; k < (long long)pos; k++) {
        v = v * 10ull + (unsigned long long)(text[k] - '0');
        if (v > 0xFFFFFFFFull) { err = RE_CIGAR_PARSE; return false; }  // u32::from_str overflow
    }
    if (v > MAX_OP_LEN) { err = RE_UNSUPPORTED; return false; }
    len = (uint32_t)v;
    return true;
}

// ---- async bulk copy (TMA engine, 1-D) + mbarrier: global -> shared staging of a text tile ----
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, unsigned long long* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// shared -> global through the same engine: smem writes of the block must be fenced into the async proxy first
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void bulk_s2g(void* dst, const void* src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(smem_u32(src)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// 4 ASCII digits (most significant in the LOW byte; zeroed bytes count as leading zeros) -> value
__device__ __forceinline__ uint32_t parse4(uint32_t x) {
    x &= 0x0F0F0F0Fu;
    const uint32_t pairs = ((x * 2561u) >> 8) & 0x00FF00FFu;  // d0*10+d1 | d2*10+d3
    return (pairs * 6553601u) >> 16;                          // (d0d1)*100 + d2d3
}

// One tile = TOK_TILE text bytes.  (1) bulk-copy tile + 16-byte look-behind halo into shared memory,
// (2) per thread: 16-byte vector load, op-character bitmask, count; block scan + decoupled look-back give
// the global op index, (3) op positions are compacted into shared memory, (4) one op per thread:
// the 8 bytes in front of the op character are decoded with two SWAR multiplies, stores are coalesced.
__global__ void __launch_bounds__(TOK_THREADS)
k_tokenise(const uint8_t* __restrict__ text, uint32_t* __restrict__ ops, unsigned long long* tile_state, unsigned int* ticket,
           ErrSlots err, uint32_t* misc_flags) {
    __shared__ __align__(16) uint8_t s_text[16 + TOK_TILE + 16];
    __shared__ uint16_t s_pos[TOK_TILE / 2];
#if RB_TOK_EARLY_PUBLISH
    __shared__ uint32_t s_opw[TOK_TILE / 2];  // decoded op words wait here for the tile's place in the op array
#endif
    __shared__ uint8_t s_lut[256];  // byte -> BAM op code (15 = not an op character)
    __shared__ __align__(8) unsigned long long s_bar;
    __shared__ uint32_t s_warp[TOK_THREADS / 32];
    __shared__ unsigned long long s_base;
    __shared__ unsigned int s_tile;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid < 256) s_lut[tid] = (uint8_t)code_of_char((uint32_t)tid);
    if (tid == 0) {
        s_tile = atomicAdd(ticket, 1u);
        mbar_init(&s_bar, 1);
    }
    __syncthreads();
    const uint64_t tile = s_tile;
    const uint64_t tbase = tile * (uint64_t)TOK_TILE;
    if (tid == 0) {
        mbar_expect_tx(&s_bar, 16 + TOK_TILE);
        bulk_g2s(s_text, text + tbase - 16, 16 + TOK_TILE, &s_bar);  // text[-16..0) is 0xFF padding
    }
    mbar_wait(&s_bar, 0);

    const uint4 c = *reinterpret_cast<const uint4*>(s_text + 16 + tid * 16);
    const uint32_t M = 0x01020408u;  // gathers the low bit of each byte into a nibble
    const uint32_t m16 = ((((nondigit_bytes(c.x) >> 7) * M) >> 24) & 0xFu) | (((((nondigit_bytes(c.y) >> 7) * M) >> 24) & 0xFu) << 4) |
                         (((((nondigit_bytes(c.z) >> 7) * M) >> 24) & 0xFu) << 8) | (((((nondigit_bytes(c.w) >> 7) * M) >> 24) & 0xFu) << 12);
    const uint32_t cnt = __popc(m16);

    uint32_t inc = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += t;
    }
    if (lane == 31) s_warp[warp] = inc;
    {   // compact this thread's op positions (tile-relative) while the scan totals settle
        uint32_t mm = m16, k = 0;
        // exclusive index inside the warp is known now; the warp offset is added after the barrier
        const uint32_t wex = inc - cnt;
        __syncthreads();
        uint32_t wpre = 0, total = 0;
#pragma unroll
        for (int w = 0; w < TOK_THREADS / 32; w++) {
            const uint32_t t = s_warp[w];
            if (w < warp) wpre += t;
            total += t;
        }
#if RB_TOK_EARLY_PUBLISH
        // The tile's op count is published NOW and its place in the op array asked for only after the ops are decoded: the
        // decode needs no global index, and by then the tiles in front have published theirs (the block used to sit at a
        // barrier while warp 0 walked the look-back: a third of the kernel's stall samples)
        if (tid == 0) lb_publish(tile_state, tile, total);
#else
        if (warp == 0) {
            const unsigned long long ex = lookback_u64(tile_state, tile, total);
            if (lane == 0) s_base = ex;
        }
#endif
        uint32_t idx = wpre + wex;
        while (mm) {
            const uint32_t j = __ffs(mm) - 1;
            mm &= mm - 1;
            s_pos[idx + k] = (uint16_t)(tid * 16 + j);
            k++;
        }
        __syncthreads();
        const uint32_t* s_w = reinterpret_cast<const uint32_t*>(s_text);
        uint32_t seen_codes = 0;                            // bit c set: an op of code c was seen
#if !RB_TOK_EARLY_PUBLISH
        const uint64_t base = s_base;
        uint32_t* out_ops = ops + base;
#endif
        for (uint32_t q = tid; q < total; q += TOK_THREADS) {
            const uint32_t e = s_pos[q];                    // op character at tile byte e
            const uint32_t a = (e + 8) >> 2, sh = ((e + 8) & 3) * 8;
            const uint32_t w0 = s_w[a], w1 = s_w[a + 1], w2 = s_w[a + 2];
            uint32_t lo = __funnelshift_r(w0, w1, sh);      // bytes e-8 .. e-5
            uint32_t hi = __funnelshift_r(w1, w2, sh);      // bytes e-4 .. e-1
            uint32_t nd;                                    // digits right before e (capped at 8)
            if (q > 0) {
                nd = e - s_pos[q - 1] - 1u;                 // everything between two op characters is digits
                nd = nd > 8u ? 8u : nd;
            } else {                                        // first op of the tile: the run may reach into the halo
                const uint32_t nh = nondigit_bytes(hi), nl = nondigit_bytes(lo);
                nd = nh ? (__clz(nh) >> 3) : (4u + (nl ? (__clz(nl) >> 3) : 4u));
            }
            const uint32_t code = s_lut[s_text[16 + e]];
            uint32_t len;
            if (nd - 1u >= 7u || code == 15u) {             // rare: empty length, >= 8 digits, bad op character
                uint32_t ecode = RE_CIGAR_PARSE;
                len = 0;
                if (code == 15u || !exact_len(text, tbase + e, len, ecode)) { report(err.tok, tbase + e, ecode); len = 0; }
            } else {
                // zero the bytes in front of the digit run (they read as leading zeros): one 64-bit mask
                const unsigned long long x = (((unsigned long long)hi << 32) | lo) & (~0ull << (8u * (8u - nd)));
                len = parse4((uint32_t)(x >> 32));
                if (nd > 4u) len += parse4((uint32_t)x) * 10000u;
            }
            seen_codes |= 1u << code;
            const uint32_t word = (len << 4) | (code == 15u ? (uint32_t)OP_P : code);  // invalid characters were reported above
#if RB_TOK_EARLY_PUBLISH
            s_opw[q] = word;
#else
            out_ops[q] = word;
#endif
        }
        const uint32_t seen_clip = seen_codes & ((1u << OP_S) | (1u << OP_H));
        if (seen_clip) atomicOr(misc_flags, 1u);
#if RB_TOK_EARLY_PUBLISH
        if (warp == 0) {
            const unsigned long long ex = lb_walk(tile_state, tile, total);
            if (lane == 0) s_base = ex;
        }
        __syncthreads();
        uint32_t* out_ops = ops + s_base;
        for (uint32_t q = tid; q < total; q += TOK_THREADS) out_ops[q] = s_opw[q];
#endif
    }
}

// K1b: warp per record (r = 0..n_rec inclusive; r == n_rec yields the total)
__global__ void __launch_bounds__(256)
k_rec_ops(const uint8_t* __restrict__ text, const uint64_t* __restrict__ cigar_off, uint32_t n_rec,
          const unsigned long long* __restrict__ tile_state, uint64_t* __restrict__ op_off, uint32_t* heads, ErrSlots err) {
    const uint32_t r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (r > n_rec) return;
    const uint64_t c = cigar_off[r];
    const uint64_t tile = c / TOK_TILE, tbase = tile * (uint64_t)TOK_TILE;
    const uint64_t prefix = tile ? (tile_state[tile - 1] & LB_VAL) : 0ull;
    const uint32_t nfull = (uint32_t)((c - tbase) >> 4), rem = (uint32_t)((c - tbase) & 15u);
    uint32_t cnt = 0;
    for (uint32_t j = lane; j < nfull; j += 32) cnt += nondigit_count(ld_nc_v4(text + tbase + (uint64_t)j * 16u));
    if (lane == 0 && rem) {
        const uint4 x = ld_nc_v4(text + tbase + (uint64_t)nfull * 16u);
        const uint32_t xw[4] = {x.x, x.y, x.z, x.w};
        for (uint32_t j = 0; j < rem; j++) cnt += ((((xw[j >> 2] >> ((j & 3) * 8)) & 0xFFu) - 48u) >= 10u);
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, d);
    if (lane == 0) {
        const uint64_t o = prefix + cnt;
        op_off[r] = o;
        if (r < n_rec) {
            const uint64_t len = cigar_off[r + 1] - c;
            if (len > 0) {
                atomicOr(&heads[o >> 5], 1u << (o & 31u));
                const uint32_t last = text[c + len - 1], first = text[c];
                if ((last - 48u) < 10u) report(err.rec, r, RE_CIGAR_PARSE);   // "10" : `&bytes[j]` out of bounds
                if ((first - 48u) >= 10u) report(err.rec, r, RE_CIGAR_PARSE); // "M.." : expected length
            }
        }
    }
}

// liftover --qbed: cigar_swap_target_query (paf.rs:1050-1066) in place.  Thread per op; on a '-' record the thread of
// op i (first half) exchanges it with its mirror image, flipping both.
__device__ __forceinline__ uint32_t flip_indel(uint32_t w) {
    const uint32_t c = op_code(w);
    return (c == OP_I || c == OP_D) ? (w ^ 3u) : w;  // codes 1 <-> 2
}
__global__ void __launch_bounds__(256)
k_invert_ops(uint32_t* __restrict__ ops, const uint64_t* __restrict__ op_off, uint32_t n_rec, const uint8_t* __restrict__ strand) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (n_rec == 0 || k >= op_off[n_rec]) return;
    uint32_t lo = 0, hi = n_rec;  // largest r with op_off[r] <= k and op_off[r+1] > k
    while (lo < hi) {
        const uint32_t mid = lo + ((hi - lo) >> 1);
        if (op_off[mid] <= k) lo = mid + 1; else hi = mid;
    }
    const uint32_t r = lo - 1;
    const uint64_t a = op_off[r], b = op_off[r + 1];
    if (strand[r] != '-') { ops[k] = flip_indel(ops[k]); return; }
    const uint64_t i = k - a, m = b - 1 - i;  // mirror position
    if (k < m) {
        const uint32_t x = ops[k], y = ops[m];
        ops[k] = flip_indel(y);
        ops[m] = flip_indel(x);
    } else if (k == m) {
        ops[k] = flip_indel(ops[k]);
    }
}
void launch_invert_ops(uint32_t* ops, const uint64_t* op_off, uint32_t n_rec, const uint8_t* strand, uint64_t n_ops_bound,
                       cudaStream_t s) {
    if (n_rec == 0 || n_ops_bound == 0) return;
    k_invert_ops<<<(unsigned)((n_ops_bound + 255) / 256), 256, 0, s>>>(ops, op_off, n_rec, strand);
}

// rust-htslib placement rules for clips (rare; only launched when the tokeniser saw S or H):
// H only as the first or last op; S only at the ends or separated from them by H only.
__global__ void k_check_clips(const uint32_t* __restrict__ ops, const uint64_t* __restrict__ op_off, uint32_t n_rec, ErrSlots err) {
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rec) return;
    const uint64_t a = op_off[r], b = op_off[r + 1];
    for (uint64_t k = a; k < b; k++) {
        const uint32_t code = op_code(ops[k]);
        if (code == OP_H) {
            if (k != a && k + 1 != b) { report(err.rec, r, RE_CIGAR_PARSE); return; }
        } else if (code == OP_S) {
            bool ok = (k == a) || (k + 1 == b) || (op_code(ops[k - 1]) == OP_H);
            if (!ok) {
                ok = true;
                for (uint64_t j = k + 1; j < b; j++)
                    if (op_code(ops[j]) != OP_H) { ok = false; break; }
            }
            if (!ok) { report(err.rec, r, RE_CIGAR_PARSE); return; }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// K2  sampled segmented scan of the prefix counters
// ------------------------------------------------------------------------------------------------
struct SegVal {
    Ctr c;
    uint32_t flag;
};
// a = earlier span, b = later span
__device__ __forceinline__ SegVal seg_combine(const SegVal& a, const SegVal& b) {
    SegVal r = b;
    if (!b.flag) {
        r.c = a.c;
        ctr_add(r.c, b.c);
    }
    r.flag = a.flag | b.flag;
    return r;
}
__device__ __forceinline__ SegVal seg_shfl(const SegVal& v, int src_lane) {
    SegVal r;
    const uint32_t* in = reinterpret_cast<const uint32_t*>(&v);
    uint32_t* out = reinterpret_cast<uint32_t*>(&r);
#pragma unroll
    for (int k = 0; k < 13; k++) out[k] = __shfl_sync(0xffffffffu, in[k], src_lane);
    return r;
}
__device__ __forceinline__ SegVal seg_identity() {
    SegVal r;
    r.c = ctr_zero();
    r.flag = 0;
    return r;
}
__device__ __forceinline__ void payload_store(ScanPayload* p, const SegVal& v) {
    const uint32_t* in = reinterpret_cast<const uint32_t*>(&v);
    uint4* o = reinterpret_cast<uint4*>(p);
    o[0] = make_uint4(in[0], in[1], in[2], in[3]);
    o[1] = make_uint4(in[4], in[5], in[6], in[7]);
    o[2] = make_uint4(in[8], in[9], in[10], in[11]);
    o[3] = make_uint4(in[12], 0, 0, 0);
}
__device__ __forceinline__ SegVal payload_load(const ScanPayload* p) {
    SegVal v;
    uint32_t* out = reinterpret_cast<uint32_t*>(&v);
    const uint4 a = ld_cg_v4(reinterpret_cast<const uint4*>(p) + 0), b = ld_cg_v4(reinterpret_cast<const uint4*>(p) + 1),
                c = ld_cg_v4(reinterpret_cast<const uint4*>(p) + 2), d = ld_cg_v4(reinterpret_cast<const uint4*>(p) + 3);
    out[0] = a.x; out[1] = a.y; out[2] = a.z; out[3] = a.w;
    out[4] = b.x; out[5] = b.y; out[6] = b.z; out[7] = b.w;
    out[8] = c.x; out[9] = c.y; out[10] = c.z; out[11] = c.w;
    out[12] = d.x;
    return v;
}

// Warp-parallel decoupled look-back with a (Ctr, head flag) payload.  Executed by one full warp.
// Returns the segmented exclusive prefix of block `b` (flag set if a head lies in front inside the chain).
__device__ __forceinline__ SegVal lookback_seg(uint32_t* state, ScanPayload* agg, ScanPayload* pre, uint64_t b, const SegVal& mine) {
    const int lane = threadIdx.x & 31;
    SegVal acc = seg_identity();
    if (b == 0) {
        if (lane == 0) {
            payload_store(&pre[0], mine);
            __threadfence();
            atomicExch(&state[0], 2u);
        }
        return acc;
    }
    if (lane == 0) {
        payload_store(&agg[b], mine);
        __threadfence();
        atomicExch(&state[b], 1u);
    }
    long long look = (long long)b - 1;
    for (;;) {
        const long long idx = look - lane;
        uint32_t st = 2u;
        SegVal x = seg_identity();
        if (idx >= 0) {
            do { st = ld_volatile_u32(&state[idx]); } while (st == 0);
            __threadfence();
            x = payload_load(st == 2u ? &pre[idx] : &agg[idx]);
        }
        // the chain stops at the nearest predecessor that already has its prefix, or whose span holds a head
        const unsigned stopm = __ballot_sync(0xffffffffu, st == 2u || x.flag);
        const int stop = stopm ? (__ffs(stopm) - 1) : 31;
        if (lane > stop) x = seg_identity();
        // ordered reduction: lane l absorbs the EARLIER span held by lane l + d
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const SegVal y = seg_shfl(x, (lane + d) & 31);
            if (lane + d < 32) x = seg_combine(y, x);
        }
        const SegVal tot = seg_shfl(x, 0);
        acc = seg_combine(tot, acc);
        if (stopm) break;
        look -= 32;
        if (look < 0) break;
    }
    if (lane == 0) {
        const SegVal incl = seg_combine(acc, mine);
        payload_store(&pre[b], incl);
        __threadfence();
        atomicExch(&state[b], 2u);
    }
    return acc;
}

// The same look-back with ONE trip to L2 per round and no fences (k_samples2).  A block's slot is four 16-byte vectors, each
// three counter words + a tag (0 = nothing yet, 1 = aggregate, 2 = inclusive prefix; the head flag rides in bit 30 of aux):
// every vector is written and read with a single-copy-atomic 128-bit access (st / ld.relaxed.gpu.b128), a reader that finds four
// equal non-zero tags holds one consistent version — the aggregate and the prefix that later replaces it carry different
// tags, so a mix of the two is seen as such and read again.  The slots are zeroed before every launch.
// Compiled in with -DRB_SMP2_LB2=1 only: measured, it does not pay (rb_kernels.cuh).
__device__ __forceinline__ void st_b128(void* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    const unsigned long long lo = ((unsigned long long)b << 32) | a, hi = ((unsigned long long)d << 32) | c;
    asm volatile("{\n .reg .b128 r;\n mov.b128 r, {%1, %2};\n st.relaxed.gpu.global.b128 [%0], r;\n}" ::"l"(p), "l"(lo), "l"(hi) : "memory");
}
__device__ __forceinline__ uint4 ld_b128(const void* p) {
    unsigned long long lo, hi;
    asm volatile("{\n .reg .b128 r;\n ld.relaxed.gpu.global.b128 r, [%2];\n mov.b128 {%0, %1}, r;\n}" : "=l"(lo), "=l"(hi) : "l"(p) : "memory");
    return make_uint4((uint32_t)lo, (uint32_t)(lo >> 32), (uint32_t)hi, (uint32_t)(hi >> 32));
}
__device__ __forceinline__ void slot_store(ScanPayload* slot, const SegVal& v, uint32_t tag) {
    const uint32_t* in = reinterpret_cast<const uint32_t*>(&v);  // 12 counter words (aux last), then the flag
    const uint32_t aux = (in[11] & ~SUB_ABS) | (v.flag ? SUB_ABS : 0u);
    uint4* o = reinterpret_cast<uint4*>(slot);
    st_b128(o + 0, in[0], in[1], in[2], tag);
    st_b128(o + 1, in[3], in[4], in[5], tag);
    st_b128(o + 2, in[6], in[7], in[8], tag);
    st_b128(o + 3, in[9], in[10], aux, tag);
}
__device__ __forceinline__ uint32_t slot_load(const ScanPayload* slot, SegVal& v) {  // the tag, 0 = not there yet (or torn: read again)
    const uint4* p = reinterpret_cast<const uint4*>(slot);
    const uint4 a = ld_b128(p + 0), b = ld_b128(p + 1), c = ld_b128(p + 2), d = ld_b128(p + 3);
    if (a.w != b.w || b.w != c.w || c.w != d.w) return 0u;
    uint32_t* out = reinterpret_cast<uint32_t*>(&v);
    out[0] = a.x; out[1] = a.y; out[2] = a.z; out[3] = b.x; out[4] = b.y; out[5] = b.z;
    out[6] = c.x; out[7] = c.y; out[8] = c.z; out[9] = d.x; out[10] = d.y;
    out[11] = d.z & ~SUB_ABS;
    v.flag = (d.z & SUB_ABS) ? 1u : 0u;
    return a.w;
}
__device__ __forceinline__ SegVal lookback_seg2(ScanPayload* slots, uint64_t b, const SegVal& mine) {
    const int lane = threadIdx.x & 31;
    SegVal acc = seg_identity();
    if (b == 0) {
        if (lane == 0) slot_store(&slots[0], mine, 2u);
        return acc;
    }
    if (lane == 0) slot_store(&slots[b], mine, 1u);
    long long look = (long long)b - 1;
    for (;;) {
        const long long idx = look - lane;
        uint32_t st = 2u;
        SegVal x = seg_identity();
        if (idx >= 0) {
            do { st = slot_load(&slots[idx], x); } while (st == 0u);
        }
        // the chain stops at the nearest predecessor that already has its prefix, or whose span holds a head
        const unsigned stopm = __ballot_sync(0xffffffffu, st == 2u || x.flag);
        const int stop = stopm ? (__ffs(stopm) - 1) : 31;
        if (lane > stop) x = seg_identity();
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {  // ordered reduction: lane l absorbs the EARLIER span held by lane l + d
            const SegVal y = seg_shfl(x, (lane + d) & 31);
            if (lane + d < 32) x = seg_combine(y, x);
        }
        const SegVal tot = seg_shfl(x, 0);
        acc = seg_combine(tot, acc);
        if (stopm) break;
        look -= 32;
        if (look < 0) break;
    }
    if (lane == 0) slot_store(&slots[b], seg_combine(acc, mine), 2u);
    return acc;
}

// Windows of one record staged in shared memory as relative boundary positions (stream_core.cuh)
struct WinStaged {
    const uint32_t* s_ps;  // ps(j) for j in [js0, ..)
    const uint32_t* s_pe;  // pe(j) for j in [je0, ..)
    uint32_t js0, je0;
    __device__ __forceinline__ uint32_t ps(uint32_t j) const { return s_ps[j - js0]; }
    __device__ __forceinline__ uint32_t pe(uint32_t j) const { return s_pe[j - je0]; }
};
__device__ __forceinline__ void store_half(void* dst, const void* src) {  // 64-byte half result, 4 vector stores
    const uint4* s4 = reinterpret_cast<const uint4*>(src);
    uint4* d4 = reinterpret_cast<uint4*>(dst);
#pragma unroll
    for (int k = 0; k < 4; k++) d4[k] = s4[k];
}

// K2 (+K4 on the sorted-BED fast path).  One thread per 32-op chunk:
//   walk 1   class sums of the chunk -> block-level segmented scan -> decoupled look-back -> samples[chunk]
//   walk 2   (LIFT) the chunk re-walks its ops from shared memory with exact counters and resolves every window
//            boundary whose target position falls into it (stream_core.cuh) -> one 64-byte half result per boundary.
// When the whole block lies inside one record (the common case at scale) the record's window boundaries that fall
// into the block's target range are staged in shared memory first, so the per-chunk searches never leave the SM.
template <bool LIFT>
__global__ void __launch_bounds__(SMP_THREADS, LIFT ? 2 : RB_SMP_MINB)
k_scan_lift(const uint32_t* __restrict__ ops, const uint64_t* __restrict__ n_ops_dev, const uint32_t* __restrict__ heads,
            Ctr* __restrict__ samples, uint32_t* blk_state, ScanPayload* blk_agg, ScanPayload* blk_pre, unsigned int* ticket,
            LiftArgs la) {
    extern __shared__ __align__(16) uint32_t s_dyn[];
    uint32_t* s_ops = s_dyn;                                   // SMP_THREADS * (SAMPLE + 1)
    uint32_t* s_acc = s_ops + SMP_THREADS * (SAMPLE + 1);      // 9 * SMP_THREADS
    uint32_t* s_ps = s_acc + 9 * SMP_THREADS;                  // LIFT: SL_WCAP
    uint32_t* s_pe = s_ps + SL_WCAP;                           // LIFT: SL_WCAP
    __shared__ SegVal s_warp[SMP_THREADS / 32];
    __shared__ SegVal s_blk;
    __shared__ unsigned int s_b;
    __shared__ uint32_t s_hc[SMP_THREADS / 32];
    __shared__ uint32_t s_rblk;
    __shared__ uint32_t s_jr[4];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint64_t n_ops = *n_ops_dev;
    if (tid == 0) s_b = atomicAdd(ticket, 1u);
    __syncthreads();
    const uint64_t b = s_b;
    const uint64_t op0 = b * (uint64_t)SMP_OPS;
    if (op0 >= n_ops && !(n_ops == 0 && b == 0)) return;  // blocks past the end have no successors

    // coalesced load, transposed into a 33-word pitch so that thread t owns s_ops[t*33 .. t*33+31]
    if (op0 + SMP_OPS <= n_ops) {  // full block: 16-byte loads (op0 is a multiple of 8192 -> aligned), 4 ops per thread per step
        const uint4* src = reinterpret_cast<const uint4*>(ops + op0);
#pragma unroll
        for (int i = 0; i < (int)SAMPLE / 4; i++) {
            const uint32_t v4 = (uint32_t)i * SMP_THREADS + tid;  // vector index; ops 4*v4 .. 4*v4+3 lie in one chunk
            const uint4 x = src[v4];
            uint32_t* d = s_ops + (v4 >> (SAMPLE_LOG2 - 2)) * (SAMPLE + 1) + ((v4 << 2) & (SAMPLE - 1));
            d[0] = x.x; d[1] = x.y; d[2] = x.z; d[3] = x.w;
        }
    } else {
#pragma unroll 8
        for (int i = 0; i < (int)SAMPLE; i++) {
            const uint32_t idx = (uint32_t)i * SMP_THREADS + tid;
            const uint64_t g = op0 + idx;
            s_ops[(idx >> SAMPLE_LOG2) * (SAMPLE + 1) + (idx & (SAMPLE - 1))] = (g < n_ops) ? ops[g] : 0u;
        }
    }
    if (LIFT && tid == 32) {  // record that holds the block's first op (largest r with op_off[r] <= op0), off the critical path
        uint32_t lo = 0, hi = la.n_rec;
        while (lo < hi) {
            const uint32_t mid = lo + ((hi - lo) >> 1);
            if (la.op_off[mid] <= op0) lo = mid + 1; else hi = mid;
        }
        s_rblk = lo ? lo - 1 : 0u;
    }
    __syncthreads();

    const uint64_t chunk = b * SMP_THREADS + tid;
    const uint64_t first = chunk << SAMPLE_LOG2;
    int nvalid = 0;
    if (first < n_ops) nvalid = (n_ops - first) < SAMPLE ? (int)(n_ops - first) : (int)SAMPLE;
    const uint32_t h = nvalid ? (uint32_t)((heads[first >> 5] >> (first & 31u)) & (uint32_t)((1ull << SAMPLE) - 1ull)) : 0u;
    uint32_t prev_code = 99u;
    if (nvalid) {
        if (tid > 0) prev_code = op_code(s_ops[(tid - 1) * (SAMPLE + 1) + (SAMPLE - 1)]);
        else if (first > 0) prev_code = op_code(ops[first - 1]);
    }
    SegVal mine = seg_identity();
    ClassAcc acc;
    acc.sum = s_acc + tid; acc.stride = SMP_THREADS;
    acc_reset(acc);
    uint32_t slowc = 0;
    const uint32_t* my_ops = s_ops + tid * (SAMPLE + 1);
    for (int j = 0; j < nvalid; j++) {
        const uint32_t w = my_ops[j];
        const bool head = (h >> j) & 1u;
        if (head) { acc_reset(acc); slowc = 0; }  // a record starts here: the span before it is not part of this aggregate
        if (j && (j & (int)(SUB_OPS - 1)) == 0) {  // sub-sample: counters since the chunk start (or since the last head)
            Ctr sub = ctr_zero();
            if (acc.big >= ACC_BIG) {  // a class sum may have wrapped: exact counters
                int j0 = 0;
                for (int t = 0; t <= j; t++)
                    if ((h >> t) & 1u) j0 = t;
                for (int t = j0; t < j; t++) ctr_add_op(sub, my_ops[t]);
            } else {
                acc_flush(acc, sub);
            }
            sub.aux = (((h >> 1) & ((1u << j) - 1u)) != 0u) ? SUB_ABS : 0u;
            uint4* dst = reinterpret_cast<uint4*>(samples + chunk * SUBS + (uint32_t)(j >> SUB_LOG2));
            const uint32_t* sw = reinterpret_cast<const uint32_t*>(&sub);
            dst[0] = make_uint4(sw[0], sw[1], sw[2], sw[3]);
            dst[1] = make_uint4(sw[4], sw[5], sw[6], sw[7]);
            dst[2] = make_uint4(sw[8], sw[9], sw[10], sw[11]);
        }
        const uint32_t code = op_code(w);
        slowc += (op_len(w) == 0u) | (op_len(w) >= ACC_BIG) | ((!head) & (code == prev_code));
        acc_add_op(acc, w);
        prev_code = code;
    }
    if (acc.big >= ACC_BIG) {  // huge ops: a class sum may have wrapped, redo the chunk with exact counters
        int j0 = 0;
        for (int j = 0; j < nvalid; j++)
            if ((h >> j) & 1u) j0 = j;
        for (int j = j0; j < nvalid; j++) ctr_add_op(mine.c, my_ops[j]);
    } else {
        acc_flush(acc, mine.c);
    }
    mine.c.aux = (mine.c.aux & AUX_OVF) | (slowc & AUX_CNT);
    mine.flag = (h != 0u);

    // block-level segmented scan of the per-chunk aggregates (+ LIFT: count of record heads after the block's first op)
    SegVal inc = mine;
    const uint32_t hc = LIFT ? (uint32_t)__popc(tid == 0 ? (h & ~1u) : h) : 0u;
    uint32_t hinc = hc;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const SegVal y = seg_shfl(inc, (lane - d) & 31);
        if (lane >= d) inc = seg_combine(y, inc);
        if (LIFT) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, hinc, d);
            if (lane >= d) hinc += t;
        }
    }
    if (lane == 31) { s_warp[warp] = inc; if (LIFT) s_hc[warp] = hinc; }
    SegVal exl = seg_shfl(inc, (lane - 1) & 31);
    if (lane == 0) exl = seg_identity();
    __syncthreads();
    SegVal wpre = seg_identity(), btot = seg_identity();
    uint32_t hpre = 0, htot = 0;
    if (LIFT) {
#pragma unroll
        for (int k = 0; k < SMP_THREADS / 32; k++) {
            const SegVal t = s_warp[k];
            if (k < warp) wpre = seg_combine(wpre, t);
            btot = seg_combine(btot, t);
            const uint32_t u = s_hc[k];
            if (k < warp) hpre += u;
            htot += u;
        }
    } else if (warp == 0) {  // only the look-back warp needs the block total ...
#pragma unroll
        for (int k = 0; k < SMP_THREADS / 32; k++) btot = seg_combine(btot, s_warp[k]);
    } else {                 // ... the others the warps in front of them (warp-uniform trip count)
        for (int k = 0; k < warp; k++) wpre = seg_combine(wpre, s_warp[k]);
    }
    if (warp == 0) {
        const SegVal ex = lookback_seg(blk_state, blk_agg, blk_pre, b, btot);
        if (lane == 0) s_blk = ex;
    }
    __syncthreads();
    SegVal pre = seg_combine(seg_combine(s_blk, wpre), exl);
    if (h & 1u) pre.c = ctr_zero();  // op 32c starts a record
    if (nvalid) samples[chunk * SUBS] = pre.c;
    if (!LIFT) return;

    // ---------------- walk 2: window boundaries that fall into this chunk ----------------
    OpsView v;
    v.ops = ops; v.samples = nullptr;
    const uint32_t r_blk = s_rblk;
    const bool one_record = (htot == 0u) && r_blk < la.n_rec;  // block-uniform
    if (one_record) {
        const RecInfo& R = la.recs[r_blk];
        SegRec sr;
        sr.eo0 = R.eo0; sr.eo1 = R.eo1; sr.wlo = R.wlo; sr.whi = R.whi;
        if (sr.whi <= sr.wlo || op0 < R.op_first || op0 >= R.op_end) return;  // block-uniform
        sr.pair0 = la.pair_off[la.rec_rank[r_blk]];
        const WinGlobal wg{la.w_st, la.w_en, R.t_st, R.t_en};
        // the block's own target range -> the slice of window boundaries to stage
        if (warp == 0) {
            const uint32_t T0b = __shfl_sync(0xffffffffu, pre.c.T, 0);  // thread 0's prefix == the block's
            const uint32_t T1b = T0b + btot.c.T;
            uint32_t x = 0;
            if (lane == 0) x = first_true(sr.wlo, sr.whi, [&](uint32_t j) { return wg.ps(j) >= T0b; });
            if (lane == 1) x = first_true(sr.wlo, sr.whi, [&](uint32_t j) { return wg.ps(j) >= T1b; });
            if (lane == 2) x = first_true(sr.wlo, sr.whi, [&](uint32_t j) { return wg.pe(j) > T0b; });
            if (lane == 3) x = first_true(sr.wlo, sr.whi, [&](uint32_t j) { return wg.pe(j) > T1b; });
            if (lane < 4) s_jr[lane] = x;
        }
        __syncthreads();
        const uint32_t js0 = s_jr[0], js1 = s_jr[1], je0 = s_jr[2], je1 = s_jr[3];
        if (js1 <= js0 && je1 <= je0) return;  // no boundary in this block (block-uniform)
        const bool staged = (js1 - js0 <= (uint32_t)SL_WCAP) && (je1 - je0 <= (uint32_t)SL_WCAP);
        if (staged) {
            for (uint32_t i = tid; i < js1 - js0; i += SMP_THREADS) s_ps[i] = wg.ps(js0 + i);
            for (uint32_t i = tid; i < je1 - je0; i += SMP_THREADS) s_pe[i] = wg.pe(je0 + i);
        }
        __syncthreads();
        if (nvalid == 0) return;
        auto seg_op = [&](uint32_t j) { return my_ops[j]; };
        auto emit_s = [&](uint64_t p, const HalfS& hh) { store_half(&la.hs[p], &hh); };
        auto emit_e = [&](uint64_t p, const HalfE& hh) { store_half(&la.he[p], &hh); };
        if (staged) {
            SegRec s2 = sr;
            s2.s_lo = js0; s2.s_hi = js1; s2.e_lo = je0; s2.e_hi = je1;
            const WinStaged ws{s_ps, s_pe, js0, je0};
            stream_segment(v, s2, ws, first, (uint32_t)nvalid, seg_op, pre.c, mine.c.T, acc, emit_s, emit_e);
        } else {
            sr.s_lo = sr.e_lo = sr.wlo; sr.s_hi = sr.e_hi = sr.whi;
            stream_segment(v, sr, wg, first, (uint32_t)nvalid, seg_op, pre.c, mine.c.T, acc, emit_s, emit_e);
        }
        return;
    }

    // general layout: records start inside the block -> every chunk handles its own segments against global memory
    if (nvalid == 0) return;
    const uint32_t hex = hpre + (hinc - hc);  // heads after op0 and before this chunk
    uint32_t r = r_blk + hex + ((tid > 0) ? (h & 1u) : 0u);
    int jb = 0;
    Ctr base = pre.c;
    for (;;) {
        const uint32_t hm = (jb >= 31) ? 0u : (h & ~((2u << jb) - 1u));
        const int je = hm ? (__ffs(hm) - 1) : nvalid;
        const uint64_t k0 = first + (uint64_t)jb;
        if (r < la.n_rec && la.op_off[r] <= k0 && k0 < la.op_off[r + 1]) {
            const RecInfo& R = la.recs[r];
            SegRec sr;
            sr.eo0 = R.eo0; sr.eo1 = R.eo1; sr.wlo = R.wlo; sr.whi = R.whi;
            sr.s_lo = sr.e_lo = sr.wlo; sr.s_hi = sr.e_hi = sr.whi;
            if (sr.whi > sr.wlo) {
                sr.pair0 = la.pair_off[la.rec_rank[r]];
                const WinGlobal wg{la.w_st, la.w_en, R.t_st, R.t_en};
                uint32_t Tseg = 0;
                for (int j = jb; j < je; j++) {
                    const uint32_t w = my_ops[j];
                    if (is_ref(op_code(w))) Tseg += op_len(w);
                }
                stream_segment(v, sr, wg, k0, (uint32_t)(je - jb), [&](uint32_t j) { return my_ops[jb + (int)j]; }, base, Tseg, acc,
                               [&](uint64_t p, const HalfS& hh) { store_half(&la.hs[p], &hh); },
                               [&](uint64_t p, const HalfE& hh) { store_half(&la.he[p], &hh); });
            }
        }
        if (je >= nvalid) break;
        jb = je;
        r++;
        base = ctr_zero();
    }
}

// K2 for rb_liftover / rb_stats (no boundary resolution): the same samples as k_scan_lift<false>, leaner.
//   - op words staged with 16-byte stores into a SWIZZLED tile (unit u of chunk row t sits at t*8 + (u ^ (t & 7))): a thread
//     reads its 32 ops with eight conflict-free 16-byte loads instead of 32 word loads from a 33-word pitch
//   - chunks without a record head that lie fully inside the op array (all but ~1 in 2 000) take a fully unrolled walk:
//     no per-op head / end / sub-sample tests, the zero-length / oversized test is one compare
//   - everything else (scan, look-back, sample layout) is k_scan_lift's
#ifndef RB_SMP2_MINB
#define RB_SMP2_MINB 4
#endif
#ifndef RB_SMP2_MINB_NOSUBS
#define RB_SMP2_MINB_NOSUBS 5
#endif
// NOSUBS (wide windows): absolute samples only.  Its own instantiation: without the sub-sample flushes the walk needs fewer
// registers, and a fifth resident block per SM hides more of the two barriers the profile shows (after the walk, behind the look-back)
template <bool LOCAL, bool NOSUBS = false>
__global__ void __launch_bounds__(SMP_THREADS, NOSUBS ? RB_SMP2_MINB_NOSUBS : RB_SMP2_MINB)
k_samples2(const uint32_t* __restrict__ ops, const uint64_t* __restrict__ n_ops_dev, const uint32_t* __restrict__ heads,
           Ctr* __restrict__ samples, uint32_t* blk_state, ScanPayload* blk_agg, ScanPayload* blk_pre, unsigned int* ticket,
           uint32_t no_subs_arg /* != 0: absolute samples only, marked SUB_ABS (lift_core.cuh: OpsView::no_subs) */) {
    const bool no_subs = NOSUBS || no_subs_arg != 0u;
    static_assert(SAMPLE == 32u, "k_samples2 walks 32-op chunks");
    extern __shared__ __align__(16) uint32_t s_dyn2[];
    uint4* s_ops4 = reinterpret_cast<uint4*>(s_dyn2);             // SMP_THREADS rows of 8 units
    uint32_t* s_acc = s_dyn2 + SMP_THREADS * SAMPLE;              // 9 * SMP_THREADS class sums
    __shared__ SegVal s_warp[SMP_THREADS / 32];
    __shared__ SegVal s_blk;
    __shared__ unsigned int s_b;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint64_t n_ops = *n_ops_dev;
    if (!LOCAL) {  // look-back order = ticket order
        if (tid == 0) s_b = atomicAdd(ticket, 1u);
        __syncthreads();
    }
    const uint64_t b = LOCAL ? (uint64_t)blockIdx.x : (uint64_t)s_b;
    const uint64_t op0 = b * (uint64_t)SMP_OPS;
    if (op0 >= n_ops && !(n_ops == 0 && b == 0)) {  // blocks past the end
        if (LOCAL && tid == 0) payload_store(&blk_agg[b], seg_identity());
        return;
    }

    {   // coalesced 16-byte loads (op0 is a multiple of 8192 ops), swizzled 16-byte stores
        const uint4* src = reinterpret_cast<const uint4*>(ops + op0);
#pragma unroll
        for (int i = 0; i < (int)SAMPLE / 4; i++) {
            const uint32_t v4 = (uint32_t)i * SMP_THREADS + tid;
            uint4 x = make_uint4(0u, 0u, 0u, 0u);
            if (op0 + (uint64_t)v4 * 4u < n_ops) x = src[v4];  // (the op array has slack behind n_ops: a straddling vector is in bounds)
            const uint32_t row = v4 >> 3, u = v4 & 7u;
            s_ops4[row * 8u + (u ^ (row & 7u))] = x;
        }
    }
    __syncthreads();

    const uint64_t chunk = b * SMP_THREADS + tid;
    const uint64_t first = chunk << SAMPLE_LOG2;
    int nvalid = 0;
    if (first < n_ops) nvalid = (n_ops - first) < SAMPLE ? (int)(n_ops - first) : (int)SAMPLE;
    const uint32_t h = nvalid ? heads[first >> 5] : 0u;  // (first is a multiple of 32: one heads word per chunk)
    const uint32_t sw = (uint32_t)tid & 7u;
    const uint4* row = s_ops4 + (uint32_t)tid * 8u;
    auto op_at = [&](int j) { return reinterpret_cast<const uint32_t*>(&row[((uint32_t)j >> 2) ^ sw])[j & 3]; };
    uint32_t prev_code = 99u;
    if (nvalid) {
        if (tid > 0) prev_code = op_code(s_ops4[(uint32_t)(tid - 1) * 8u + (7u ^ ((uint32_t)(tid - 1) & 7u))].w);
        else if (first > 0) prev_code = op_code(ops[first - 1]);
    }
    SegVal mine = seg_identity();
    ClassAcc acc;
    acc.sum = s_acc + tid; acc.stride = SMP_THREADS;
    acc_reset(acc);
    uint32_t slowc = 0;
    auto store_sub = [&](const Ctr& sub, uint32_t k) {
        uint4* dst = reinterpret_cast<uint4*>(samples + chunk * SUBS + k);
        const uint32_t* w = reinterpret_cast<const uint32_t*>(&sub);
        dst[0] = make_uint4(w[0], w[1], w[2], w[3]);
        dst[1] = make_uint4(w[4], w[5], w[6], w[7]);
        dst[2] = make_uint4(w[8], w[9], w[10], w[11]);
    };
    if (nvalid == (int)SAMPLE && h == 0u) {
        // ---- the usual chunk: 32 ops of one record ----
        uint32_t iev = 0, dev = 0, txt = 0, big = 0;
#pragma unroll
        for (int u = 0; u < 8; u++) {
            if (u && !(u & 1) && !no_subs) {  // ops 8, 16, 24: sub-sample = counters since the chunk start
                Ctr sub = ctr_zero();
                acc.iev = iev; acc.dev = dev; acc.txt = txt; acc.big = big;
                if (big >= ACC_BIG) { for (int t = 0; t < 4 * u; t++) ctr_add_op(sub, op_at(t)); }  // a class sum may have wrapped: exact
                else acc_flush(acc, sub);
                sub.aux = 0u;
                store_sub(sub, (uint32_t)u >> 1);
            }
            const uint4 x = row[(uint32_t)u ^ sw];
            const uint32_t ws[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const uint32_t w = ws[k], code = op_code(w), n = op_len(w);
                acc.sum[code * SMP_THREADS] += n;
                iev += (code == OP_I);
                dev += (code == OP_D);
                txt += ndigits32(n) + 1u;
                big |= n;
                slowc += ((n - 1u) >= (ACC_BIG - 1u)) | (code == prev_code);  // zero-length, oversized, or the class of the op before
                prev_code = code;
            }
        }
        acc.iev = iev; acc.dev = dev; acc.txt = txt; acc.big = big;
        if (big >= ACC_BIG) { for (int j = 0; j < (int)SAMPLE; j++) ctr_add_op(mine.c, op_at(j)); }
        else acc_flush(acc, mine.c);
    } else {
        // ---- a record starts inside the chunk, or the op array ends in it: k_scan_lift's general walk ----
        for (int j = 0; j < nvalid; j++) {
            const uint32_t w = op_at(j);
            const bool head = (h >> j) & 1u;
            if (head) { acc_reset(acc); slowc = 0; }
            if (j && (j & (int)(SUB_OPS - 1)) == 0 && !no_subs) {
                Ctr sub = ctr_zero();
                if (acc.big >= ACC_BIG) {
                    int j0 = 0;
                    for (int t = 0; t <= j; t++)
                        if ((h >> t) & 1u) j0 = t;
                    for (int t = j0; t < j; t++) ctr_add_op(sub, op_at(t));
                } else {
                    acc_flush(acc, sub);
                }
                sub.aux = (((h >> 1) & ((1u << j) - 1u)) != 0u) ? SUB_ABS : 0u;
                store_sub(sub, (uint32_t)(j >> SUB_LOG2));
            }
            const uint32_t code = op_code(w);
            slowc += (op_len(w) == 0u) | (op_len(w) >= ACC_BIG) | ((!head) & (code == prev_code));
            acc_add_op(acc, w);
            prev_code = code;
        }
        if (acc.big >= ACC_BIG) {
            int j0 = 0;
            for (int j = 0; j < nvalid; j++)
                if ((h >> j) & 1u) j0 = j;
            for (int j = j0; j < nvalid; j++) ctr_add_op(mine.c, op_at(j));
        } else {
            acc_flush(acc, mine.c);
        }
    }
    mine.c.aux = (mine.c.aux & AUX_OVF) | (slowc & AUX_CNT);
    mine.flag = (h != 0u);

    // block-level segmented scan of the per-chunk aggregates, look-back, absolute samples (as k_scan_lift)
    SegVal inc = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const SegVal y = seg_shfl(inc, (lane - d) & 31);
        if (lane >= d) inc = seg_combine(y, inc);
    }
    if (lane == 31) s_warp[warp] = inc;
    SegVal exl = seg_shfl(inc, (lane - 1) & 31);
    if (lane == 0) exl = seg_identity();
    __syncthreads();
    SegVal wpre = seg_identity(), btot = seg_identity();
    if (LOCAL) {
        // no look-back: the samples stay relative to the block's first op (SUB_ABS in aux: a record starts in between, the
        // sample is complete), the block's aggregate goes to blk_agg; k_blk_scan + k_smp_fix add the part in front of the block.
        // (A chain of 64-byte look-backs over ~6 000 blocks per 50 M ops is what used to bound this kernel, not its walk.)
        for (int k = 0; k < warp; k++) wpre = seg_combine(wpre, s_warp[k]);
        if (tid == SMP_THREADS - 1) payload_store(&blk_agg[b], seg_combine(wpre, inc));
        SegVal pre = seg_combine(wpre, exl);
        if (h & 1u) { pre.c = ctr_zero(); pre.flag = 1u; }  // op 32c starts a record
        if (nvalid) {
            pre.c.aux = (pre.c.aux & ~SUB_ABS) | (pre.flag ? SUB_ABS : 0u);
            samples[chunk * SUBS] = pre.c;
        }
        return;
    }
    if (warp == 0) {
#pragma unroll
        for (int k = 0; k < SMP_THREADS / 32; k++) btot = seg_combine(btot, s_warp[k]);
#if RB_SMP2_LB2
        const SegVal ex = lookback_seg2(blk_agg, b, btot);
#else
        const SegVal ex = lookback_seg(blk_state, blk_agg, blk_pre, b, btot);
#endif
        if (lane == 0) s_blk = ex;
    } else {
        for (int k = 0; k < warp; k++) wpre = seg_combine(wpre, s_warp[k]);
    }
    __syncthreads();
    SegVal pre = seg_combine(seg_combine(s_blk, wpre), exl);
    if (h & 1u) pre.c = ctr_zero();  // op 32c starts a record
    if (no_subs) pre.c.aux = (pre.c.aux & ~SUB_ABS) | SUB_ABS;  // (the slow-op count keeps bits 0..29)
    if (nvalid) samples[chunk * SUBS] = pre.c;
}

// ------------------------------------------------------------------------------------------------
// K1 + K2 fused: tokeniser + sampled segmented scan in ONE pass over the text (rb_liftover / rb_stats / rb trim-paf /
// rb break-paf; not --qbed / rb invert, whose op order changes after tokenising).  The op words never travel back from
// HBM to be summed: a tile's ops are decoded into shared memory, eight-op groups ALIGNED TO THE GLOBAL OP INDEX (the first
// look-back — op counts — has given the tile's base by then) are summed by one thread each, a block-level segmented scan +
// a second decoupled look-back (64-byte counter payload, the one k_samples uses) turns the sums into the record-relative
// prefix at every 8th op, and those go straight into `samples` — entry k >> 3 of the array is the prefix in front of op k.
// Sub-samples written here are ABSOLUTE (SUB_ABS set; lift_core.cuh reads both forms).
// Record heads come from a table built by k_rec_heads: the byte position of every record's first op character and, per
// tile, the first record whose first op lies in it.
// ------------------------------------------------------------------------------------------------
constexpr uint32_t TS_NONE = 0xFFFFFFFFu;
__global__ void __launch_bounds__(256)
k_rec_heads(const uint8_t* __restrict__ text, const uint64_t* __restrict__ cigar_off, uint32_t n_rec, uint64_t* __restrict__ head_pos,
            uint32_t* tile_first) {
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rec) return;
    const uint64_t c = cigar_off[r], e = cigar_off[r + 1];
    uint64_t hp = ~0ull;
    // first op character of the record (a length has <= 10 digits; longer digit runs are parse errors the tokeniser reports)
    const uint64_t lim = (e - c > 16u) ? c + 16u : e;
    for (uint64_t p = c; p < lim; p++)
        if (((uint32_t)text[p] - 48u) >= 10u) { hp = p; break; }
    head_pos[r] = hp;
    if (hp != ~0ull) atomicMin(&tile_first[hp / TOK_TILE], r);
}

#ifndef RB_TOKSCAN_MINB
#define RB_TOKSCAN_MINB 4
#endif
__global__ void __launch_bounds__(TOK_THREADS, RB_TOKSCAN_MINB)
k_tok_scan(const uint8_t* __restrict__ text, uint32_t* __restrict__ ops, unsigned long long* tile_state, unsigned int* ticket,
           ErrSlots err, uint32_t* misc_flags, const uint32_t* __restrict__ tile_first, const uint64_t* __restrict__ head_pos,
           uint32_t n_rec, Ctr* __restrict__ samples, uint32_t* seg_state, ScanPayload* seg_agg, ScanPayload* seg_pre) {
    __shared__ __align__(16) uint8_t s_text[16 + TOK_TILE + 16];
    __shared__ uint16_t s_pos[TOK_TILE / 2];
    __shared__ uint32_t s_opw[TOK_TILE / 2];
    __shared__ uint32_t s_head[TOK_TILE / 64 + 1];  // bit j: tile-local op j is the first op of a record
    __shared__ uint16_t s_excl[TOK_THREADS], s_m16[TOK_THREADS];
    __shared__ uint8_t s_lut[256];
    __shared__ __align__(8) unsigned long long s_bar;
    __shared__ uint32_t s_warp[TOK_THREADS / 32];
    __shared__ SegVal s_wagg[TOK_THREADS / 32];
    __shared__ SegVal s_blk;
    __shared__ unsigned long long s_base;
    __shared__ unsigned int s_tile;
    __shared__ uint32_t s_prev0;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid < 256) s_lut[tid] = (uint8_t)code_of_char((uint32_t)tid);
    if (tid < TOK_TILE / 64 + 1) s_head[tid] = 0u;
    if (tid == 0) {
        s_tile = atomicAdd(ticket, 1u);
        mbar_init(&s_bar, 1);
        s_prev0 = 99u;
    }
    __syncthreads();
    const uint64_t tile = s_tile;
    const uint64_t tbase = tile * (uint64_t)TOK_TILE;
    if (tid == 0) {
        mbar_expect_tx(&s_bar, 16 + TOK_TILE);
        bulk_g2s(s_text, text + tbase - 16, 16 + TOK_TILE, &s_bar);  // text[-16..0) is 0xFF padding
    }
    uint32_t r_first = TS_NONE;
    if (warp == TOK_THREADS / 32 - 1) r_first = tile_first[tile];  // (in flight while the tile arrives)
    mbar_wait(&s_bar, 0);

    const uint4 c = *reinterpret_cast<const uint4*>(s_text + 16 + tid * 16);
    const uint32_t M = 0x01020408u;  // gathers the low bit of each byte into a nibble
    const uint32_t m16 = ((((nondigit_bytes(c.x) >> 7) * M) >> 24) & 0xFu) | (((((nondigit_bytes(c.y) >> 7) * M) >> 24) & 0xFu) << 4) |
                         (((((nondigit_bytes(c.z) >> 7) * M) >> 24) & 0xFu) << 8) | (((((nondigit_bytes(c.w) >> 7) * M) >> 24) & 0xFu) << 12);
    const uint32_t cnt = __popc(m16);
    uint32_t inc = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += t;
    }
    if (lane == 31) s_warp[warp] = inc;
    s_m16[tid] = (uint16_t)m16;
    __syncthreads();
    uint32_t wpre = 0, total = 0;
#pragma unroll
    for (int w = 0; w < TOK_THREADS / 32; w++) {
        const uint32_t t = s_warp[w];
        if (w < warp) wpre += t;
        total += t;
    }
    if (warp == 0) {
        const unsigned long long ex = lookback_u64(tile_state, tile, total);
        if (lane == 0) s_base = ex;
    }
    {
        uint32_t mm = m16, k = 0;
        const uint32_t idx = wpre + inc - cnt;
        s_excl[tid] = (uint16_t)idx;
        while (mm) {
            const uint32_t j = __ffs(mm) - 1;
            mm &= mm - 1;
            s_pos[idx + k] = (uint16_t)(tid * 16 + j);
            k++;
        }
    }
    __syncthreads();
    const uint64_t base = s_base;
    if (r_first != TS_NONE) {  // (last warp only) records whose first op lies in this tile -> head bits
        const uint64_t tend = tbase + TOK_TILE;
        for (uint64_t r = (uint64_t)r_first + lane; r < n_rec; r += 32) {
            const uint64_t hp = head_pos[r];
            if (hp == ~0ull) continue;  // empty CIGAR
            if (hp >= tend) break;
            const uint32_t bpos = (uint32_t)(hp - tbase), t = bpos >> 4;
            const uint32_t j = (uint32_t)s_excl[t] + __popc((uint32_t)s_m16[t] & ((1u << (bpos & 15u)) - 1u));
            atomicOr(&s_head[j >> 5], 1u << (j & 31u));
        }
    }
    {
        const uint32_t* s_w = reinterpret_cast<const uint32_t*>(s_text);
        uint32_t seen_codes = 0;                            // bit c set: an op of code c was seen
        uint32_t* out_ops = ops + base;
        for (uint32_t q = tid; q < total; q += TOK_THREADS) {
            const uint32_t e = s_pos[q];                    // op character at tile byte e
            const uint32_t a = (e + 8) >> 2, sh = ((e + 8) & 3) * 8;
            const uint32_t w0 = s_w[a], w1 = s_w[a + 1], w2 = s_w[a + 2];
            uint32_t lo = __funnelshift_r(w0, w1, sh);      // bytes e-8 .. e-5
            uint32_t hi = __funnelshift_r(w1, w2, sh);      // bytes e-4 .. e-1
            uint32_t nd;                                    // digits right before e (capped at 8)
            if (q > 0) {
                nd = e - s_pos[q - 1] - 1u;                 // everything between two op characters is digits
                nd = nd > 8u ? 8u : nd;
            } else {                                        // first op of the tile: the run may reach into the halo
                const uint32_t nh = nondigit_bytes(hi), nl = nondigit_bytes(lo);
                nd = nh ? (__clz(nh) >> 3) : (4u + (nl ? (__clz(nl) >> 3) : 4u));
                // the op character in front of that run (the previous tile's last op): the same-class test of op 0 needs it
                int p = 16 + (int)e - 1;
                while (p >= 0 && ((uint32_t)s_text[p] - 48u) < 10u) p--;
                s_prev0 = (p >= 0) ? (uint32_t)s_lut[s_text[p]] : 99u;
            }
            const uint32_t code = s_lut[s_text[16 + e]];
            uint32_t len;
            if (nd - 1u >= 7u || code == 15u) {             // rare: empty length, >= 8 digits, bad op character
                uint32_t ecode = RE_CIGAR_PARSE;
                len = 0;
                if (code == 15u || !exact_len(text, tbase + e, len, ecode)) { report(err.tok, tbase + e, ecode); len = 0; }
            } else {
                const unsigned long long x = (((unsigned long long)hi << 32) | lo) & (~0ull << (8u * (8u - nd)));
                len = parse4((uint32_t)(x >> 32));
                if (nd > 4u) len += parse4((uint32_t)x) * 10000u;
            }
            seen_codes |= 1u << code;
            const uint32_t word = (len << 4) | (code == 15u ? (uint32_t)OP_P : code);  // invalid characters were reported above
            out_ops[q] = word;
            s_opw[q] = word;
        }
        const uint32_t seen_clip = seen_codes & ((1u << OP_S) | (1u << OP_H));
        if (seen_clip) atomicOr(misc_flags, 1u);
    }
    __syncthreads();

    // ---- eight-op groups aligned to the global op index: group g = tile-local ops [8g - off, 8g - off + 8) ----
    const uint32_t off = (uint32_t)(base & 7u);
    const uint32_t ngroups = total ? ((total + off + 7u) >> 3) : 0u;
    const uint32_t per = (ngroups + TOK_THREADS - 1) / TOK_THREADS;  // 1; 2 only for a tile of ~2-byte ops (> 2040 of them)
    const uint32_t g0 = (uint32_t)tid * per;
    const int lo_op = (int)(g0 * 8u) - (int)off;
    const uint32_t j_lo = lo_op < 0 ? 0u : (uint32_t)lo_op;
    uint32_t j_hi = (g0 + per) * 8u - off;
    j_hi = j_hi > total ? total : j_hi;
    SegVal mine = seg_identity();
    if (g0 < ngroups) {
        uint32_t slowc = 0;
        uint32_t prev_code = j_lo ? op_code(s_opw[j_lo - 1]) : s_prev0;
        for (uint32_t j = j_lo; j < j_hi; j++) {
            const uint32_t w = s_opw[j];
            const bool head = (s_head[j >> 5] >> (j & 31u)) & 1u;
            if (head) { mine.c = ctr_zero(); slowc = 0; mine.flag = 1u; }
            const uint32_t code = op_code(w), n = op_len(w);
            slowc += ((n - 1u) >= (ACC_BIG - 1u)) | ((!head) & (code == prev_code));
            ctr_add_op(mine.c, w);
            prev_code = code;
        }
        mine.c.aux = (mine.c.aux & AUX_OVF) | (slowc & AUX_CNT);
    }
    SegVal sinc = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const SegVal y = seg_shfl(sinc, (lane - d) & 31);
        if (lane >= d) sinc = seg_combine(y, sinc);
    }
    if (lane == 31) s_wagg[warp] = sinc;
    SegVal exl = seg_shfl(sinc, (lane - 1) & 31);
    if (lane == 0) exl = seg_identity();
    __syncthreads();
    SegVal wp = seg_identity();
    if (warp == 0) {
        SegVal btot = seg_identity();
#pragma unroll
        for (int k = 0; k < TOK_THREADS / 32; k++) btot = seg_combine(btot, s_wagg[k]);
#ifdef RB_TS_NOLB  // (timing experiment only: wrong prefixes)
        const SegVal ex = btot;
#else
        const SegVal ex = lookback_seg(seg_state, seg_agg, seg_pre, tile, btot);
#endif
        if (lane == 0) s_blk = ex;
    } else {
        for (int k = 0; k < warp; k++) wp = seg_combine(wp, s_wagg[k]);
    }
    __syncthreads();
    if (g0 >= ngroups) return;
    SegVal pre = seg_combine(seg_combine(s_blk, wp), exl);
    // the prefix in front of each of this thread's groups -> samples[(base + first op of the group) >> 3]
    for (uint32_t gi = 0; gi < per && g0 + gi < ngroups; gi++) {
        const int ls = (int)((g0 + gi) * 8u) - (int)off;  // first op of the group, tile-local (< 0: the group began in the tile before)
        if (gi) {  // (rare) advance over the previous group
            const uint32_t a0 = (ls - 8) < 0 ? 0u : (uint32_t)(ls - 8);
            uint32_t slowc = pre.c.aux & AUX_CNT, ovf = pre.c.aux & AUX_OVF;
            uint32_t prev_code = a0 ? op_code(s_opw[a0 - 1]) : s_prev0;
            for (uint32_t j = a0; j < (uint32_t)ls; j++) {
                const uint32_t w = s_opw[j];
                const bool head = (s_head[j >> 5] >> (j & 31u)) & 1u;
                if (head) { pre.c = ctr_zero(); slowc = 0; ovf = 0; }
                const uint32_t code = op_code(w), n = op_len(w);
                slowc += ((n - 1u) >= (ACC_BIG - 1u)) | ((!head) & (code == prev_code));
                pre.c.aux = 0;
                ctr_add_op(pre.c, w);
                ovf |= pre.c.aux & AUX_OVF;
                prev_code = code;
            }
            pre.c.aux = ovf | (slowc & AUX_CNT);
        }
        if (ls < 0 || (uint32_t)ls >= total) continue;
        Ctr out = pre.c;
        if ((s_head[(uint32_t)ls >> 5] >> ((uint32_t)ls & 31u)) & 1u) out = ctr_zero();  // the group starts a record
        const uint64_t k = base + (uint32_t)ls;
        if (k & (SAMPLE - 1)) {  // sub-sample, absolute: the marker + the sticky overflow bit + the (saturated) slow-op count
            const uint32_t cntv = out.aux & AUX_CNT;
            out.aux = SUB_ABS | (out.aux & AUX_OVF) | (cntv >= SUB_ABS ? SUB_ABS - 1u : cntv);
        }
        uint4* dst = reinterpret_cast<uint4*>(samples + (k >> SUB_LOG2));
        const uint32_t* ow = reinterpret_cast<const uint32_t*>(&out);
        dst[0] = make_uint4(ow[0], ow[1], ow[2], ow[3]);
        dst[1] = make_uint4(ow[4], ow[5], ow[6], ow[7]);
        dst[2] = make_uint4(ow[8], ow[9], ow[10], ow[11]);
    }
}

// segmented exclusive scan of the block aggregates k_samples2<true> left (one block: the array is small — one 64-byte entry
// per 8192 ops), then every chunk sample that is not complete yet gets its block's prefix added
__global__ void __launch_bounds__(1024)
k_blk_scan(const uint64_t* __restrict__ n_ops_dev, const ScanPayload* __restrict__ blk_agg, ScanPayload* __restrict__ blk_pre) {
    __shared__ SegVal s_w[32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint64_t n_ops = *n_ops_dev;
    const uint64_t n_blk = (n_ops + SMP_OPS - 1) / SMP_OPS;
    const uint64_t per = (n_blk + 1023) / 1024;  // consecutive entries per thread
    const uint64_t lo = (uint64_t)tid * per, hi = (lo + per < n_blk) ? lo + per : n_blk;
    SegVal mine = seg_identity();
    for (uint64_t i = lo; i < hi; i++) mine = seg_combine(mine, payload_load(&blk_agg[i]));
    SegVal inc = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const SegVal y = seg_shfl(inc, (lane - d) & 31);
        if (lane >= d) inc = seg_combine(y, inc);
    }
    if (lane == 31) s_w[warp] = inc;
    SegVal exl = seg_shfl(inc, (lane - 1) & 31);
    if (lane == 0) exl = seg_identity();
    __syncthreads();
    SegVal wpre = seg_identity();
    for (int k = 0; k < warp; k++) wpre = seg_combine(wpre, s_w[k]);
    SegVal run = seg_combine(wpre, exl);
    for (uint64_t i = lo; i < hi; i++) {
        payload_store(&blk_pre[i], run);
        run = seg_combine(run, payload_load(&blk_agg[i]));
    }
}
__global__ void __launch_bounds__(256)
k_smp_fix(const uint64_t* __restrict__ n_ops_dev, const ScanPayload* __restrict__ blk_pre, Ctr* __restrict__ samples) {
    const uint64_t chunk = (uint64_t)blockIdx.x * 256 + threadIdx.x;
    const uint64_t n_ops = *n_ops_dev;
    if ((chunk << SAMPLE_LOG2) >= n_ops) return;
    uint4* p = reinterpret_cast<uint4*>(samples + chunk * SUBS);
    uint4 c = p[2];  // words 8..11: IEV DEV TXT aux
    if (c.w & SUB_ABS) {  // complete already: only the marker goes
        c.w &= ~SUB_ABS;
        p[2] = c;
        return;
    }
    const SegVal pre = payload_load(&blk_pre[chunk / SMP_THREADS]);  // (the same 64 bytes for 256 consecutive chunks)
    Ctr v;
    uint32_t* w = reinterpret_cast<uint32_t*>(&v);
    const uint4 a = p[0], b2 = p[1];
    w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w; w[4] = b2.x; w[5] = b2.y; w[6] = b2.z; w[7] = b2.w;
    w[8] = c.x; w[9] = c.y; w[10] = c.z; w[11] = c.w;
    Ctr r = pre.c;
    ctr_add(r, v);
    const uint32_t* o = reinterpret_cast<const uint32_t*>(&r);
    p[0] = make_uint4(o[0], o[1], o[2], o[3]);
    p[1] = make_uint4(o[4], o[5], o[6], o[7]);
    p[2] = make_uint4(o[8], o[9], o[10], o[11]);
}

// ------------------------------------------------------------------------------------------------
// K3  per-record preparation
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ Ctr ctr_range(const OpsView& v, const RecInfo& r, uint64_t a, uint64_t b, ClassAcc& acc) {  // ops [a, b), b > a
    Ctr hi = ctr_before(v, r, b - 1, acc);
    ctr_add_op(hi, v.op(b - 1));
    const Ctr lo = ctr_before(v, r, a, acc);
    Ctr d = hi;
    ctr_sub(d, lo);
    d.aux = hi.aux;  // flags/slow count of the whole prefix (conservative)
    return d;
}

__device__ __forceinline__ void write_stats(const StatsDev& st, uint64_t i, uint32_t equal, uint32_t diff, uint32_t ins, uint32_t del,
                                            uint32_t ins_ev, uint32_t del_ev, uint32_t matches) {
    st.equal[i] = equal; st.diff[i] = diff; st.ins[i] = ins; st.del[i] = del;
    st.ins_ev[i] = ins_ev; st.del_ev[i] = del_ev; st.matches[i] = matches;
    // bamstats.rs:138-142 — f32: (100.0 * equal as f32) / (u32 sum) as f32 ; IEEE mul + div, no contraction
    const float num = __fmul_rn(100.0f, __uint2float_rn(equal));
    st.id_a[i] = __fdiv_rn(num, __uint2float_rn(equal + diff + del + ins));
    st.id_e[i] = __fdiv_rn(num, __uint2float_rn(equal + diff + del_ev + ins_ev));
    st.id_m[i] = __fdiv_rn(num, __uint2float_rn(equal + diff));
}

// mode 0  rb stats --paf (after the scan): integrity + counters of the record as read
// mode 1  liftover phase A (needs ops only, runs BEFORE the scan): indel strip + window join -> RecInfo, pair_cnt
// mode 2  liftover phase B (after the scan): integrity, RF_SLOW, counters of the stripped op range
__global__ void __launch_bounds__(128)
k_rec_prep(int mode, RecInput in, const uint64_t* __restrict__ op_off, const uint32_t* __restrict__ ops,
           const Ctr* __restrict__ samples, WinView win, RecInfo* __restrict__ recs, uint32_t* __restrict__ pair_cnt, StatsDev st,
           ErrSlots err) {
    __shared__ uint32_t s_acc[9 * 128];
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= in.n_rec) return;
    OpsView v;
    v.ops = ops; v.samples = samples;
    ClassAcc acc;
    acc.sum = s_acc + threadIdx.x; acc.stride = 128;
    RecInfo ri;
    if (mode == 2) {
        ri = recs[r];
    } else {
        ri.op_first = op_off[r]; ri.op_end = op_off[r + 1];
        ri.eo0 = ri.op_first; ri.eo1 = ri.op_end;
        ri.t_st = in.t_st[r]; ri.t_en = in.t_en[r];
        ri.q_st0 = in.q_st[r]; ri.q_en0 = in.q_en[r];
        ri.q_st = ri.q_st0; ri.q_en = ri.q_en0;
        ri.q_len = in.q_len[r]; ri.t_len = in.t_len[r]; ri.mapq = in.mapq[r];
        ri.q_name = in.q_id[r]; ri.t_name = in.t_id[r];
        ri.flags = (in.strand[r] == '-') ? RF_MINUS : 0u;
        ri.a_lead = 0; ri.n_lead = 0; ri.n_trail = 0; ri.id_len = 0; ri.wlo = 0; ri.whi = 0; ri.lead_txt = 0;
        ri.text_off = in.cigar_off[r]; ri.pad2 = 0;
        ri.line_const = line_const_bytes(ri, (uint32_t)(in.names_off[ri.q_name + 1] - in.names_off[ri.q_name]),
                                         (uint32_t)(in.names_off[ri.t_name + 1] - in.names_off[ri.t_name]));
        ri.tot = ctr_zero();
    }

    if (mode == 1) {
        const uint32_t e = strip_record(ops, ri);
        if (e != RE_OK) {
            report(err.rec, r, e);
            pair_cnt[r] = 0;
            recs[r] = ri;
            return;
        }
        // join: windows of this contig with en > t_st && st < t_en (paf.rs:622-627, on stripped coordinates)
        uint32_t cnt = 0;
        if (win.st != nullptr && !win.general) {
            const uint32_t clo = win.cont_lo[ri.t_name], chi = win.cont_hi[ri.t_name];
            uint32_t lo = clo, hi = chi;
            while (lo < hi) {  // first window whose running max of `en` exceeds t_st
                const uint32_t mid = lo + ((hi - lo) >> 1);
                if (win.en_pm[mid] > ri.t_st) hi = mid; else lo = mid + 1;
            }
            ri.wlo = lo;
            hi = chi;
            while (lo < hi) {  // first window with st >= t_en
                const uint32_t mid = lo + ((hi - lo) >> 1);
                if (win.st[mid] >= ri.t_en) hi = mid; else lo = mid + 1;
            }
            ri.whi = lo;
            cnt = ri.whi - ri.wlo;
        }
        pair_cnt[r] = cnt;
        recs[r] = ri;
        return;
    }

    // integrity at load (paf.rs:70): spans of the UNSTRIPPED record against the full CIGAR
    const uint64_t t_en_in = (mode == 2) ? in.t_en[r] : ri.t_en;
    Ctr full = ctr_zero();
    if (ri.op_end > ri.op_first) full = ctr_range(v, ri, ri.op_first, ri.op_end, acc);
    if (full.aux & 0x80000000u) report(err.rec, r, RE_UNSUPPORTED);
    uint64_t span_t = full.T, span_q = full.Q;
    if (mode == 0 && in.no_text) {
        // `rb invert`: the reference checks the record as read, before the swap (paf.rs:70) — undo the I<->D exchange
        // (N and S keep their side, so the swapped sums are not simply the other span)
        const uint64_t both = (uint64_t)full.M + full.EQ + full.X;
        const uint64_t n_skip = (uint64_t)full.T - both - full.D, n_clip = (uint64_t)full.Q - both - full.I;  // N, S bases
        span_t = both + full.I + n_skip;  // what the file's CIGAR spends on the file's target (= our query columns): M = X D N
        span_q = both + full.D + n_clip;  // ... and on the file's query: M = X I S
        if (span_t != ri.q_en0 - ri.q_st0 || span_q != t_en_in - ri.t_st) report(err.rec, r, RE_INTEGRITY);
    } else if (span_t != t_en_in - ri.t_st || span_q != ri.q_en0 - ri.q_st0) {
        report(err.rec, r, RE_INTEGRITY);
    }
    if (full.aux & AUX_CNT) ri.flags |= RF_SLOW;
    if (!in.no_text && (uint64_t)full.TXT == in.cigar_off[r + 1] - in.cigar_off[r]) ri.flags |= RF_CANON;  // no op is spelled with leading zeros
    if (ri.op_end > ri.op_first) {  // the sampled count stops at the last chunk boundary: look at the tail ops too
        const uint64_t base = ((ri.op_end - 1) >> SAMPLE_LOG2) << SAMPLE_LOG2;
        for (uint64_t k = base > ri.op_first ? base : ri.op_first; k < ri.op_end; k++) {
            const uint32_t w = ops[k];
            if (op_len(w) == 0u || op_len(w) >= ACC_BIG || (k > ri.op_first && op_code(w) == op_code(ops[k - 1]))) ri.flags |= RF_SLOW;
        }
    }
    if (mode == 0) {  // rb stats --paf: counters of the record as read (bamstats.rs:91-105)
        ri.tot = full;
        write_stats(st, r, full.EQ, full.X + full.M, full.I, full.D, full.IEV, full.DEV, full.M);
        recs[r] = ri;
        return;
    }
    ri.tot = (ri.eo0 == ri.op_first && ri.eo1 == ri.op_end) ? full : ctr_range(v, ri, ri.eo0, ri.eo1, acc);
    recs[r] = ri;
}

// `rb invert` (main.rs:176-182): one row per record, the whole (already inverted) CIGAR, nothing stripped or merged.
// Fills what k_lift would have: PairRes, line lengths, the identity pair list and the per-block plans of the serialiser.
__global__ void __launch_bounds__(128)
k_whole_rows(uint32_t n_rec, const RecInfo* __restrict__ recs, PairRes* __restrict__ res, uint32_t* __restrict__ line_len,
             uint64_t* __restrict__ pair_off, LiftPlan* __restrict__ plans) {
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r == 0) pair_off[n_rec] = n_rec;
    if (r >= n_rec) return;
    const RecInfo ri = recs[r];
    PairRes pr;
    pair_clear(pr);
    pair_early(ri, pr);
    pr.kind = PK_WHOLE;
    if (ri.op_end <= ri.op_first) { pr.si = 1; pr.ei = 0; pr.cg_bytes = 0; pr.mid_len = 0; }  // "cg:Z:" with nothing behind it
    res[r] = pr;
    line_len[r] = ri.line_const + line_var_bytes(pr, 0u);
    pair_off[r] = r;
    if (r % LIFT_THREADS == 0) {
        LiftPlan pl;
        pl.k0 = r; pl.uniform = 0u; pl.c_lo = pl.c_hi = ~0ull;
        plans[r / LIFT_THREADS] = pl;
    }
}

// Window table checks (the host never walks the 3 M-row table): bit 0 = not sorted by (t_id, st) or t_id out of
// range, bit 1 = general layout (inside a contig `en` or the BED row number decreases somewhere: nested rows, or a file
// order that is not the sorted order) -> the brute-force join keeps the reference's emission order (Q5).
__global__ void __launch_bounds__(256)
k_win_check(const uint32_t* __restrict__ t_id, const uint64_t* __restrict__ st, const uint64_t* __restrict__ en,
            const uint32_t* __restrict__ row, uint32_t n_win, uint32_t n_names, uint32_t* flags) {
    uint32_t f = 0;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_win; i += gridDim.x * blockDim.x) {
        const uint32_t t = t_id[i];
        if (t >= n_names) f |= 1u;
        if (i) {
            const uint32_t tp = t_id[i - 1];
            if (t < tp) f |= 1u;
            if (t == tp) {
                if (st[i] < st[i - 1]) f |= 1u;
                if (en[i] < en[i - 1] || row[i] < row[i - 1]) f |= 2u;
            }
        }
    }
    f = __reduce_or_sync(0xffffffffu, f);
    if ((threadIdx.x & 31) == 0 && f) atomicOr(flags, f);
}

// pair offsets in emission order: exclusive scan of pair_cnt[rec_order[k]] (single block; n_rec is small)
__global__ void __launch_bounds__(1024) k_pair_scan(const uint32_t* __restrict__ pair_cnt, const uint32_t* __restrict__ rec_order,
                                                    uint32_t n_rec, uint64_t* __restrict__ pair_off) {
    __shared__ unsigned long long s_warp[32];
    __shared__ unsigned long long s_carry;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < n_rec; base += 1024) {
        const uint32_t k = base + tid;
        const unsigned long long x = (k < n_rec) ? pair_cnt[rec_order[k]] : 0ull;
        unsigned long long inc = x;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned long long t = __shfl_up_sync(0xffffffffu, inc, d);
            if (lane >= d) inc += t;
        }
        if (lane == 31) s_warp[warp] = inc;
        __syncthreads();
        unsigned long long wpre = 0, tot = 0;
        for (int j = 0; j < 32; j++) {
            const unsigned long long t = s_warp[j];
            if (j < warp) wpre += t;
            tot += t;
        }
        const unsigned long long carry = s_carry;
        if (k < n_rec) pair_off[k] = carry + wpre + inc - x;
        __syncthreads();
        if (tid == 0) s_carry = carry + tot;
        __syncthreads();
    }
    if (tid == 0) pair_off[n_rec] = s_carry;
}

// general path: cartesian product + overlap filter in BED file order (liftover.rs:123-127); block per record
__global__ void __launch_bounds__(256) k_pair_count_bf(const RecInfo* __restrict__ recs, uint32_t n_rec, WinView win, uint32_t* pair_cnt) {
    const uint32_t r = blockIdx.x;
    if (r >= n_rec) return;
    const RecInfo& ri = recs[r];
    const uint32_t clo = win.cont_lo[ri.t_name], chi = win.cont_hi[ri.t_name];
    uint32_t cnt = 0;
    for (uint32_t w = clo + threadIdx.x; w < chi; w += blockDim.x) cnt += (ri.t_en > win.st[w] && ri.t_st < win.en[w]);
    __shared__ uint32_t s[8];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, d);
    if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
        for (int k = 0; k < 8; k++) t += s[k];
        pair_cnt[r] = t;
    }
}
__global__ void __launch_bounds__(256) k_pair_fill_bf(const RecInfo* __restrict__ recs, const uint32_t* __restrict__ rec_rank,
                                                     uint32_t n_rec, WinView win, const uint64_t* __restrict__ pair_off,
                                                     uint32_t* __restrict__ pair_win) {
    const uint32_t r = blockIdx.x;
    if (r >= n_rec) return;
    const RecInfo& ri = recs[r];
    const uint32_t clo = win.cont_lo[ri.t_name], chi = win.cont_hi[ri.t_name];
    __shared__ uint32_t s_w[8];
    __shared__ uint32_t s_base;
    if (threadIdx.x == 0) s_base = 0;
    __syncthreads();
    const uint64_t out0 = pair_off[rec_rank[r]];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (uint32_t w0 = clo; w0 < chi; w0 += blockDim.x) {
        const uint32_t w = w0 + threadIdx.x;
        const bool hit = (w < chi) && (ri.t_en > win.st[w] && ri.t_st < win.en[w]);
        const unsigned m = __ballot_sync(0xffffffffu, hit);
        if (lane == 0) s_w[warp] = __popc(m);
        __syncthreads();
        uint32_t pre = s_base, tot = 0;
        for (int k = 0; k < 8; k++) {
            if (k < warp) pre += s_w[k];
            tot += s_w[k];
        }
        if (hit) pair_win[out0 + pre + __popc(m & ((1u << lane) - 1u))] = w;
        __syncthreads();
        if (threadIdx.x == 0) s_base += tot;
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------
// K4  lift: one thread per (window, record) pair
// ------------------------------------------------------------------------------------------------
// bytes of Region.id of window w: BED column 4, else "{chrom}:{st+1}-{en}" (bed.rs:150-153)
__device__ __forceinline__ uint32_t win_id_len(const WinView& win, uint32_t w, uint32_t t_name_len, uint64_t w_st, uint64_t w_en) {
    if (win.ids_off) return (uint32_t)(win.ids_off[w + 1] - win.ids_off[w]);
    return t_name_len + 1u + ndigits64(w_st + 1) + 1u + ndigits64(w_en);
}
__device__ __forceinline__ uint32_t rank_of_pair(const uint64_t* __restrict__ pair_off, uint32_t n_rec, uint64_t p) {
    uint32_t lo = 0, hi = n_rec;  // largest k with pair_off[k] <= p
    while (hi - lo > 1) {
        const uint32_t mid = lo + ((hi - lo) >> 1);
        if (pair_off[mid] <= p) lo = mid; else hi = mid;
    }
    return lo;
}

// One thread per block of LIFT_THREADS consecutive pairs: which record the block belongs to (if it is a single one)
// and which run of 32-op chunks its pairs touch.  Doing the searches here, all blocks in parallel, keeps them out of
// the prologue of k_lift / k_serialise where a whole block would wait for one thread's chain of dependent loads.
__global__ void __launch_bounds__(128)
k_lift_plan(uint64_t n_pairs, uint32_t n_blocks, const uint64_t* __restrict__ pair_off, const uint32_t* __restrict__ rec_order,
            uint32_t n_rec, const RecInfo* __restrict__ recs, const Ctr* __restrict__ samples, WinView win, LiftPlan* __restrict__ plans,
            uint32_t mark_fast) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n_blocks) return;
    const uint64_t p0 = (uint64_t)b * LIFT_THREADS;
    const uint64_t plast = (p0 + LIFT_THREADS <= n_pairs ? p0 + LIFT_THREADS : n_pairs) - 1;
    LiftPlan pl;
    pl.k0 = rank_of_pair(pair_off, n_rec, p0);
    pl.uniform = (pl.k0 == rank_of_pair(pair_off, n_rec, plast)) ? (uint32_t)PLAN_UNIFORM : 0u;
    pl.c_lo = pl.c_hi = ~0ull;
    if (pl.uniform && win.pair_win == nullptr) {
        const RecInfo& R = recs[rec_order[pl.k0]];
        if (R.op_end > R.op_first && R.t_en > R.t_st) {
            OpsView v;
            v.ops = nullptr; v.samples = samples;
            const uint64_t pbase = pair_off[pl.k0];
            const uint64_t t_st = R.t_st, t_en = R.t_en;
            const uint64_t st = win.st[R.wlo + (uint32_t)(p0 - pbase)];     // start boundary of the block's first pair
            const uint64_t en = win.en[R.wlo + (uint32_t)(plast - pbase)];  // end boundary of its last pair
            pl.c_lo = chunk_of(v, R, (uint32_t)((st > t_st ? st : t_st) - t_st));
            pl.c_hi = chunk_of(v, R, (uint32_t)((en < t_en ? en : t_en) - 1 - t_st));
            // the op run and its samples fit k_emit's staging area and the record needs no special care: k_emit lifts the block
            if (mark_fast && pl.c_hi >= pl.c_lo && pl.c_hi - pl.c_lo < (uint64_t)LIFT_CCAP && !(R.flags & RF_SLOW)) pl.uniform |= PLAN_FAST;
        }
    }
    plans[b] = pl;
}

// ---- chained boundaries (tiling windows) ----
// On a tiling BED the end boundary of window j (last base, position pe) and the start boundary of window j + 1
// (position pe + 1) are neighbours: the start lookup of a pair is one step past the end lookup its left neighbour
// just finished, so it is derived from that instead of being searched for again.
struct ChainSlot {  // what lane 31 of a warp leaves for lane 0 of the next one
    uint64_t i;
    uint32_t o, pe, ok, pad;
    Ctr c;
};
// (i, o, counters before i) of target position p  ->  the same for p + 1
__device__ __forceinline__ bool advance_one(const OpsView& v, const RecInfo& r, uint64_t i, uint32_t o, const Ctr& before, uint64_t& ni,
                                            uint32_t& no, Ctr& nbefore) {
    const uint32_t w = v.op(i);
    if (o + 1u < op_len(w)) { ni = i; no = o + 1u; nbefore = before; return true; }
    Ctr c = before;
    ctr_add_op(c, w);
    uint64_t k = i + 1;
    for (; k < r.op_end; k++) {  // the next reference-consuming op of non-zero length (same condition as find_op)
        const uint32_t w2 = v.op(k);
        if (is_ref(op_code(w2)) && op_len(w2) > 0u) break;
        ctr_add_op(c, w2);
    }
    if (k >= r.op_end) return false;
    ni = k; no = 0u; nbefore = c;
    return true;
}
// lift_pair (lift_core.cuh) with the END boundary looked up first and the START boundary chained to the left
// neighbour's END where the two are adjacent positions of the same record (`chain` is block-uniform: every pair of the
// block belongs to one record, windows consecutive).  Same results as lift_pair by construction: find_op is a pure
// function of (record, position), and the failure checks are applied in lift_pair's order.
__device__ __forceinline__ uint32_t lift_pair_chain(const OpsView& v, const RecInfo& r, uint64_t w_st, uint64_t w_en, int policy,
                                                    bool enabled, bool chain, PairRes& out, ClassAcc& acc, ChainSlot* s_x) {
    constexpr unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t status = LIFT_OK;
    bool live = enabled;
    pair_clear(out);
    if (live && r.t_st > w_st && r.t_en < w_en) {
        pair_early(r, out);
        live = false;
    } else if (live && r.t_en <= r.t_st) {
        status = LIFT_ERR_NOT_FOUND;
        live = false;
    }
    const uint32_t ps = live ? (uint32_t)((w_st > r.t_st ? w_st : r.t_st) - r.t_st) : 0u;
    const uint32_t pe = live ? (uint32_t)((w_en < r.t_en ? w_en : r.t_en) - 1 - r.t_st) : 0u;

    uint64_t ie = 0; uint32_t oe = 0; Ctr be = ctr_zero();
    const bool fe = find_op(v, r, live, pe, ie, oe, be, acc);

    // hand (ie, oe, be) to the right neighbour
    bool derive = false;
    uint64_t pi = 0; uint32_t po = 0; Ctr pb = ctr_zero();
    if (chain) {
        const uint32_t ok = (live && fe) ? 1u : 0u;
        if (lane == 31) {
            ChainSlot& x = s_x[warp];
            x.i = ie; x.o = oe; x.pe = pe; x.ok = ok; x.c = be;
        }
        __syncthreads();
        uint32_t p_ok = __shfl_up_sync(FULL, ok, 1), p_pe = __shfl_up_sync(FULL, pe, 1);
        po = __shfl_up_sync(FULL, oe, 1);
        pi = __shfl_up_sync(FULL, ie, 1);
        uint32_t* dw = reinterpret_cast<uint32_t*>(&pb);
        const uint32_t* sw = reinterpret_cast<const uint32_t*>(&be);
#pragma unroll
        for (int t = 0; t < 12; t++) dw[t] = __shfl_up_sync(FULL, sw[t], 1);
        if (lane == 0) {
            p_ok = 0u;
            if (warp > 0) {
                const ChainSlot& x = s_x[warp - 1];
                p_ok = x.ok; p_pe = x.pe; po = x.o; pi = x.i; pb = x.c;
            }
        }
        derive = live && p_ok && ps == p_pe + 1u;
    }
    uint64_t i = 0; uint32_t o = 0; Ctr before = ctr_zero();
    bool fs = false;
    const bool search = live && !derive;
    if (__any_sync(FULL, search)) fs = find_op(v, r, search, ps, i, o, before, acc);
    if (derive) fs = advance_one(v, r, pi, po, pb, i, o, before);
    __syncwarp();
    if (!fs && live) { status = LIFT_ERR_NOT_FOUND; live = false; }
    uint64_t si = 0; uint32_t so = 0; Ctr cs = ctr_zero();
    if (live && !lift_start(v, r.eo1, r.a_lead, r.tot.A, policy, i, o, before, si, so, cs)) live = false;
    __syncwarp();
    if (live && !fe) { status = LIFT_ERR_NOT_FOUND; live = false; }
    if (live) {
        uint64_t ei; uint32_t eo; Ctr ce; uint32_t txt_before_ei;
        if (lift_end(v, r.eo0, ie, oe, be, ei, eo, ce, txt_before_ei))
            lift_finish(v, r, si, so, cs, op_len(v.op(si)), ei, eo, ce, txt_before_ei, out);
    }
    __syncwarp();
    return status;
}

// CTA = LIFT_THREADS consecutive pairs in emission order.  On the sorted-BED path the pairs of a block that belong
// to one record touch a contiguous run of ops (start of the first window .. end of the last one): that run and
// its samples are staged in shared memory once (coalesced), so the per-pair searches and <=7-op walks of
// lift_pair never leave the SM.  Blocks that straddle records, explicit pair lists (general path) and runs that
// do not fit fall back to global memory through the same OpsView accessor.
#ifndef RB_LIFT_MINB_WIDE
#define RB_LIFT_MINB_WIDE 8
#endif
// STAGE == false: the wide-window form.  No block of such a call fits the staging area (a block's pairs span tens of thousands of
// ops), so the 31 KB of staging arrays are left out and the register cap lowered: eight resident blocks instead of six for a
// kernel whose pairs each wait on a chain of dependent trips to L2 / HBM.
template <bool STAGE>
__global__ void __launch_bounds__(LIFT_THREADS, STAGE ? RB_LIFT_MINB : RB_LIFT_MINB_WIDE)
k_lift(uint64_t n_pairs, const uint64_t* __restrict__ pair_off, const uint32_t* __restrict__ rec_order, uint32_t n_rec,
       const RecInfo* __restrict__ recs, const uint32_t* __restrict__ ops, const Ctr* __restrict__ samples, WinView win,
       const uint64_t* __restrict__ names_off, int policy, const LiftPlan* __restrict__ plans, PairRes* __restrict__ res,
       uint32_t* __restrict__ line_len, ErrSlots err, uint32_t skip_fast) {
    __shared__ uint32_t s_acc[9 * LIFT_THREADS];
    __shared__ __align__(16) uint32_t s_ops[STAGE ? (LIFT_CCAP + 1) * SAMPLE : 4];
#if RB_LIFT_STAGE_SMP
    __shared__ __align__(16) Ctr s_smp[STAGE ? (LIFT_CCAP + 2) * SUBS : 1];
#endif
    __shared__ __align__(16) RecInfo s_rec;
#if RB_LIFT_CHAIN
    __shared__ __align__(16) ChainSlot s_chain[LIFT_THREADS / 32];
#endif
    __shared__ __align__(8) unsigned long long s_bar;
    const int tid = threadIdx.x;
    const uint64_t p0 = (uint64_t)blockIdx.x * LIFT_THREADS;
    const uint64_t p = p0 + tid;
    OpsView v;
    v.ops = ops; v.samples = samples;
    const LiftPlan pl = plans[blockIdx.x];
    if (skip_fast && (pl.uniform & PLAN_FAST)) return;  // k_emit lifts this block itself (block-uniform)
    const bool uniform = (pl.uniform & PLAN_UNIFORM) != 0;
    uint32_t r_blk = 0;
    bool staged = false;
    if (uniform) {  // block-uniform: the record and (if it fits) the op run + samples of the block go to shared memory
        r_blk = rec_order[pl.k0];
        static_assert(sizeof(RecInfo) % 16 == 0, "RecInfo is copied in 16-byte vectors");
        if (tid < (int)(sizeof(RecInfo) / 16)) reinterpret_cast<uint4*>(&s_rec)[tid] = reinterpret_cast<const uint4*>(&recs[r_blk])[tid];
        const uint64_t c_lo = pl.c_lo, c_hi = pl.c_hi;
        if (STAGE && c_lo != ~0ull && c_hi != ~0ull && c_hi >= c_lo && c_hi - c_lo < (uint64_t)LIFT_CCAP) {
            const uint64_t op_end = recs[r_blk].op_end;
            const uint64_t o_lo = c_lo << SAMPLE_LOG2;
            uint64_t o_hi = (c_hi + 2) << SAMPLE_LOG2;  // one extra chunk for the look-ahead of the slide rules
            if (o_hi > op_end) o_hi = op_end;
            // both runs are contiguous in HBM and 16-byte aligned (o_lo is a multiple of 32 ops): one thread hands them to
            // the bulk-copy engine, the block waits on the mbarrier — no per-thread load / store loop, everything in flight
            const uint32_t n_stage = (uint32_t)(o_hi - o_lo), n4 = n_stage >> 2;
            const uint64_t c_max = (op_end - 1) >> SAMPLE_LOG2;
            const uint64_t c_top = (c_hi + 1 <= c_max) ? c_hi + 1 : c_max;  // samples (+ sub-samples) of chunks [c_lo, c_top]
            const uint32_t smp_bytes = RB_LIFT_STAGE_SMP ? (uint32_t)((c_top - c_lo + 1) * SUBS * sizeof(Ctr)) : 0u;
            if (tid == 0) {
                mbar_init(&s_bar, 1);
                mbar_expect_tx(&s_bar, n4 * 16u + smp_bytes);
                if (n4) bulk_g2s(s_ops, ops + o_lo, n4 * 16u, &s_bar);
#if RB_LIFT_STAGE_SMP
                bulk_g2s(s_smp, samples + c_lo * SUBS, smp_bytes, &s_bar);
#endif
            }
            for (uint32_t k = (n4 << 2) + tid; k < n_stage; k += LIFT_THREADS) s_ops[k] = ops[o_lo + k];  // the (< 4 op) tail
#if RB_LIFT_STAGE_SMP
            v.s_smp = s_smp; v.sc_lo = c_lo; v.sc_hi = c_top + 1;
#endif
            v.s_ops = s_ops; v.so_lo = o_lo; v.so_hi = o_hi;
            staged = true;
        }
    }
    const bool in_range = p < n_pairs;  // (no early return: the chained lookup below has a block barrier)
    const uint64_t pc = in_range ? p : n_pairs - 1;
    ClassAcc acc;
    acc.sum = s_acc + tid; acc.stride = LIFT_THREADS;
    uint32_t k, r;
    if (uniform) {  // the block's record sits in shared memory: no per-thread search, no per-thread 208-byte load
        k = pl.k0; r = r_blk;
    } else {
        k = rank_of_pair(pair_off, n_rec, pc);
        r = rec_order[k];
    }
    // this pair's window: loaded while the bulk copies above are still in flight
    const uint64_t j = pc - pair_off[k];
    const uint32_t w = win.pair_win ? win.pair_win[pc] : (recs[r].wlo + (uint32_t)j);
    const uint64_t w_st = win.st[w], w_en = win.en[w];
    if (uniform) {
        __syncthreads();  // s_rec, the tail ops and the mbarrier's initialisation are visible to everybody
        if (staged) mbar_wait(&s_bar, 0);
    }
    const RecInfo& ri = uniform ? s_rec : recs[r];
    PairRes pr;
    uint32_t len = 0;
    // the brute-force / nested-window candidates can be a superset; break-paf pieces of zero length are never built
    const bool overlaps = in_range && ri.t_en > w_st && ri.t_st < w_en && !(win.from_record && w_en <= w_st);
#if RB_LIFT_CHAIN
    const bool chain = uniform && win.pair_win == nullptr;  // block-uniform
    const uint32_t e = lift_pair_chain(v, ri, w_st, w_en, policy, overlaps, chain, pr, acc, s_chain);
#else
    const uint32_t e = lift_pair(v, ri, w_st, w_en, policy, overlaps, pr, acc);
#endif
    __syncwarp();
    if (!in_range) return;
    if (e != LIFT_OK) { report(err.rec, r, RE_INDEX_PANIC); pr.kind = PK_DROP; }
    if (pr.kind != PK_DROP) {
        uint32_t idl = ri.id_len;  // early rows and break-paf pieces carry their record's id
        if (pr.kind != PK_EARLY && !win.from_record) {
            const uint32_t tn = win.ids_off ? 0u : (uint32_t)(names_off[ri.t_name + 1] - names_off[ri.t_name]);
            idl = win_id_len(win, w, tn, w_st, w_en);
        }
        len = ri.line_const + line_var_bytes(pr, idl);
    }
    res[p] = pr;
    line_len[p] = len;
}

// K4' (fast path): joins the two half results k_scan_lift left for each pair -> PairRes + line size
__global__ void __launch_bounds__(128)
k_combine(uint64_t n_pairs, const uint64_t* __restrict__ pair_off, const uint32_t* __restrict__ rec_order, uint32_t n_rec,
          const RecInfo* __restrict__ recs, const uint32_t* __restrict__ ops, WinView win, const uint64_t* __restrict__ names_off,
          const HalfS* __restrict__ hs, const HalfE* __restrict__ he, PairRes* __restrict__ res, uint32_t* __restrict__ line_len,
          ErrSlots err) {
    const uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_pairs) return;
    const uint32_t k = rank_of_pair(pair_off, n_rec, p);
    const uint32_t r = rec_order[k];
    const RecInfo ri = recs[r];
    const uint32_t w = ri.wlo + (uint32_t)(p - pair_off[k]);
    const uint64_t w_st = win.st[w], w_en = win.en[w];
    HalfS a;
    HalfE b;
    {
        const uint4* pa = reinterpret_cast<const uint4*>(hs + p);
        const uint4* pb = reinterpret_cast<const uint4*>(he + p);
        uint4* qa = reinterpret_cast<uint4*>(&a);
        uint4* qb = reinterpret_cast<uint4*>(&b);
#pragma unroll
        for (int i = 0; i < 4; i++) { qa[i] = ld_nc_v4(pa + i); qb[i] = ld_nc_v4(pb + i); }
    }
    OpsView v;
    v.ops = ops; v.samples = nullptr;
    PairRes pr;
    uint32_t len = 0;
    const uint32_t e = combine_pair(v, ri, w_st, w_en, a, b, pr);
    if (e != LIFT_OK) { report(err.rec, r, RE_INDEX_PANIC); pr.kind = PK_DROP; }
    if (pr.kind != PK_DROP) {
        uint32_t idl = ri.id_len;  // early rows and break-paf pieces carry their record's id
        if (pr.kind != PK_EARLY && !win.from_record) {
            const uint32_t tn = win.ids_off ? 0u : (uint32_t)(names_off[ri.t_name + 1] - names_off[ri.t_name]);
            idl = win_id_len(win, w, tn, w_st, w_en);
        }
        len = ri.line_const + line_var_bytes(pr, idl);
    }
    res[p] = pr;
    line_len[p] = len;
}

// ------------------------------------------------------------------------------------------------
// exclusive scan of line sizes and of valid-row flags (decoupled look-back, 16-byte payload)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ ulonglong2 lookback_2u64(uint32_t* state, ulonglong2* agg, ulonglong2* pre, uint64_t b, ulonglong2 mine) {
    const int lane = threadIdx.x & 31;
    ulonglong2 acc = make_ulonglong2(0, 0);
    if (b == 0) {
        if (lane == 0) {
            pre[0] = mine;
            __threadfence();
            atomicExch(&state[0], 2u);
        }
        return acc;
    }
    if (lane == 0) {
        agg[b] = mine;
        __threadfence();
        atomicExch(&state[b], 1u);
    }
    long long look = (long long)b - 1;
    for (;;) {
        const long long idx = look - lane;
        uint32_t st = 2u;
        ulonglong2 x = make_ulonglong2(0, 0);
        if (idx >= 0) {
            do { st = ld_volatile_u32(&state[idx]); } while (st == 0);
            __threadfence();
            const uint4 raw = ld_cg_v4(st == 2u ? &pre[idx] : &agg[idx]);
            x.x = ((unsigned long long)raw.y << 32) | raw.x;
            x.y = ((unsigned long long)raw.w << 32) | raw.z;
        }
        const unsigned pm = __ballot_sync(0xffffffffu, st == 2u);
        const int first = pm ? (__ffs(pm) - 1) : 32;
        if (lane > first) x = make_ulonglong2(0, 0);
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            x.x += __shfl_xor_sync(0xffffffffu, x.x, d);
            x.y += __shfl_xor_sync(0xffffffffu, x.y, d);
        }
        acc.x += x.x; acc.y += x.y;
        if (pm) break;
        look -= 32;
        if (look < 0) break;
    }
    if (lane == 0) {
        pre[b] = make_ulonglong2(acc.x + mine.x, acc.y + mine.y);
        __threadfence();
        atomicExch(&state[b], 2u);
    }
    return acc;
}

constexpr int LNS_ITEMS = 16;                       // items per thread and tile
constexpr int LNS_TILE = LNS_THREADS * LNS_ITEMS;   // 4096 items
// A few hundred blocks, each owning a contiguous span of whole tiles: pass 1 reduces the span (coalesced), one
// decoupled look-back over <= LNS_MAX_BLOCKS predecessors gives the span's prefix, pass 2 scans the span tile by tile
// with a running carry.  (One tile per block meant ~800 chained look-backs at 3 M items: the kernel was pure latency.)
constexpr int LNS_MAX_BLOCKS = 296;
__global__ void __launch_bounds__(LNS_THREADS)
k_scan_lines(const uint32_t* __restrict__ line_len, uint64_t n, uint64_t span, uint64_t* __restrict__ line_off,
             uint64_t* __restrict__ out_idx, uint32_t* blk_state, ulonglong2* blk_agg, ulonglong2* blk_pre, unsigned int* ticket) {
    __shared__ ulonglong2 s_warp[LNS_THREADS / 32];
    __shared__ ulonglong2 s_blk;
    __shared__ unsigned int s_b;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_b = atomicAdd(ticket, 1u);
    __syncthreads();
    const uint64_t b = s_b;
    const uint64_t lo = b * span, hi = (lo + span < n) ? lo + span : n;
    if (n == 0) {
        if (b == 0 && tid == 0) { line_off[0] = 0; out_idx[0] = 0; }
        return;
    }
    // ---- pass 1: aggregate of the span ----
    unsigned long long sb = 0, sc = 0;
    for (uint64_t i = lo + tid; i < hi; i += LNS_THREADS) {
        const uint32_t x = line_len[i];
        sb += x;
        sc += (x != 0u);
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        sb += __shfl_xor_sync(0xffffffffu, sb, d);
        sc += __shfl_xor_sync(0xffffffffu, sc, d);
    }
    if (lane == 0) s_warp[warp] = make_ulonglong2(sb, sc);
    __syncthreads();
    if (warp == 0) {
        unsigned long long tb = 0, tc = 0;
#pragma unroll
        for (int k = 0; k < LNS_THREADS / 32; k++) { tb += s_warp[k].x; tc += s_warp[k].y; }
        const ulonglong2 ex = lookback_2u64(blk_state, blk_agg, blk_pre, b, make_ulonglong2(tb, tc));
        if (lane == 0) s_blk = ex;
    }
    __syncthreads();
    unsigned long long base_b = s_blk.x, base_c = s_blk.y;
    // ---- pass 2: rows of LNS_THREADS consecutive items (coalesced loads and stores), one block scan per row ----
    for (uint64_t r0 = lo; r0 < hi; r0 += LNS_THREADS) {
        const uint64_t i = r0 + tid;
        const uint32_t x = (i < hi) ? line_len[i] : 0u;
        unsigned long long ib = x, ic = (x != 0u);
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned long long ub = __shfl_up_sync(0xffffffffu, ib, d), uc = __shfl_up_sync(0xffffffffu, ic, d);
            if (lane >= d) { ib += ub; ic += uc; }
        }
        __syncthreads();  // s_warp is reused from the previous row / pass 1
        if (lane == 31) s_warp[warp] = make_ulonglong2(ib, ic);
        __syncthreads();
        unsigned long long wb = 0, wc = 0, allb = 0, allc = 0;
#pragma unroll
        for (int k = 0; k < LNS_THREADS / 32; k++) {
            const ulonglong2 t = s_warp[k];
            if (k < warp) { wb += t.x; wc += t.y; }
            allb += t.x; allc += t.y;
        }
        if (i < hi) { line_off[i] = base_b + wb + ib - x; out_idx[i] = base_c + wc + ic - (x != 0u); }
        base_b += allb; base_c += allc;
    }
    // the block whose span ends the array also writes the totals at index n
    if (hi == n && lo < n && tid == 0) { line_off[n] = base_b; out_idx[n] = base_c; }
}

// ------------------------------------------------------------------------------------------------
// K5  serialiser
// ------------------------------------------------------------------------------------------------
template <class P>
__device__ __forceinline__ P put_op(P p, uint32_t len, uint32_t code) {
    p = put_u32(p, len);
    *p = (uint8_t)char_of_code(code);
    return p + 1;
}

struct SerArgs {
    const RecInfo* recs;
    OpsView v;
    WinView win;
    const uint64_t* names_off;
    const uint8_t* names;
    const uint8_t* text;  // the input CIGAR text (device copy)
};

// "_TO.<leading ops>.<trailing ops, last first>" (paf.rs:726-732)
template <class P>
__device__ __forceinline__ P put_strip_id(P p, const RecInfo& ri, const OpsView& v) {
    *p++ = '_'; *p++ = 'T'; *p++ = 'O'; *p++ = '.';
    for (uint64_t k = ri.op_first; k < ri.eo0; k++) p = put_op(p, op_len(v.op(k)), op_code(v.op(k)));
    *p++ = '.';
    for (uint64_t k = ri.op_end; k > ri.eo1; k--) p = put_op(p, op_len(v.op(k - 1)), op_code(v.op(k - 1)));
    return p;
}

// the 12 columns + "id:Z:..." + "\tcg:Z:" (paf.rs:923-943), sequential
template <class P>
__device__ __forceinline__ P put_header(P p, const SerArgs& a, const RecInfo& ri, const PairRes& pr, uint32_t w) {
    p = put_bytes(p, a.names + a.names_off[ri.q_name], (uint32_t)(a.names_off[ri.q_name + 1] - a.names_off[ri.q_name]));
    *p++ = '\t'; p = put_u64(p, ri.q_len);
    *p++ = '\t'; p = put_u64(p, pr.q_st);
    *p++ = '\t'; p = put_u64(p, pr.q_en);
    *p++ = '\t'; *p++ = (ri.flags & RF_MINUS) ? '-' : '+';
    *p++ = '\t';
    p = put_bytes(p, a.names + a.names_off[ri.t_name], (uint32_t)(a.names_off[ri.t_name + 1] - a.names_off[ri.t_name]));
    *p++ = '\t'; p = put_u64(p, ri.t_len);
    *p++ = '\t'; p = put_u64(p, pr.t_st);
    *p++ = '\t'; p = put_u64(p, pr.t_en);
    *p++ = '\t'; p = put_u32(p, pr.nmatch);
    *p++ = '\t'; p = put_u32(p, pr.aln_len);
    *p++ = '\t'; p = put_u64(p, ri.mapq);
    *p++ = '\t'; *p++ = 'i'; *p++ = 'd'; *p++ = ':'; *p++ = 'Z'; *p++ = ':';
    if (pr.kind == PK_EARLY || a.win.from_record) {
        if (ri.flags & RF_STRIPPED) p = put_strip_id(p, ri, a.v);
    } else {
        if (a.win.ids_off) {
            p = put_bytes(p, a.win.ids + a.win.ids_off[w], (uint32_t)(a.win.ids_off[w + 1] - a.win.ids_off[w]));
        } else {  // bed.rs:150-153: "{chrom}:{st+1}-{en}"
            p = put_bytes(p, a.names + a.names_off[ri.t_name], (uint32_t)(a.names_off[ri.t_name + 1] - a.names_off[ri.t_name]));
            *p++ = ':'; p = put_u64(p, a.win.st[w] + 1);
            *p++ = '-'; p = put_u64(p, a.win.en[w]);
        }
    }
    *p++ = '\t'; *p++ = 'c'; *p++ = 'g'; *p++ = ':'; *p++ = 'Z'; *p++ = ':';
    return p;
}

// up to 64 bytes of the input CIGAR text -> p: every load is issued before the first store (the byte stores go through a
// generic pointer, which keeps the compiler from hoisting loads over them: in put_text's loop every load waits for the
// stores of the word before it), so the line pays one round trip to L2 instead of one per word
template <class P>
__device__ __forceinline__ P put_text64(P p, const uint8_t* __restrict__ src, uint32_t n) {
    const uint32_t* w = reinterpret_cast<const uint32_t*>(reinterpret_cast<uintptr_t>(src) & ~(uintptr_t)3);
    const uint32_t sh = (uint32_t)(reinterpret_cast<uintptr_t>(src) & 3u) * 8u;
    const uint32_t nw = (n + 3u) >> 2;  // output words
    uint32_t x[17];
#pragma unroll
    for (int i = 0; i < 17; i++) x[i] = ((uint32_t)i <= nw) ? __ldg(w + i) : 0u;
#pragma unroll
    for (int i = 0; i < 16; i++) {
        if ((uint32_t)i * 4u < n) {
            const uint32_t y = __funnelshift_r(x[i], x[i + 1], sh);
            const uint32_t b = (uint32_t)i * 4u;
            p[b] = (uint8_t)y;
            if (b + 1 < n) p[b + 1] = (uint8_t)(y >> 8);
            if (b + 2 < n) p[b + 2] = (uint8_t)(y >> 16);
            if (b + 3 < n) p[b + 3] = (uint8_t)(y >> 24);
        }
    }
    return p + n;
}

// n bytes of the input CIGAR text -> p, 64 bytes per round: the 17 source words of a round are all requested before its first
// byte is stored (see put_text64: with one word per iteration every load waited for the stores before it — one trip to L2 per
// 4 bytes, the reason the 10 kb-window rows, ~430 bytes of untouched ops each, ran at 15 % issue utilisation).  The text buffer
// is padded on both sides, so the over-read of up to 7 bytes stays inside it.
template <class P>
__device__ __forceinline__ P put_text(P p, const uint8_t* __restrict__ src, uint32_t n) {
    while (n > 64u) {
        p = put_text64(p, src, 64u);
        src += 64;
        n -= 64u;
    }
    return put_text64(p, src, n);
}

// trimmed / early-return CIGAR text, sequential.  Ops the trim leaves untouched are copied from the input text when
// the record spells them canonically (RF_CANON) instead of being re-formatted from the op words.
template <class P>
__device__ __forceinline__ P put_cigar_seq(P p, const SerArgs& a, const RecInfo& ri, const PairRes& pr) {
    const OpsView& v = a.v;
    const bool canon = (ri.flags & RF_CANON) != 0;
    if (pr.kind == PK_EARLY) {
        if (canon) return put_text(p, a.text + pr.mid_off, pr.mid_len);
        for (uint64_t k = pr.si; k <= pr.ei; k++) { const uint32_t w = v.op(k); p = put_op(p, op_len(w), op_code(w)); }
    } else if (ri.flags & RF_SLOW) {
        merged_walk(v, pr.si, pr.ei, pr.s_len, pr.e_len, [&](uint32_t len, uint32_t code) { p = put_op(p, len, code); });
    } else {
        p = put_op(p, pr.s_len, op_code(v.op(pr.si)));
        if (pr.ei > pr.si) {
            if (canon) p = put_text(p, a.text + pr.mid_off, pr.mid_len);
            else for (uint64_t k = pr.si + 1; k < pr.ei; k++) { const uint32_t w = v.op(k); p = put_op(p, op_len(w), op_code(w)); }
            p = put_op(p, pr.e_len, op_code(v.op(pr.ei)));
        }
    }
    return p;
}

__global__ void __launch_bounds__(SER_LINES)
k_serialise(uint64_t n_pairs, const uint64_t* __restrict__ pair_off, const uint32_t* __restrict__ rec_order, uint32_t n_rec,
            SerArgs a, const LiftPlan* __restrict__ plans, const PairRes* __restrict__ res, const uint64_t* __restrict__ line_off,
            const uint64_t* __restrict__ out_idx,
            uint8_t* __restrict__ out_text, uint64_t* __restrict__ out_line_off, NumDev num, StatsDev st, uint64_t byte_base,
            uint32_t rec_base, const uint32_t* __restrict__ orig_idx, uint32_t group, uint32_t defer_big,
            const uint32_t* __restrict__ only_flagged) {
    // only_flagged != nullptr: the call finishes what k_emit left (blocks of SER_LINES pairs whose flag is set)
    if (only_flagged && only_flagged[(uint64_t)blockIdx.x * group / SER_LINES] == 0u) return;
    // `group` = lines per block: SER_LINES normally; 8 when the rows are few and long (100 kb windows: a 4 KB line
    // per pair), so that the warp-per-line path below spreads over 16x more blocks
    extern __shared__ __align__(16) uint8_t s_buf[];
    __shared__ uint8_t s_stage[SER_LINES / 32][384];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint64_t p0 = (uint64_t)blockIdx.x * group;
    const uint64_t p = p0 + tid;
    const uint64_t pend = (p0 + group < n_pairs) ? (p0 + group) : n_pairs;
    const uint64_t byte0 = line_off[p0], byte1 = line_off[pend];
    const uint64_t region = byte1 - byte0;

    PairRes pr;
    pr.kind = PK_DROP;
    uint64_t my_off = 0, my_len = 0;
    uint32_t r = 0, w = 0;
    if (p < pend) {
        pr = res[p];
        my_off = line_off[p];
        my_len = line_off[p + 1] - my_off;
    }
    const bool live = (pr.kind != PK_DROP);
    static_assert(SER_LINES == LIFT_THREADS, "k_serialise reuses the per-block plan of k_lift");
    const LiftPlan pl = plans[p0 / SER_LINES];  // one record for the whole block (the usual case at scale): no per-thread search
    const bool uniform = (pl.uniform & PLAN_UNIFORM) != 0;
    if (live) {
        const uint32_t k = uniform ? pl.k0 : rank_of_pair(pair_off, n_rec, p);
        r = rec_order[k];
        w = a.win.pair_win ? a.win.pair_win[p] : (a.recs[r].wlo + (uint32_t)(p - pair_off[k]));
        const uint64_t o = out_idx[p];
        if (out_line_off) out_line_off[o] = my_off + byte_base;  // slices: offsets in the caller's concatenated text
        if (num.q_st) {
            num.q_st[o] = pr.q_st; num.q_en[o] = pr.q_en; num.t_st[o] = pr.t_st; num.t_en[o] = pr.t_en;
            num.nmatch[o] = pr.nmatch; num.aln_len[o] = pr.aln_len;
            num.rec_idx[o] = orig_idx ? orig_idx[r] : r + rec_base; num.win_idx[o] = a.win.bed_row ? a.win.bed_row[w] : w;
        }
        if (st.equal) write_stats(st, o, pr.equal, pr.diff, pr.ins, pr.del, pr.ins_ev, pr.del_ev, pr.matches);
    }
    if (out_line_off && p0 + group >= n_pairs && tid == 0) out_line_off[out_idx[n_pairs]] = line_off[n_pairs] + byte_base;
    if (out_text == nullptr || region == 0) return;

    const bool small = __syncthreads_and(my_len <= 2048) && region <= (uint64_t)(SER_CAP - 16);
    if (small) {
        // compose the whole line group in shared memory, one thread per line, then stream it out
        const uint32_t shift = (uint32_t)((uintptr_t)(out_text + byte0) & 15u);  // keep smem/global 16-byte phase equal
        if (live) {
            const RecInfo& ri = a.recs[r];
            uint8_t* q = s_buf + shift + (my_off - byte0);
            q = put_header(q, a, ri, pr, w);
            if (pr.kind == PK_WHOLE) q += pr.cg_bytes;  // k_whole_text fills these bytes afterwards
            else q = put_cigar_seq(q, a, ri, pr);
            *q = '\n';
        }
        fence_proxy_async();
        __syncthreads();
        uint8_t* dst = out_text + byte0;
        const uint32_t n = (uint32_t)region;
        const uint32_t head = (16u - shift) & 15u;  // bytes until dst is 16-byte aligned
        const uint32_t hb = head < n ? head : n;
        const uint32_t nvec = (n - hb) >> 4;
        // the 16-byte aligned body goes out as one bulk copy (shared -> global) issued by one thread ...
        if (tid == 0 && nvec) bulk_s2g(dst + hb, s_buf + shift + hb, nvec << 4);
        // ... the ragged ends by the others
        for (uint32_t i = tid; i < hb; i += SER_LINES) dst[i] = s_buf[shift + i];
        for (uint32_t i = hb + (nvec << 4) + tid; i < n; i += SER_LINES) dst[i] = s_buf[shift + i];
        if (tid == 0 && nvec) bulk_wait_read();  // the block's shared memory must outlive the engine's read of it
        return;
    }

    // long lines: one warp per line, straight to global memory
    for (uint64_t q = p0 + warp; q < pend; q += SER_LINES / 32) {
        const PairRes lp = res[q];
        if (lp.kind == PK_DROP) continue;
        const uint32_t k = rank_of_pair(pair_off, n_rec, q);
        const uint32_t rr = rec_order[k];
        const RecInfo& ri = a.recs[rr];
        const uint32_t ww = a.win.pair_win ? a.win.pair_win[q] : (ri.wlo + (uint32_t)(q - pair_off[k]));
        uint8_t* dst = out_text + line_off[q];
        const uint64_t llen = line_off[q + 1] - line_off[q];
        const uint64_t hdr = llen - lp.cg_bytes - 1;
        if (hdr <= 384) {
            if (lane == 0) put_header(&s_stage[warp][0], a, ri, lp, ww);
            __syncwarp();
            for (uint32_t i = lane; i < hdr; i += 32) dst[i] = s_stage[warp][i];
        } else if (lane == 0) {
            put_header(dst, a, ri, lp, ww);
        }
        __syncwarp();
        dst += hdr;
        if (lp.kind == PK_WHOLE) {
            // the CIGAR of a whole-record row is written by k_whole_text, 32 ops per warp across the whole grid
        } else if ((ri.flags & RF_SLOW) && lp.kind == PK_TRIM) {
            if (lane == 0) put_cigar_seq(dst, a, ri, lp);
        } else if (ri.flags & RF_CANON) {
            // untouched ops come straight from the input text: one coalesced copy by the whole warp
            uint64_t pos = 0;
            if (lp.kind == PK_TRIM) {
                if (lane == 0) {
                    uint8_t* e = put_op(dst, lp.s_len, op_code(a.v.op(lp.si)));
                    if (lp.ei > lp.si) put_op(e + lp.mid_len, lp.e_len, op_code(a.v.op(lp.ei)));
                }
                pos = ndigits32(lp.s_len) + 1;
            }
            if ((lp.kind == PK_EARLY || lp.ei > lp.si) && !(defer_big && mid_is_big(ri, lp))) {  // (big runs: k_copy_mid)
                const uint8_t* src = a.text + lp.mid_off;
                for (uint32_t i = lane; i < lp.mid_len; i += 32) dst[pos + i] = src[i];
            }
        } else {
            // 32 ops per round: per-lane text, warp scan of sizes, stage, coalesced byte copy
            uint64_t pos = 0;
            for (uint64_t k0 = lp.si; k0 <= lp.ei; k0 += 32) {
                const uint64_t kk = k0 + lane;
                uint32_t len = 0, code = 0, nb = 0;
                if (kk <= lp.ei) {
                    const uint32_t ow = a.v.op(kk);
                    code = op_code(ow);
                    len = op_len(ow);
                    if (lp.kind == PK_TRIM) {
                        if (kk == lp.si) len = lp.s_len;
                        else if (kk == lp.ei) len = lp.e_len;
                    }
                    nb = ndigits32(len) + 1;
                }
                uint32_t inc = nb;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const uint32_t t = __shfl_up_sync(0xffffffffu, inc, d);
                    if (lane >= d) inc += t;
                }
                const uint32_t tot = __shfl_sync(0xffffffffu, inc, 31);
                __syncwarp();
                if (nb) put_op(&s_stage[warp][inc - nb], len, code);
                __syncwarp();
                for (uint32_t i = lane; i < tot; i += 32) dst[pos + i] = s_stage[warp][i];
                pos += tot;
            }
        }
        if (lane == 0) out_text[line_off[q + 1] - 1] = '\n';
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------------
// K4+K5  k_emit: lift + line scan + serialiser in ONE pass over the pairs
// ------------------------------------------------------------------------------------------------
// A block owns SER_LINES consecutive pairs (dynamic ticket order).
//   FAST blocks (k_lift_plan: one record, op run + samples fit the staging area, no RF_SLOW, right-most policy) lift their
//   pairs right here, out of shared memory (same stages as k_lift, lift_core.cuh) — their results never exist in HBM.
//   Other blocks read the PairRes / line size k_lift left for them.
// Then: block scan of (bytes, rows); two single-word decoupled look-backs (warp 0: bytes, warp 1: rows) give the block's
// place in the output WHILE the other warps already compose their lines in shared memory (the 12 columns come from
// block-constant fragments, untouched ops are formatted from the staged op words: no global load on that path); the lines
// leave with 16-byte stores, re-aligned from the staging buffer with funnel shifts (the block's byte offset is not known
// when composing starts, so shared and global memory are in different 16-byte phases).  Rows that do not fit one buffer
// go in rounds.  No line_off / out_idx / PairRes arrays, no second pass.
// The output sizes are only known when the kernel ends, so the caller hands in the capacity of its text buffer: a block
// whose lines would not fit writes no text and raises the overflow flag (the caller grows the buffer to the exact size —
// the totals are right either way — and runs the kernel again; steady-state calls reuse the buffer of the call before).
// Blocks holding a line longer than EMIT_LONG bytes are left to k_serialise's warp-per-line path: they publish their
// results, offsets (line_off / out_idx of their pairs) and a flag.
constexpr uint32_t EMIT_LONG = 2048;
constexpr int EMIT_OPS_BYTES = (LIFT_CCAP + 1) * (int)SAMPLE * 4;                 // staged op words of a FAST block
constexpr int EMIT_SMP_BYTES = (LIFT_CCAP + 2) * (int)SUBS * (int)sizeof(Ctr);    // ... and its samples
constexpr int EMIT_ACC_BYTES = 9 * SER_LINES * 4;                                 // class sums of the walks
constexpr int EMIT_UNI_BYTES = EMIT_SMP_BYTES + EMIT_ACC_BYTES;                   // after the lift: line buffer of a FAST block
constexpr int EMIT_DYN_BYTES = EMIT_OPS_BYTES + EMIT_UNI_BYTES;                   // (other blocks compose in all of it)
constexpr uint32_t FRAG_CAP = 96, FRAG_NAME_MAX = 64;
constexpr int EMIT_MID_BYTES = SER_LINES * 16;  // the descriptors of copy_mids (blocks that do not lift)
// Wide-window calls (no block lifts here: launch_lift_plan was told not to mark any) take less shared memory per block, which the
// SM hands to L1: their loads are per-thread reads of results, record fields and names plus the streaming text copies, and the
// full 35 KB x 6 blocks left L1 under 30 KB.  Room for the 128 lines of a DIRECT block (~150 B each without their runs).
constexpr int EMIT_DYN_WIDE = 22 * 1024 + SER_LINES * 16 + (SER_LINES + 4) * 4;
constexpr int EMIT_REL2_BYTES = (SER_LINES + 4) * 4;  // ... and, in front of them, the prefix of their line sizes without the direct runs
constexpr uint32_t MID_COOP = 96;  // runs of untouched ops at least this long are copied by a warp instead of their line's thread
static_assert(EMIT_OPS_BYTES % 16 == 0 && EMIT_SMP_BYTES % 16 == 0, "staging areas are 16-byte aligned");
static_assert(EMIT_UNI_BYTES >= (int)EMIT_LONG + 64, "one round holds at least one line");

struct EmitArgs {
    uint64_t n_pairs;
    const uint64_t* pair_off;
    const uint32_t* rec_order;
    uint32_t n_rec;
    SerArgs a;            // a.v.samples is set: FAST blocks lift
    const LiftPlan* plans;
    PairRes* res;         // read by the blocks k_lift handled; written by FAST blocks that have to defer
    const uint32_t* line_len;
    uint64_t* line_off;   // written for deferred blocks only
    uint64_t* out_idx;
    uint32_t* blk_flags;  // per block: 1 = its text is left to k_serialise
    uint8_t* out_text;
    uint64_t cap_text;
    uint64_t* out_line_off;
    NumDev num;
    StatsDev st;
    uint64_t byte_base;
    uint32_t rec_base;
    const uint32_t* orig_idx;
    unsigned long long* lb_bytes;  // look-back words (one per block), zeroed by the caller
    unsigned long long* lb_rows;
    unsigned int* ticket;
    unsigned long long* totals;  // [0] bytes of text, [1] rows, [2] != 0: the text did not fit, [3] deferred blocks
    ErrSlots err;
    uint32_t stats_text;         // RB_WANT_STATS_TEXT: the rows `rb stats --paf` prints for the lifted rows instead of the PAF rows
    uint32_t dyn_bytes;          // dynamic shared memory of this launch: EMIT_DYN_BYTES, or EMIT_DYN_WIDE when no block lifts (wide windows)
};

// bamstats.rs:138-142 — the three f32 identities of a row (IEEE mul + div, no contraction), as bit patterns
__device__ __forceinline__ void identities(const PairRes& pr, uint32_t bits[3]) {
    const float num = __fmul_rn(100.0f, __uint2float_rn(pr.equal));
    bits[0] = __float_as_uint(__fdiv_rn(num, __uint2float_rn(pr.equal + pr.diff)));                            // by matches
    bits[1] = __float_as_uint(__fdiv_rn(num, __uint2float_rn(pr.equal + pr.diff + pr.del_ev + pr.ins_ev)));    // by events
    bits[2] = __float_as_uint(__fdiv_rn(num, __uint2float_rn(pr.equal + pr.diff + pr.del + pr.ins)));          // by all
}

// n bytes from a 4-byte aligned shared-memory fragment
__device__ __forceinline__ uint8_t* put_frag(uint8_t* p, const uint8_t* frag, uint32_t n) {
    const uint32_t* w = reinterpret_cast<const uint32_t*>(frag);
    uint32_t i = 0;
    for (; i + 4 <= n; i += 4) {
        const uint32_t x = w[i >> 2];
        p[i] = (uint8_t)x; p[i + 1] = (uint8_t)(x >> 8); p[i + 2] = (uint8_t)(x >> 16); p[i + 3] = (uint8_t)(x >> 24);
    }
    if (i < n) {
        const uint32_t x = w[i >> 2];
        p[i] = (uint8_t)x;
        if (i + 1 < n) p[i + 1] = (uint8_t)(x >> 8);
        if (i + 2 < n) p[i + 2] = (uint8_t)(x >> 16);
    }
    return p + n;
}

// n bytes of shared memory (any alignment) -> global memory: 16-byte stores where the destination allows, source words
// re-aligned with funnel shifts.  Executed by the whole block.
__device__ __forceinline__ void copy_out_shifted(uint8_t* __restrict__ dst, const uint8_t* sbuf, uint32_t n) {
    const int tid = threadIdx.x;
    const uint32_t head = (uint32_t)((16u - ((uintptr_t)dst & 15u)) & 15u);
    const uint32_t hb = head < n ? head : n;
    const uint32_t nvec = (n - hb) >> 4;
    for (uint32_t i = tid; i < hb; i += SER_LINES) dst[i] = sbuf[i];
    const uint8_t* sb = sbuf + hb;
    const uint32_t sa = smem_u32(sb);
    const uint32_t sh = (sa & 3u) * 8u;
    const uint32_t* w0 = reinterpret_cast<const uint32_t*>(sb - (sa & 3u));  // (over-reads <= 7 bytes behind the data: inside the buffer's slack)
    uint4* d4 = reinterpret_cast<uint4*>(dst + hb);
    for (uint32_t v = tid; v < nvec; v += SER_LINES) {
        const uint32_t* w = w0 + (size_t)v * 4;
        const uint32_t a0 = w[0], a1 = w[1], a2 = w[2], a3 = w[3], a4 = w[4];
        uint4 x;
        x.x = __funnelshift_r(a0, a1, sh); x.y = __funnelshift_r(a1, a2, sh); x.z = __funnelshift_r(a2, a3, sh); x.w = __funnelshift_r(a3, a4, sh);
        d4[v] = x;
    }
    for (uint32_t i = hb + (nvec << 4) + tid; i < n; i += SER_LINES) dst[i] = sbuf[i];
}

// lift_pair_chain of k_lift, specialised for FAST blocks (everything in shared memory, right-most policy, no RF_SLOW)
__device__ __forceinline__ uint32_t lift_pair_fast(const OpsView& v, const RecInfo& r, uint64_t w_st, uint64_t w_en, bool enabled,
                                                   PairRes& out, ClassAcc& acc, ChainSlot* s_x) {
    constexpr unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t status = LIFT_OK;
    bool live = enabled;
    pair_clear(out);
    if (live && r.t_st > w_st && r.t_en < w_en) {
        pair_early(r, out);
        live = false;
    } else if (live && r.t_en <= r.t_st) {
        status = LIFT_ERR_NOT_FOUND;
        live = false;
    }
    const uint32_t ps = live ? (uint32_t)((w_st > r.t_st ? w_st : r.t_st) - r.t_st) : 0u;
    const uint32_t pe = live ? (uint32_t)((w_en < r.t_en ? w_en : r.t_en) - 1 - r.t_st) : 0u;
    uint64_t ie = 0; uint32_t oe = 0; Ctr be = ctr_zero();
    const bool fe = find_op<true>(v, r, live, pe, ie, oe, be, acc);
    // hand (ie, oe, be) to the right neighbour (tiling windows: its start boundary is one base further)
    const uint32_t ok = (live && fe) ? 1u : 0u;
    if (lane == 31) {
        ChainSlot& x = s_x[warp];
        x.i = ie; x.o = oe; x.pe = pe; x.ok = ok; x.c = be;
    }
    __syncthreads();
    uint32_t p_ok = __shfl_up_sync(FULL, ok, 1), p_pe = __shfl_up_sync(FULL, pe, 1);
    uint32_t po = __shfl_up_sync(FULL, oe, 1);
    uint64_t pi = __shfl_up_sync(FULL, ie, 1);
    Ctr pb;
    {
        uint32_t* dw = reinterpret_cast<uint32_t*>(&pb);
        const uint32_t* sw = reinterpret_cast<const uint32_t*>(&be);
#pragma unroll
        for (int t = 0; t < 12; t++) dw[t] = __shfl_up_sync(FULL, sw[t], 1);
    }
    if (lane == 0) {
        p_ok = 0u;
        if (warp > 0) {
            const ChainSlot& x = s_x[warp - 1];
            p_ok = x.ok; p_pe = x.pe; po = x.o; pi = x.i; pb = x.c;
        }
    }
    const bool derive = live && p_ok && ps == p_pe + 1u;
    uint64_t i = 0; uint32_t o = 0; Ctr before = ctr_zero();
    bool fs = false;
    const bool search = live && !derive;
    if (__any_sync(FULL, search)) fs = find_op<true>(v, r, search, ps, i, o, before, acc);
    if (derive) fs = advance_one(v, r, pi, po, pb, i, o, before);
    __syncwarp();
    if (!fs && live) { status = LIFT_ERR_NOT_FOUND; live = false; }
    uint64_t si = 0; uint32_t so = 0; Ctr cs = ctr_zero();
    if (live && !lift_start(v, r.eo1, r.a_lead, r.tot.A, POLICY_RIGHTMOST, i, o, before, si, so, cs)) live = false;
    __syncwarp();
    if (live && !fe) { status = LIFT_ERR_NOT_FOUND; live = false; }
    if (live) {
        uint64_t ei; uint32_t eo; Ctr ce; uint32_t txt_before_ei;
        if (lift_end(v, r.eo0, ie, oe, be, ei, eo, ce, txt_before_ei))
            lift_finish<true>(v, r, si, so, cs, op_len(v.op(si)), ei, eo, ce, txt_before_ei, out);
    }
    __syncwarp();
    return status;
}

// n bytes of staged input text (shared memory, any alignment) -> the line buffer (shared memory, any alignment): word stores
// once the destination is aligned, the source words re-aligned with funnel shifts (reads < 4 bytes past the run: staged slack)
__device__ __forceinline__ uint8_t* put_text_smem(uint8_t* q, const uint8_t* src, uint32_t n) {
    uint32_t h = (4u - (smem_u32(q) & 3u)) & 3u;
    h = h < n ? h : n;
    for (uint32_t i = 0; i < h; i++) q[i] = src[i];
    q += h; src += h; n -= h;
    const uint32_t sa = smem_u32(src);
    const uint32_t sh = (sa & 3u) * 8u;
    const uint32_t* w = reinterpret_cast<const uint32_t*>(src - (sa & 3u));
    uint32_t* d = reinterpret_cast<uint32_t*>(q);
    const uint32_t nw = n >> 2;
    uint32_t lo = w[0];
    for (uint32_t i = 0; i < nw; i++) {
        const uint32_t hi = w[i + 1];
        d[i] = __funnelshift_r(lo, hi, sh);
        lo = hi;
    }
    for (uint32_t i = nw << 2; i < n; i++) q[i] = src[i];
    return q + n;
}

template <bool STATS_TEXT>  // (a template: the f32 digit generation of the stats rows stays out of the PAF instantiation's registers)
__global__ void __launch_bounds__(SER_LINES, RB_EMIT_MINB)
k_emit(const __grid_constant__ EmitArgs e) {
    extern __shared__ __align__(16) uint8_t s_emit[];
    __shared__ uint32_t s_rel[SER_LINES + 1];
    __shared__ unsigned long long s_wb[SER_LINES / 32];
    __shared__ uint32_t s_wc[SER_LINES / 32], s_w2[SER_LINES / 32];
    __shared__ unsigned long long s_tlo[SER_LINES / 32], s_thi[SER_LINES / 32];
    __shared__ unsigned long long s_base[2];
    __shared__ unsigned int s_blk;
    __shared__ __align__(16) RecInfo s_rec;
    __shared__ __align__(16) ChainSlot s_chain[SER_LINES / 32];
    __shared__ __align__(8) unsigned long long s_bar;
    __shared__ __align__(16) uint8_t s_frag[4][FRAG_CAP];
    __shared__ uint32_t s_flen[4];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_blk = atomicAdd(e.ticket, 1u);
    __syncthreads();
    const uint64_t blk = s_blk;
    const uint64_t p0 = blk * SER_LINES;
    if (p0 >= e.n_pairs) return;
    const uint64_t p = p0 + tid;
    const uint64_t pend = (p0 + SER_LINES < e.n_pairs) ? (p0 + SER_LINES) : e.n_pairs;
    const uint32_t nlines = (uint32_t)(pend - p0);
    const LiftPlan pl = e.plans[blk];
    const bool fast = (pl.uniform & PLAN_FAST) != 0;  // block-uniform
    const bool in_range = p < pend;

    PairRes pr;
    pr.kind = PK_DROP;
    uint32_t len = 0, r = 0, w = 0;
    uint64_t w_st = 0, w_en = 0;
    OpsView v = e.a.v;
    uint8_t* s_buf;       // line buffer of this block
    uint32_t buf_cap;
    // Blocks that lift here: the record goes to shared memory and the block-constant pieces of the rows are composed once — no
    // thread loads names or record fields again.  (The same for uniform blocks that do NOT lift was measured at 10 kb windows:
    // 16 % slower — without the wait for the staged ops to hide behind, four lanes chasing names hold up the whole block.)
    const bool uni = fast;  // block-uniform
    const RecInfo* gr = nullptr;
    if (uni) {
        r = e.rec_order[pl.k0];
        gr = &e.a.recs[r];
        if (tid < (int)(sizeof(RecInfo) / 16)) reinterpret_cast<uint4*>(&s_rec)[tid] = reinterpret_cast<const uint4*>(gr)[tid];
    if (warp == 3 && lane < 4) {  // block-constant pieces of the 12 columns (paf.rs:923-943), one lane each
        const uint32_t qn = gr->q_name, tn = gr->t_name;
        const uint64_t qo = e.a.names_off[qn], to = e.a.names_off[tn];
        const uint32_t ql = (uint32_t)(e.a.names_off[qn + 1] - qo), tl = (uint32_t)(e.a.names_off[tn + 1] - to);
        uint8_t* f = s_frag[lane];
        uint8_t* q = f;
        if (ql <= FRAG_NAME_MAX && tl <= FRAG_NAME_MAX && STATS_TEXT) {  // bamstats.rs:239-270 (reference block first)
            if (lane == 0) {         // t_name \t
                q = put_bytes(q, e.a.names + to, tl); *q++ = '\t';
            } else if (lane == 1) {  // \t t_len \t strand \t q_name \t
                *q++ = '\t'; q = put_u64(q, gr->t_len); *q++ = '\t'; *q++ = (gr->flags & RF_MINUS) ? '-' : '+'; *q++ = '\t';
                q = put_bytes(q, e.a.names + qo, ql); *q++ = '\t';
            } else if (lane == 2) {  // \t q_len \t
                *q++ = '\t'; q = put_u64(q, gr->q_len); *q++ = '\t';
            }
            s_flen[lane] = (uint32_t)(q - f);
        } else if (ql <= FRAG_NAME_MAX && tl <= FRAG_NAME_MAX) {
            if (lane == 0) {         // q_name \t q_len \t
                q = put_bytes(q, e.a.names + qo, ql); *q++ = '\t'; q = put_u64(q, gr->q_len); *q++ = '\t';
            } else if (lane == 1) {  // \t strand \t t_name \t t_len \t
                *q++ = '\t'; *q++ = (gr->flags & RF_MINUS) ? '-' : '+'; *q++ = '\t';
                q = put_bytes(q, e.a.names + to, tl); *q++ = '\t'; q = put_u64(q, gr->t_len); *q++ = '\t';
            } else if (lane == 2) {  // \t mapq \t id:Z:
                *q++ = '\t'; q = put_u64(q, gr->mapq);
                *q++ = '\t'; *q++ = 'i'; *q++ = 'd'; *q++ = ':'; *q++ = 'Z'; *q++ = ':';
            } else {                 // default window id: t_name :
                q = put_bytes(q, e.a.names + to, tl); *q++ = ':';
            }
            s_flen[lane] = (uint32_t)(q - f);
        } else {
            s_flen[lane] = 0xFFFFFFFFu;  // long names: the generic header writer
        }
    }
    }
    bool txt_mode = false;          // FAST block composing from staged input text (block-uniform)
    unsigned long long txt_lo = 0;  // text offset of the first staged byte
    uint32_t code_s = 0, code_e = 0;
    if (fast) {
        // ---- stage the block's op run + samples (bulk-copy engine); lift ----
        uint32_t* s_ops = reinterpret_cast<uint32_t*>(s_emit);
        Ctr* s_smp = reinterpret_cast<Ctr*>(s_emit + EMIT_OPS_BYTES);
        uint32_t* s_acc = reinterpret_cast<uint32_t*>(s_emit + EMIT_OPS_BYTES + EMIT_SMP_BYTES);
        const uint64_t c_lo = pl.c_lo, c_hi = pl.c_hi;
        const uint64_t op_end = gr->op_end;
        const uint64_t o_lo = c_lo << SAMPLE_LOG2;
        uint64_t o_hi = (c_hi + 2) << SAMPLE_LOG2;  // one extra chunk for the look-ahead of the slide rules
        if (o_hi > op_end) o_hi = op_end;
        const uint32_t n_stage = (uint32_t)(o_hi - o_lo), n4 = n_stage >> 2;
        const uint64_t c_max = (op_end - 1) >> SAMPLE_LOG2;
        const uint64_t c_top = (c_hi + 1 <= c_max) ? c_hi + 1 : c_max;
        const uint32_t smp_bytes = (uint32_t)((c_top - c_lo + 1) * SUBS * sizeof(Ctr));
        if (tid == 0) {
            mbar_init(&s_bar, 1);
            mbar_expect_tx(&s_bar, n4 * 16u + smp_bytes);
            if (n4) bulk_g2s(s_ops, v.ops + o_lo, n4 * 16u, &s_bar);
            bulk_g2s(s_smp, v.samples + c_lo * SUBS, smp_bytes, &s_bar);
        }
        for (uint32_t k = (n4 << 2) + tid; k < n_stage; k += SER_LINES) s_ops[k] = v.ops[o_lo + k];  // the (< 4 op) tail
        v.s_smp = s_smp; v.sc_lo = c_lo; v.sc_hi = c_top + 1;
        v.s_ops = s_ops; v.so_lo = o_lo; v.so_hi = o_hi;
        const uint64_t pc = in_range ? p : e.n_pairs - 1;
        w = gr->wlo + (uint32_t)(pc - e.pair_off[pl.k0]);
        w_st = e.a.win.st[w]; w_en = e.a.win.en[w];
        __syncthreads();  // s_rec, the fragments, the tail ops and the mbarrier's initialisation are visible
        mbar_wait(&s_bar, 0);
        const RecInfo& ri = s_rec;
        ClassAcc acc;
        acc.sum = s_acc + tid; acc.stride = SER_LINES;
        const bool overlaps = in_range && ri.t_en > w_st && ri.t_st < w_en && !(e.a.win.from_record && w_en <= w_st);
        const uint32_t st = lift_pair_fast(v, ri, w_st, w_en, overlaps, pr, acc, s_chain);
        if (in_range && st != LIFT_OK) { report(e.err.rec, r, RE_INDEX_PANIC); pr.kind = PK_DROP; }
        if (!in_range) pr.kind = PK_DROP;
        if (pr.kind != PK_DROP) {
            uint32_t idl = ri.id_len;  // early rows and break-paf pieces carry their record's id
            if (pr.kind != PK_EARLY && !e.a.win.from_record) {
                const uint32_t tn = e.a.win.ids_off ? 0u : (uint32_t)(e.a.names_off[ri.t_name + 1] - e.a.names_off[ri.t_name]);
                idl = win_id_len(e.a.win, w, tn, w_st, w_en);
            }
            len = ri.line_const + line_var_bytes(pr, idl);
        }
        // the op words stay staged for the serialiser; samples + class sums make room for the lines
        v.s_smp = nullptr; v.sc_lo = v.sc_hi = 0;
        s_buf = s_emit + EMIT_OPS_BYTES;
        buf_cap = (uint32_t)EMIT_UNI_BYTES;
#if RB_EMIT_STAGE_TEXT
        // ... unless the record spells its CIGAR canonically: then the rows' untouched ops ARE bytes of the input text, and the
        // span of it this block's rows cover (~6 KB at 1 kb windows) takes the place of the op words — a row copies ~45 bytes
        // shared -> shared instead of formatting ~15 ops (a quarter of this kernel's instructions at C4)
        if (!STATS_TEXT && (ri.flags & RF_CANON)) {
            const bool has_mid = pr.kind == PK_TRIM && pr.ei > pr.si && pr.mid_len > 0u;
            if (pr.kind == PK_TRIM) { code_s = op_code(v.op(pr.si)); code_e = op_code(v.op(pr.ei)); }
            unsigned long long lo = has_mid ? pr.mid_off : ~0ull, hi = has_mid ? pr.mid_off + pr.mid_len : 0ull;
#pragma unroll
            for (int d = 16; d >= 1; d >>= 1) {
                const unsigned long long ol = __shfl_xor_sync(0xffffffffu, lo, d), oh = __shfl_xor_sync(0xffffffffu, hi, d);
                lo = ol < lo ? ol : lo; hi = oh > hi ? oh : hi;
            }
            if (lane == 0) { s_tlo[warp] = lo; s_thi[warp] = hi; }
            __syncthreads();  // every thread has read what it needs of the op words
            lo = s_tlo[0]; hi = s_thi[0];
#pragma unroll
            for (int k = 1; k < SER_LINES / 32; k++) { lo = s_tlo[k] < lo ? s_tlo[k] : lo; hi = s_thi[k] > hi ? s_thi[k] : hi; }
            if (hi > lo) {
                txt_lo = lo & ~15ull;
                const unsigned long long bytes = ((hi + 15ull) & ~15ull) - txt_lo;
                if (bytes + 16u <= (unsigned long long)EMIT_OPS_BYTES) {  // (block-uniform)
                    txt_mode = true;
                    v.s_ops = nullptr; v.so_lo = v.so_hi = 0;  // the op words are gone: early rows / strip ids read HBM
                    if (tid == 0) {
                        mbar_expect_tx(&s_bar, (uint32_t)bytes);
                        bulk_g2s(s_emit, e.a.text + txt_lo, (uint32_t)bytes, &s_bar);  // (the text buffer is padded on both sides)
                    }
                }
            }
        }
#endif
        __syncthreads();
    } else {
        if (in_range) {
            len = e.line_len[p];
            if (len) pr = e.res[p];
        }
        s_buf = s_emit;
        buf_cap = e.dyn_bytes - (uint32_t)(EMIT_MID_BYTES + EMIT_REL2_BYTES);
    }
    // blocks that do not lift keep, behind their line buffer, one descriptor per line: a run of input text its owner left to the
    // warps (src lo, src hi, dst offset, bytes)
    uint4* s_mid = reinterpret_cast<uint4*>(s_emit + e.dyn_bytes - EMIT_MID_BYTES);
    uint32_t* s_rel2 = reinterpret_cast<uint32_t*>(s_emit + e.dyn_bytes - EMIT_MID_BYTES - EMIT_REL2_BYTES);  // (blocks that do not lift only)
    bool live = len != 0u;
    if (!live) { r = 0; w = 0; }
    else if (!fast) {
        const uint32_t k = (pl.uniform & PLAN_UNIFORM) ? pl.k0 : rank_of_pair(e.pair_off, e.n_rec, p);
        r = e.rec_order[k];
        w = e.a.win.pair_win ? e.a.win.pair_win[p] : (e.a.recs[r].wlo + (uint32_t)(p - e.pair_off[k]));
    }
    // RB_WANT_STATS_TEXT: the row is the `rb stats --paf` row of the lifted record — shortest-round-trip digits of the three
    // identities now (their lengths decide where the rows go), printed when the row is composed
    uint32_t id_bits[3] = {0u, 0u, 0u};
    F32Dec id_dec[3];
    id_dec[0].n = id_dec[1].n = id_dec[2].n = 0;
    if (STATS_TEXT && live) {
        const RecInfo& ri = uni ? s_rec : e.a.recs[r];
        identities(pr, id_bits);
        uint32_t n = 0;
#pragma unroll
        for (int i = 0; i < 3; i++) {
            id_dec[i] = f32_shortest_fast(id_bits[i]);
            n += f32_display_len(id_bits[i], id_dec[i]);
        }
        uint32_t cst;  // the record's part: both names, t_len, q_len, strand
        if (uni && s_flen[0] != 0xFFFFFFFFu) cst = s_flen[0] + s_flen[1] + s_flen[2];
        else cst = (uint32_t)(e.a.names_off[ri.t_name + 1] - e.a.names_off[ri.t_name]) + (uint32_t)(e.a.names_off[ri.q_name + 1] - e.a.names_off[ri.q_name]) +
                   ndigits64(ri.t_len) + ndigits64(ri.q_len) + 1u + 7u;
        len = cst + ndigits64(pr.t_st) + ndigits64(pr.t_en) + ndigits64(pr.q_st) + ndigits64(pr.q_en) + n + ndigits32(pr.equal) +
              ndigits32(pr.diff) + ndigits32(pr.del_ev) + ndigits32(pr.ins_ev) + ndigits32(pr.del) + ndigits32(pr.ins) + 2u + 8u + 1u;
    }

    // A long run of untouched ops (wide windows: ~430 bytes of a ~560-byte row at 10 kb) can leave the input text for the
    // output without passing through the line buffer (DIRECT blocks, below): which of my line's bytes are such a run
    uint32_t dml = 0;
    if (!STATS_TEXT && !fast && live && pr.mid_len >= MID_COOP) {
        const uint32_t fl = e.a.recs[r].flags;
        if ((fl & RF_CANON) && (pr.kind == PK_EARLY || (pr.kind == PK_TRIM && pr.ei > pr.si && !(fl & RF_SLOW)))) dml = pr.mid_len;
    }
    // ---- block scan of (bytes, rows, bytes without the direct runs) ----
    unsigned long long ib = len;
    uint32_t ic = live ? 1u : 0u, i2 = len - dml;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const unsigned long long ub = __shfl_up_sync(0xffffffffu, ib, d);
        const uint32_t uc = __shfl_up_sync(0xffffffffu, ic, d);
        if (lane >= d) { ib += ub; ic += uc; }
    }
    if (!fast) {  // (block-uniform: blocks that lift never go DIRECT and skip the third scan)
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t u2 = __shfl_up_sync(0xffffffffu, i2, d);
            if (lane >= d) i2 += u2;
        }
        if (lane == 31) s_w2[warp] = i2;
    }
    if (lane == 31) { s_wb[warp] = ib; s_wc[warp] = ic; }
    const bool small = __syncthreads_and(len <= EMIT_LONG) != 0;
    unsigned long long wb = 0, tb = 0;
    uint32_t wc = 0, tc = 0, w2 = 0, t2 = 0;
#pragma unroll
    for (int k = 0; k < SER_LINES / 32; k++) {
        if (k < warp) { wb += s_wb[k]; wc += s_wc[k]; }
        tb += s_wb[k]; tc += s_wc[k];
    }
    const unsigned long long rel = wb + ib - len;  // bytes of the block's lines in front of mine
    uint32_t rel2 = 0;                             // ... without the direct runs
    s_rel[tid] = (uint32_t)rel;
    if (tid == 0) s_rel[SER_LINES] = (uint32_t)tb;
    if (!fast) {
#pragma unroll
        for (int k = 0; k < SER_LINES / 32; k++) {
            if (k < warp) w2 += s_w2[k];
            t2 += s_w2[k];
        }
        rel2 = w2 + i2 - (len - dml);
        s_rel2[tid] = rel2;
        if (tid == 0) s_rel2[SER_LINES] = t2;
    }

    const bool want_text = e.out_text != nullptr && tb != 0;
    const bool compose_early = want_text && small;  // (block-uniform)
    // DIRECT (block-uniform): a block that does not lift, whose runs are at least half of its bytes, and whose lines WITHOUT
    // them fit the buffer at once.  Its lines are composed side by side without the runs (one round instead of three at
    // 10 kb windows), each line's two pieces go out separately, and the runs are copied text -> output by a warp each —
    // they used to go text -> shared memory -> output, a round of the block's barriers per 26 KB
    const bool direct = RB_EMIT_DIRECT && !STATS_TEXT && !fast && compose_early && 2ull * (tb - t2) >= tb &&
                        t2 + 32u <= e.dyn_bytes - (uint32_t)(EMIT_MID_BYTES + EMIT_REL2_BYTES);

    // one line into the staging buffer at `q` — FAST blocks: fragments + staged ops, no global loads
    auto compose = [&](uint8_t* q) {
        const RecInfo& ri = uni ? s_rec : e.a.recs[r];
        if (STATS_TEXT) {  // bamstats.rs:239-270: reference block, strand, query block, identities, counters
            if (uni && s_flen[0] != 0xFFFFFFFFu) {
                q = put_frag(q, s_frag[0], s_flen[0]);
                q = put_u64(q, pr.t_st); *q++ = '\t'; q = put_u64(q, pr.t_en);
                q = put_frag(q, s_frag[1], s_flen[1]);
                q = put_u64(q, pr.q_st); *q++ = '\t'; q = put_u64(q, pr.q_en);
                q = put_frag(q, s_frag[2], s_flen[2]);
            } else {
                q = put_bytes(q, e.a.names + e.a.names_off[ri.t_name], (uint32_t)(e.a.names_off[ri.t_name + 1] - e.a.names_off[ri.t_name]));
                *q++ = '\t'; q = put_u64(q, pr.t_st); *q++ = '\t'; q = put_u64(q, pr.t_en); *q++ = '\t'; q = put_u64(q, ri.t_len);
                *q++ = '\t'; *q++ = (ri.flags & RF_MINUS) ? '-' : '+'; *q++ = '\t';
                q = put_bytes(q, e.a.names + e.a.names_off[ri.q_name], (uint32_t)(e.a.names_off[ri.q_name + 1] - e.a.names_off[ri.q_name]));
                *q++ = '\t'; q = put_u64(q, pr.q_st); *q++ = '\t'; q = put_u64(q, pr.q_en); *q++ = '\t'; q = put_u64(q, ri.q_len); *q++ = '\t';
            }
#pragma unroll
            for (int i = 0; i < 3; i++) { q = f32_display_put(q, id_bits[i], id_dec[i]); *q++ = '\t'; }
            q = put_u32(q, pr.equal); *q++ = '\t'; q = put_u32(q, pr.diff); *q++ = '\t'; q = put_u32(q, pr.del_ev); *q++ = '\t';
            q = put_u32(q, pr.ins_ev); *q++ = '\t'; q = put_u32(q, pr.del); *q++ = '\t'; q = put_u32(q, pr.ins);
            *q = '\n';
            return;
        }
        if (uni && s_flen[0] != 0xFFFFFFFFu) {
            q = put_frag(q, s_frag[0], s_flen[0]);
            q = put_u64(q, pr.q_st); *q++ = '\t'; q = put_u64(q, pr.q_en);
            q = put_frag(q, s_frag[1], s_flen[1]);
            q = put_u64(q, pr.t_st); *q++ = '\t'; q = put_u64(q, pr.t_en);
            *q++ = '\t'; q = put_u32(q, pr.nmatch);
            *q++ = '\t'; q = put_u32(q, pr.aln_len);
            q = put_frag(q, s_frag[2], s_flen[2]);
            if (pr.kind == PK_EARLY || e.a.win.from_record) {
                if (ri.flags & RF_STRIPPED) q = put_strip_id(q, ri, v);
            } else if (e.a.win.ids_off) {
                q = put_bytes(q, e.a.win.ids + e.a.win.ids_off[w], (uint32_t)(e.a.win.ids_off[w + 1] - e.a.win.ids_off[w]));
            } else {  // bed.rs:150-153: "{chrom}:{st+1}-{en}"
                q = put_frag(q, s_frag[3], s_flen[3]);
                q = put_u64(q, w_st + 1); *q++ = '-'; q = put_u64(q, w_en);
            }
            *q++ = '\t'; *q++ = 'c'; *q++ = 'g'; *q++ = ':'; *q++ = 'Z'; *q++ = ':';
        } else {
            q = put_header(q, e.a, ri, pr, w);
        }
        const uint32_t* run = (fast && pr.kind == PK_TRIM) ? v.op_run(pr.si, (uint32_t)(pr.ei - pr.si + 1)) : nullptr;
        if (txt_mode && pr.kind == PK_TRIM) {  // first op, the untouched ops as the staged input text spells them, last op
            q = put_op(q, pr.s_len, code_s);
            if (pr.ei > pr.si) {
                if (pr.mid_len) q = put_text_smem(q, s_emit + (uint32_t)(pr.mid_off - txt_lo), pr.mid_len);
                q = put_op(q, pr.e_len, code_e);
            }
        } else if (run) {  // the trimmed op range is staged (no RF_SLOW here)
            const uint32_t n_mid = (uint32_t)(pr.ei - pr.si);
            q = put_op(q, pr.s_len, op_code(run[0]));
            if (n_mid) {
#if RB_EMIT_MID_TEXT
                if ((ri.flags & RF_CANON) && pr.mid_len <= 64u) {  // untouched ops: their bytes of the input text, loads up front
                    q = put_text64(q, e.a.text + pr.mid_off, pr.mid_len);
                } else
#endif
                {   // ... or formatted from the staged op words
                    for (uint32_t k = 1; k < n_mid; k++) q = put_op(q, op_len(run[k]), op_code(run[k]));
                }
                q = put_op(q, pr.e_len, op_code(run[n_mid]));
            }
        } else if (!fast && (ri.flags & RF_CANON) && pr.mid_len >= MID_COOP &&
                   (pr.kind == PK_EARLY || (pr.kind == PK_TRIM && pr.ei > pr.si && !(ri.flags & RF_SLOW)))) {
            // a long run of untouched ops (wide windows: ~430 bytes per row at 10 kb): the owner writes what it formats itself
            // and leaves the run to the block's warps (copy_mids below): coalesced loads of the input text by 32 lanes per
            // row instead of one lane walking it — and every thread of the block has work while the round is composed
            if (pr.kind == PK_TRIM) q = put_op(q, pr.s_len, op_code(v.op(pr.si)));
            if (direct) {  // the run is not given room here: .z = where it goes in the block's OUTPUT bytes
                const uint32_t hl = (uint32_t)(q - (s_buf + 16)) - rel2;  // (< 2^16: lines of these blocks are at most EMIT_LONG bytes)
                s_mid[tid] = make_uint4((uint32_t)pr.mid_off, (uint32_t)(pr.mid_off >> 32), (uint32_t)rel + hl, pr.mid_len | (hl << 16));
            } else {
                s_mid[tid] = make_uint4((uint32_t)pr.mid_off, (uint32_t)(pr.mid_off >> 32), (uint32_t)(q - (s_buf + 16)), pr.mid_len);
                q += pr.mid_len;
            }
            if (pr.kind == PK_TRIM) q = put_op(q, pr.e_len, op_code(v.op(pr.ei)));
        } else {
            SerArgs a2 = e.a;
            a2.v = v;
            q = put_cigar_seq(q, a2, ri, pr);
        }
        *q = '\n';
    };
    // the runs the owners of lines [a, b) left behind: a warp per line, 4 bytes per lane and step, destination-aligned
    // shared-memory words assembled from two aligned words of the text (the buffer is padded: over-reads of < 8 bytes are fine)
    uint8_t* mid_dst0 = s_buf + 16;  // (DIRECT blocks: the block's place in the output, once it is known)
    auto copy_mids = [&](uint32_t a, uint32_t b) {
        for (uint32_t L = a + (uint32_t)warp; L < b; L += SER_LINES / 32) {
            const uint4 d = s_mid[L];
            if (d.w == 0u) continue;
            const uint8_t* src = e.a.text + (((uint64_t)d.y << 32) | d.x);
            uint8_t* dst = mid_dst0 + d.z;
            const uint32_t n = direct ? (d.w & 0xFFFFu) : d.w;  // (DIRECT: the bytes in front of the run ride in the high half)
            const uint32_t head = (4u - (uint32_t)((uintptr_t)dst & 3u)) & 3u;  // (n >= MID_COOP > 3; shared or global: the low bits agree)
            if ((uint32_t)lane < head) dst[lane] = __ldg(src + lane);
            const uint32_t nw = (n - head) >> 2, rem = (n - head) & 3u;
            const uint8_t* sb = src + head;
            const uint32_t sh = (uint32_t)((uintptr_t)sb & 3u) * 8u;
            const uint32_t* w0 = reinterpret_cast<const uint32_t*>((uintptr_t)sb & ~(uintptr_t)3);
            uint32_t* dw = reinterpret_cast<uint32_t*>(dst + head);
            for (uint32_t j0 = 0; j0 < nw; j0 += 128) {  // 4 words per lane and step, every load requested before the first store
                uint32_t lo[4], hi[4];
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    const uint32_t j = j0 + (uint32_t)u * 32u + (uint32_t)lane;
                    lo[u] = (j < nw) ? __ldg(w0 + j) : 0u;
                    hi[u] = (j < nw) ? __ldg(w0 + j + 1) : 0u;
                }
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    const uint32_t j = j0 + (uint32_t)u * 32u + (uint32_t)lane;
                    if (j < nw) dw[j] = __funnelshift_r(lo[u], hi[u], sh);
                }
            }
            if ((uint32_t)lane < rem) dst[head + nw * 4u + lane] = __ldg(sb + nw * 4u + lane);
        }
    };
    // lines [cur_line, end_line) fit the buffer (whole lines; 8 bytes of slack on either side for the re-aligning copy)
    auto round_end = [&](uint32_t cur_line) {
        const uint32_t cur = s_rel[cur_line];
        uint32_t lo = cur_line + 1, hi = nlines;
        while (lo < hi) {
            const uint32_t mid = (lo + hi + 1) >> 1;
            if (s_rel[mid] - cur <= buf_cap - 32u) lo = mid; else hi = mid - 1;
        }
        return lo;  // (s_rel[nlines] is the block's total: threads past the end hold empty lines)
    };
    __syncthreads();  // s_rel
    if (txt_mode) mbar_wait(&s_bar, 1u);  // the staged text span has landed (every path below may read it, none may leave before)
    uint32_t cur_line = 0, end_line = 0;
    // the block's aggregates are published right away; its first round of lines is composed BEFORE it asks where they go,
    // so the blocks in front have that long to publish theirs (a block cannot leave before every block in front of it has
    // finished lifting: this is what keeps the wait short)
    if (tid == 0) lb_publish(e.lb_bytes, blk, tb);
    if (tid == 32) lb_publish(e.lb_rows, blk, (unsigned long long)tc);
    if (!fast) s_mid[tid].w = 0u;
    if (compose_early && direct) {  // every line at once, side by side without its run; the runs wait for the block's place
        end_line = nlines;
        if (live) compose(s_buf + 16 + rel2);
    } else if (compose_early) {
        end_line = round_end(0);
        if (live && (uint32_t)tid < end_line) compose(s_buf + 16 + (uint32_t)rel);
        if (!fast) {  // (block-uniform)
            __syncthreads();
            copy_mids(0, end_line);
        }
    }
    if (warp == 0) {
        const unsigned long long ex = lb_walk(e.lb_bytes, blk, tb);
        if (lane == 0) s_base[0] = ex;
    } else if (warp == 1) {
        const unsigned long long ex = lb_walk(e.lb_rows, blk, (unsigned long long)tc);
        if (lane == 0) s_base[1] = ex;
    }
    __syncthreads();
    const unsigned long long byte0 = s_base[0], row0 = s_base[1];
    const unsigned long long my_off = byte0 + rel, my_row = row0 + wc + ic - (live ? 1u : 0u);

    if (pend == e.n_pairs && tid == 0) {  // the last block knows the totals
        e.totals[0] = byte0 + tb;
        e.totals[1] = row0 + tc;
        if (e.out_line_off) e.out_line_off[row0 + tc] = byte0 + tb + e.byte_base;
    }
    if (live) {
        if (e.out_line_off) e.out_line_off[my_row] = my_off + e.byte_base;
        if (e.num.q_st) {
            e.num.q_st[my_row] = pr.q_st; e.num.q_en[my_row] = pr.q_en; e.num.t_st[my_row] = pr.t_st; e.num.t_en[my_row] = pr.t_en;
            e.num.nmatch[my_row] = pr.nmatch; e.num.aln_len[my_row] = pr.aln_len;
            e.num.rec_idx[my_row] = e.orig_idx ? e.orig_idx[r] : r + e.rec_base;
            e.num.win_idx[my_row] = e.a.win.bed_row ? e.a.win.bed_row[w] : w;
        }
        if (e.st.equal) write_stats(e.st, my_row, pr.equal, pr.diff, pr.ins, pr.del, pr.ins_ev, pr.del_ev, pr.matches);
    }
    if (!want_text) {
        if (tid == 0) e.blk_flags[blk] = 0u;
        return;
    }
    if (byte0 + tb > e.cap_text) {  // does not fit: totals only, the caller grows the buffer and runs again
        if (tid == 0) { e.blk_flags[blk] = 0u; atomicExch(&e.totals[2], 1ull); }
        return;
    }
    if (!small) {  // a long line in the block: k_serialise's warp-per-line path takes the block's text
        if (in_range) {
            if (fast) e.res[p] = pr;
            e.line_off[p] = my_off; e.out_idx[p] = my_row;
        }
        if (tid == 0) {
            e.line_off[pend] = byte0 + tb;
            e.out_idx[pend] = row0 + tc;
            e.blk_flags[blk] = 1u;
            atomicAdd(&e.totals[3], 1ull);
        }
        return;
    }
    if (tid == 0) e.blk_flags[blk] = 0u;
    if (direct) {  // (block-uniform) the two pieces of every line, a warp per line; then the runs, text -> output, a warp per run
        uint8_t* out0 = e.out_text + byte0;
        for (uint32_t L = (uint32_t)warp; L < nlines; L += SER_LINES / 32) {
            const uint32_t c0 = s_rel2[L], cl = s_rel2[L + 1] - c0;
            if (cl == 0u) continue;
            const uint8_t* src = s_buf + 16 + c0;
            uint8_t* dst = out0 + s_rel[L];
            const uint32_t dw = s_mid[L].w;
            uint32_t hl = cl, skip = 0u;             // one piece ...
            if (dw) { hl = dw >> 16; skip = dw & 0xFFFFu; }  // ... or two with the run in between
            for (uint32_t i = (uint32_t)lane; i < hl; i += 32u) dst[i] = src[i];
            for (uint32_t i = hl + (uint32_t)lane; i < cl; i += 32u) dst[skip + i] = src[i];
        }
        mid_dst0 = out0;
        copy_mids(0, nlines);
        return;
    }
    for (;;) {  // (block-uniform)
        const uint32_t cur = s_rel[cur_line];
        copy_out_shifted(e.out_text + byte0 + cur, s_buf + 16, s_rel[end_line] - cur);
        cur_line = end_line;
        if (cur_line >= nlines) break;
        __syncthreads();  // the buffer is written again
        end_line = round_end(cur_line);
        if (!fast) s_mid[tid].w = 0u;
        if (live && (uint32_t)tid >= cur_line && (uint32_t)tid < end_line) compose(s_buf + 16 + ((uint32_t)rel - s_rel[cur_line]));
        __syncthreads();
        if (!fast) {  // (block-uniform)
            copy_mids(cur_line, end_line);
            __syncthreads();
        }
    }
}

// The long verbatim runs k_serialise deferred (mid_is_big): block (x, y) looks at rows 16x .. 16x + 15 and copies the 64 KB
// segments y, y + gridDim.y, ... of each long run from the input text to its place in the output — 16-byte stores, the source re-aligned with funnel shifts
// (source and destination have unrelated alignments; the text buffer is padded on both sides, so word over-reads stay inside).
constexpr int CM_THREADS = 256;
constexpr uint32_t CM_SEG = 65536;
constexpr uint32_t CM_ROWS = 16;  // rows looked at by one block (a call with many rows and no long run pays one block per 16 rows)
__global__ void __launch_bounds__(CM_THREADS)
k_copy_mid(uint64_t n_pairs, const uint64_t* __restrict__ pair_off, const uint32_t* __restrict__ rec_order, uint32_t n_rec,
           const RecInfo* __restrict__ recs, const PairRes* __restrict__ res, const uint64_t* __restrict__ line_off,
           const uint8_t* __restrict__ text, uint8_t* __restrict__ out_text) {
  for (uint64_t q = (uint64_t)blockIdx.x * CM_ROWS; q < n_pairs && q < ((uint64_t)blockIdx.x + 1) * CM_ROWS; q++) {  // (block-uniform)
    const PairRes& lp = res[q];
    if (lp.kind == PK_DROP || lp.mid_len < MID_BIG) continue;
    const uint32_t k = rank_of_pair(pair_off, n_rec, q);
    const RecInfo& ri = recs[rec_order[k]];
    if (!mid_is_big(ri, lp)) continue;
    const uint64_t llen = line_off[q + 1] - line_off[q];
    const uint64_t hdr = llen - lp.cg_bytes - 1;
    uint8_t* dst0 = out_text + line_off[q] + hdr + (lp.kind == PK_TRIM ? ndigits32(lp.s_len) + 1u : 0u);
    const uint8_t* src0 = text + lp.mid_off;
    for (uint64_t seg = (uint64_t)blockIdx.y * CM_SEG; seg < lp.mid_len; seg += (uint64_t)gridDim.y * CM_SEG) {
        const uint32_t n = (uint32_t)((lp.mid_len - seg < CM_SEG) ? (lp.mid_len - seg) : CM_SEG);
        uint8_t* dst = dst0 + seg;
        const uint8_t* src = src0 + seg;
        const uint32_t head = (uint32_t)((16u - ((uintptr_t)dst & 15u)) & 15u);
        const uint32_t hb = head < n ? head : n;
        const uint32_t nvec = (n - hb) >> 4;
        for (uint32_t i = threadIdx.x; i < hb; i += CM_THREADS) dst[i] = src[i];
        const uint8_t* sb = src + hb;
        const uint32_t sh = (uint32_t)((uintptr_t)sb & 3u) * 8u;
        const uint32_t* w0 = reinterpret_cast<const uint32_t*>((uintptr_t)sb & ~(uintptr_t)3);
        uint4* d4 = reinterpret_cast<uint4*>(dst + hb);
        for (uint32_t v = threadIdx.x; v < nvec; v += CM_THREADS) {
            const uint32_t* w = w0 + (size_t)v * 4;
            const uint32_t a0 = __ldg(w), a1 = __ldg(w + 1), a2 = __ldg(w + 2), a3 = __ldg(w + 3), a4 = __ldg(w + 4);
            uint4 x;
            x.x = __funnelshift_r(a0, a1, sh); x.y = __funnelshift_r(a1, a2, sh); x.z = __funnelshift_r(a2, a3, sh); x.w = __funnelshift_r(a3, a4, sh);
            d4[v] = x;
        }
        for (uint32_t i = hb + (nvec << 4) + threadIdx.x; i < n; i += CM_THREADS) dst[i] = src[i];
    }
  }
}

// rb invert: the CIGAR text of the whole-record rows.  One warp per 32-op chunk of the (already inverted) op array:
// where an op's text starts inside its row is the TXT counter in front of it — the chunk's sample plus a warp scan —
// so 50 M ops are formatted by as many lanes instead of one warp crawling along each 65 k-op row.  Runs after
// k_serialise (which wrote the 12 columns, "cg:Z:" and the newline of every row).
constexpr int WT_THREADS = 256;
__global__ void __launch_bounds__(WT_THREADS)
k_whole_text(const uint32_t* __restrict__ ops, const uint64_t* __restrict__ op_off, uint32_t n_rec, const RecInfo* __restrict__ recs,
             const Ctr* __restrict__ samples, const uint64_t* __restrict__ line_off, uint8_t* __restrict__ out_text) {
    __shared__ uint8_t s_stage[WT_THREADS / 32][32 * 11 + 8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t c = (uint64_t)blockIdx.x * (WT_THREADS / 32) + warp;
    const uint64_t n_ops = op_off[n_rec];
    const uint64_t k0 = c << SAMPLE_LOG2;
    if (k0 >= n_ops) return;
    const uint64_t k1 = (k0 + SAMPLE < n_ops) ? k0 + SAMPLE : n_ops;
    const uint64_t k = k0 + lane;
    auto rec_of = [&](uint64_t op) {  // largest r with op_off[r] <= op (records without ops are skipped over)
        uint32_t lo = 0, hi = n_rec;
        while (lo < hi) {
            const uint32_t mid = lo + ((hi - lo) >> 1);
            if (op_off[mid] <= op) lo = mid + 1; else hi = mid;
        }
        return lo - 1;
    };
    // where the CIGAR of row r starts: the row ends with it and a newline
    auto body_of = [&](uint32_t r) { return line_off[r + 1] - 1 - recs[r].tot.TXT; };
    const uint32_t r0 = rec_of(k0);
    uint32_t w = 0, nb = 0;
    if (k < k1) { w = ops[k]; nb = ndigits32(op_len(w)) + 1u; }
    if (op_off[r0 + 1] >= k1) {  // the whole chunk lies in one record (the usual case)
        uint32_t inc = nb;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, inc, d);
            if (lane >= d) inc += t;
        }
        const uint32_t tot = __shfl_sync(0xffffffffu, inc, 31);
        const uint32_t base = (k0 > op_off[r0]) ? samples[c * SUBS].TXT : 0u;
        if (nb) put_op(&s_stage[warp][inc - nb], op_len(w), op_code(w));
        __syncwarp();
        uint8_t* dst = out_text + body_of(r0) + base;
        for (uint32_t i = lane; i < tot; i += 32) dst[i] = s_stage[warp][i];
        return;
    }
    // a chunk that holds a record boundary: every lane for itself
    if (k >= k1) return;
    const uint32_t r = rec_of(k);
    const uint64_t a = op_off[r];
    uint64_t j = a;
    uint32_t pos = 0;
    if (k0 > a) { j = k0; pos = samples[c * SUBS].TXT; }
    for (; j < k; j++) pos += ndigits32(op_len(ops[j])) + 1u;
    put_op(out_text + body_of(r) + pos, op_len(w), op_code(w));
}

// ------------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------------
static size_t samples2_smem() { return (size_t)(SMP_THREADS * SAMPLE + 9 * SMP_THREADS) * sizeof(uint32_t); }
static size_t scan_lift_smem(bool lift) {
    return (size_t)(SMP_THREADS * (SAMPLE + 1) + 9 * SMP_THREADS + (lift ? 2 * SL_WCAP : 0)) * sizeof(uint32_t);
}
// kernels that ask for more dynamic shared memory than the default limit: once per device (rb_ctx_create, after cudaSetDevice)
int init_kernel_attrs() {
    cudaError_t e = cudaFuncSetAttribute(k_scan_lift<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)scan_lift_smem(true));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_scan_lift<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)scan_lift_smem(false));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_samples2<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)samples2_smem());
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_samples2<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)samples2_smem());
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_samples2<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)samples2_smem());
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_serialise, cudaFuncAttributeMaxDynamicSharedMemorySize, SER_CAP);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_emit<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, EMIT_DYN_BYTES);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_emit<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, EMIT_DYN_BYTES);
    return e == cudaSuccess ? 0 : -1;
}
// line_off[i] += delta (multi-device calls: a device learns where its rows start in the merged text after its kernels ran)
__global__ void k_add_u64(unsigned long long* __restrict__ p, uint64_t n, unsigned long long delta) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] += delta;
}
void launch_add_u64(uint64_t* p, uint64_t n, uint64_t delta, cudaStream_t s) {
    if (n == 0 || delta == 0) return;
    k_add_u64<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(reinterpret_cast<unsigned long long*>(p), n, delta);
}
void launch_whole_text(const uint32_t* ops, const uint64_t* op_off, uint32_t n_rec, const RecInfo* recs, const Ctr* samples,
                       const uint64_t* line_off, uint8_t* out_text, uint64_t n_ops_bound, cudaStream_t s) {
    if (n_rec == 0 || n_ops_bound == 0 || out_text == nullptr) return;
    const uint64_t chunks = (n_ops_bound + SAMPLE - 1) / SAMPLE;
    k_whole_text<<<(unsigned)((chunks + WT_THREADS / 32 - 1) / (WT_THREADS / 32)), WT_THREADS, 0, s>>>(ops, op_off, n_rec, recs, samples,
                                                                                                    line_off, out_text);
}
void launch_tokenise(const uint8_t* text, uint64_t n_tiles, uint32_t* ops, unsigned long long* tile_state, unsigned int* ticket,
                     ErrSlots err, uint32_t* misc_flags, cudaStream_t s) {
    if (n_tiles == 0) return;
    k_tokenise<<<(unsigned)n_tiles, TOK_THREADS, 0, s>>>(text, ops, tile_state, ticket, err, misc_flags);
}
void launch_tok_scan(const uint8_t* text, uint64_t n_tiles, const uint64_t* cigar_off, uint32_t n_rec, uint32_t* ops,
                     unsigned long long* tile_state, unsigned int* ticket, ErrSlots err, uint32_t* misc_flags, uint32_t* tile_first,
                     uint64_t* head_pos, Ctr* samples, uint32_t* seg_state, ScanPayload* seg_agg, ScanPayload* seg_pre, cudaStream_t s) {
    if (n_tiles == 0) return;
    if (n_rec) k_rec_heads<<<(n_rec + 255) / 256, 256, 0, s>>>(text, cigar_off, n_rec, head_pos, tile_first);
    k_tok_scan<<<(unsigned)n_tiles, TOK_THREADS, 0, s>>>(text, ops, tile_state, ticket, err, misc_flags, tile_first, head_pos, n_rec,
                                                         samples, seg_state, seg_agg, seg_pre);
}
void launch_rec_ops(const uint8_t* text, const uint64_t* cigar_off, uint32_t n_rec, const unsigned long long* tile_state,
                    uint64_t* op_off, uint32_t* heads, ErrSlots err, cudaStream_t s) {
    const uint64_t warps = (uint64_t)n_rec + 1;
    k_rec_ops<<<(unsigned)((warps * 32 + 255) / 256), 256, 0, s>>>(text, cigar_off, n_rec, tile_state, op_off, heads, err);
}
void launch_scan_lift(bool lift, const uint32_t* ops, const uint64_t* n_ops_dev, uint64_t n_ops_bound, const uint32_t* heads,
                      Ctr* samples, uint32_t* blk_state, ScanPayload* blk_agg, ScanPayload* blk_pre, unsigned int* ticket,
                      LiftArgs la, cudaStream_t s, bool no_subs) {
    const uint64_t blocks = (n_ops_bound + SMP_OPS - 1) / SMP_OPS;
    if (blocks == 0) return;
    if (lift)
        k_scan_lift<true><<<(unsigned)blocks, SMP_THREADS, scan_lift_smem(true), s>>>(ops, n_ops_dev, heads, samples, blk_state, blk_agg,
                                                                                      blk_pre, ticket, la);
    else if (getenv("RB_OLD_SAMPLES"))
        k_scan_lift<false><<<(unsigned)blocks, SMP_THREADS, scan_lift_smem(false), s>>>(ops, n_ops_dev, heads, samples, blk_state,
                                                                                        blk_agg, blk_pre, ticket, la);
    else if (!getenv("RB_SAMPLES_LOCAL")) {
#if RB_SMP2_LB2
        cudaMemsetAsync(blk_agg, 0, blocks * sizeof(ScanPayload), s);  // the look-back slots of k_samples2 (tags 0 = nothing yet)
#endif
        if (no_subs)
            k_samples2<false, true><<<(unsigned)blocks, SMP_THREADS, samples2_smem(), s>>>(ops, n_ops_dev, heads, samples, blk_state, blk_agg, blk_pre,
                                                                                           ticket, 1u);
        else
            k_samples2<false><<<(unsigned)blocks, SMP_THREADS, samples2_smem(), s>>>(ops, n_ops_dev, heads, samples, blk_state, blk_agg, blk_pre, ticket,
                                                                                     0u);
    } else {  // (measured, not faster: 0.24 + 0.06 + 0.07 ms against 0.31 ms at C4) block-local samples + aggregates, a one-block
            // scan of the aggregates, the prefixes added to the incomplete samples
        k_samples2<true><<<(unsigned)blocks, SMP_THREADS, samples2_smem(), s>>>(ops, n_ops_dev, heads, samples, blk_state, blk_agg, blk_pre, ticket, 0u);
        k_blk_scan<<<1, 1024, 0, s>>>(n_ops_dev, blk_agg, blk_pre);
        const uint64_t chunks = (n_ops_bound + SAMPLE - 1) / SAMPLE;
        k_smp_fix<<<(unsigned)((chunks + 255) / 256), 256, 0, s>>>(n_ops_dev, blk_pre, samples);
    }
}
void launch_combine(uint64_t n_pairs, const uint64_t* pair_off, const uint32_t* rec_order, uint32_t n_rec, const RecInfo* recs,
                    const uint32_t* ops, WinView win, const uint64_t* names_off, const HalfS* hs, const HalfE* he, PairRes* res,
                    uint32_t* line_len, ErrSlots err, cudaStream_t s) {
    if (n_pairs == 0) return;
    k_combine<<<(unsigned)((n_pairs + 127) / 128), 128, 0, s>>>(n_pairs, pair_off, rec_order, n_rec, recs, ops, win, names_off, hs, he,
                                                                res, line_len, err);
}
void launch_check_clips(const uint32_t* ops, const uint64_t* op_off, uint32_t n_rec, ErrSlots err, cudaStream_t s) {
    if (n_rec == 0) return;
    k_check_clips<<<(n_rec + 127) / 128, 128, 0, s>>>(ops, op_off, n_rec, err);
}
void launch_rec_prep(int mode, RecInput in, const uint64_t* op_off, const uint32_t* ops, const Ctr* samples, WinView win,
                     RecInfo* recs, uint32_t* pair_cnt, StatsDev st, ErrSlots err, cudaStream_t s) {
    if (in.n_rec == 0) return;
    k_rec_prep<<<(in.n_rec + 127) / 128, 128, 0, s>>>(mode, in, op_off, ops, samples, win, recs, pair_cnt, st, err);
}
void launch_whole_rows(uint32_t n_rec, const RecInfo* recs, PairRes* res, uint32_t* line_len, uint64_t* pair_off, LiftPlan* plans,
                       cudaStream_t s) {
    k_whole_rows<<<n_rec / 128 + 1, 128, 0, s>>>(n_rec, recs, res, line_len, pair_off, plans);
}
void launch_pair_scan(const uint32_t* pair_cnt, const uint32_t* rec_order, uint32_t n_rec, uint64_t* pair_off, cudaStream_t s) {
    k_pair_scan<<<1, 1024, 0, s>>>(pair_cnt, rec_order, n_rec, pair_off);
}
void launch_lift_plan(uint64_t n_pairs, const uint64_t* pair_off, const uint32_t* rec_order, uint32_t n_rec, const RecInfo* recs,
                      const Ctr* samples, WinView win, LiftPlan* plans, cudaStream_t s, bool mark_fast) {
    if (n_pairs == 0) return;
    const uint32_t nb = (uint32_t)((n_pairs + LIFT_THREADS - 1) / LIFT_THREADS);
    k_lift_plan<<<(nb + 127) / 128, 128, 0, s>>>(n_pairs, nb, pair_off, rec_order, n_rec, recs, samples, win, plans, mark_fast ? 1u : 0u);
}
void launch_lift(uint64_t n_pairs, const uint64_t* pair_off, const uint32_t* rec_order, uint32_t n_rec, const RecInfo* recs,
                 const uint32_t* ops, const Ctr* samples, WinView win, const uint64_t* names_off, int policy, const LiftPlan* plans,
                 PairRes* res, uint32_t* line_len, ErrSlots err, cudaStream_t s, bool skip_fast, bool wide) {
    if (n_pairs == 0) return;
    const unsigned grid = (unsigned)((n_pairs + LIFT_THREADS - 1) / LIFT_THREADS);
    if (wide)
        k_lift<false><<<grid, LIFT_THREADS, 0, s>>>(n_pairs, pair_off, rec_order, n_rec, recs, ops, samples, win, names_off, policy, plans, res,
                                                    line_len, err, skip_fast ? 1u : 0u);
    else
        k_lift<true><<<grid, LIFT_THREADS, 0, s>>>(n_pairs, pair_off, rec_order, n_rec, recs, ops, samples, win, names_off, policy, plans, res,
                                                   line_len, err, skip_fast ? 1u : 0u);
}
void launch_scan_lines(const uint32_t* line_len, uint64_t n, uint64_t* line_off, uint64_t* out_idx, uint32_t* blk_state,
                       ulonglong2* blk_agg, ulonglong2* blk_pre, unsigned int* ticket, cudaStream_t s) {
    const uint64_t tiles = n ? (n + LNS_TILE - 1) / LNS_TILE : 1;
    const uint64_t blocks = tiles < (uint64_t)LNS_MAX_BLOCKS ? tiles : (uint64_t)LNS_MAX_BLOCKS;
    const uint64_t span = (tiles + blocks - 1) / blocks * LNS_TILE;  // whole tiles per block
    const uint64_t used = n ? (n + span - 1) / span : 1;              // blocks that own at least one item
    k_scan_lines<<<(unsigned)used, LNS_THREADS, 0, s>>>(line_len, n, span, line_off, out_idx, blk_state, blk_agg, blk_pre, ticket);
}
void launch_serialise(uint64_t n_pairs, const uint64_t* pair_off, const uint32_t* rec_order, uint32_t n_rec, const RecInfo* recs,
                      const uint32_t* ops, const uint8_t* text, WinView win, const uint64_t* names_off, const uint8_t* names,
                      const LiftPlan* plans, const PairRes* res, const uint64_t* line_off, const uint64_t* out_idx, uint8_t* out_text,
                      uint64_t* out_line_off, NumDev num, StatsDev st, uint64_t byte_base, uint32_t rec_base, const uint32_t* orig_idx,
                      uint32_t group, uint32_t defer_big, cudaStream_t s, const uint32_t* only_flagged) {
    if (n_pairs == 0) return;
    OpsView view;
    view.ops = ops; view.samples = nullptr;
    SerArgs a{recs, view, win, names_off, names, text};
    if (group == 0 || group > (uint32_t)SER_LINES || (SER_LINES % group)) group = SER_LINES;
    k_serialise<<<(unsigned)((n_pairs + group - 1) / group), SER_LINES, SER_CAP, s>>>(
        n_pairs, pair_off, rec_order, n_rec, a, plans, res, line_off, out_idx, out_text, out_line_off, num, st, byte_base, rec_base, orig_idx, group,
        defer_big, only_flagged);
}
void launch_emit(uint64_t n_pairs, const uint64_t* pair_off, const uint32_t* rec_order, uint32_t n_rec, const RecInfo* recs,
                 const uint32_t* ops, const Ctr* samples, const uint8_t* text, WinView win, const uint64_t* names_off, const uint8_t* names,
                 const LiftPlan* plans, PairRes* res, const uint32_t* line_len, uint64_t* line_off, uint64_t* out_idx,
                 uint32_t* blk_flags, uint8_t* out_text, uint64_t cap_text, uint64_t* out_line_off, NumDev num, StatsDev st,
                 uint64_t byte_base, uint32_t rec_base, const uint32_t* orig_idx, unsigned long long* lb_bytes,
                 unsigned long long* lb_rows, unsigned int* ticket, unsigned long long* totals, ErrSlots err, cudaStream_t s,
                 bool stats_text, bool wide) {
    if (n_pairs == 0) return;
    OpsView view;
    view.ops = ops; view.samples = samples;
    EmitArgs e{};
    e.n_pairs = n_pairs; e.pair_off = pair_off; e.rec_order = rec_order; e.n_rec = n_rec;
    e.a = SerArgs{recs, view, win, names_off, names, text};
    e.plans = plans; e.res = res; e.line_len = line_len; e.line_off = line_off; e.out_idx = out_idx; e.blk_flags = blk_flags;
    e.out_text = out_text; e.cap_text = cap_text; e.out_line_off = out_line_off; e.num = num; e.st = st;
    e.byte_base = byte_base; e.rec_base = rec_base; e.orig_idx = orig_idx;
    e.lb_bytes = lb_bytes; e.lb_rows = lb_rows; e.ticket = ticket; e.totals = totals; e.err = err;
    e.stats_text = stats_text ? 1u : 0u;
    e.dyn_bytes = (uint32_t)(wide ? EMIT_DYN_WIDE : EMIT_DYN_BYTES);  // wide: the caller's plan marked no block PLAN_FAST
    if (stats_text) k_emit<true><<<(unsigned)((n_pairs + SER_LINES - 1) / SER_LINES), SER_LINES, e.dyn_bytes, s>>>(e);
    else k_emit<false><<<(unsigned)((n_pairs + SER_LINES - 1) / SER_LINES), SER_LINES, e.dyn_bytes, s>>>(e);
}
void launch_copy_mid(uint64_t n_pairs, const uint64_t* pair_off, const uint32_t* rec_order, uint32_t n_rec, const RecInfo* recs,
                     const PairRes* res, const uint64_t* line_off, const uint8_t* text, uint8_t* out_text, uint32_t seg_y, cudaStream_t s) {
    if (n_pairs == 0 || n_pairs > 0x7FFFFFFFull) return;
    if (seg_y < 1u) seg_y = 1u;
    if (seg_y > 64u) seg_y = 64u;
    k_copy_mid<<<dim3((unsigned)((n_pairs + CM_ROWS - 1) / CM_ROWS), seg_y), CM_THREADS, 0, s>>>(n_pairs, pair_off, rec_order, n_rec, recs, res, line_off, text, out_text);
}
// ------------------------------------------------------------------------------------------------
// rb break-paf: windows from the record's own large indels (liftover.rs:182-226)
// ------------------------------------------------------------------------------------------------
// thread per 32-op chunk.  FILL == false: number of break ops (I / D longer than max_size, inside the stripped op range)
// of the chunk.  FILL == true: for break op number b (global, in op order) the target position where the piece in front
// of it ends (cur_tpos) and where the next piece starts (pre_tpos); per record the index of its first / one past its
// last break op.
template <bool FILL>
__global__ void __launch_bounds__(256)
k_break_scan(const uint32_t* __restrict__ ops, const uint64_t* __restrict__ n_ops_dev, const uint32_t* __restrict__ heads,
             const Ctr* __restrict__ samples, const uint64_t* __restrict__ op_off, uint32_t n_rec, const RecInfo* __restrict__ recs,
             uint32_t max_size, uint32_t* __restrict__ cnt, const uint64_t* __restrict__ bp_off, uint64_t* __restrict__ bp_end,
             uint64_t* __restrict__ bp_next, uint64_t* __restrict__ rec_bp0, uint64_t* __restrict__ rec_bp1) {
    const uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t n_ops = *n_ops_dev;
    const uint64_t first = c << SAMPLE_LOG2;
    if (first >= n_ops) return;
    const int nvalid = (n_ops - first) < SAMPLE ? (int)(n_ops - first) : (int)SAMPLE;
    const uint32_t h = (uint32_t)((heads[first >> 5] >> (first & 31u)) & (uint32_t)((1ull << SAMPLE) - 1ull));
    uint32_t r;  // record that holds op `first`: largest r with op_off[r] <= first
    {
        uint32_t lo = 0, hi = n_rec;
        while (lo < hi) {
            const uint32_t mid = lo + ((hi - lo) >> 1);
            if (op_off[mid] <= first) lo = mid + 1; else hi = mid;
        }
        r = lo ? lo - 1 : 0u;
    }
    uint64_t T = (h & 1u) ? 0ull : (uint64_t)samples[c * SUBS].T;  // target bases of the record before op `first`
    uint64_t eo0 = 0, eo1 = 0, t_st = 0, op_end = 0;
    auto load_rec = [&]() {
        if (r < n_rec) { const RecInfo& R = recs[r]; eo0 = R.eo0; eo1 = R.eo1; t_st = R.t_st; op_end = R.op_end; }
        else { eo0 = eo1 = 0; op_end = 0; }
    };
    load_rec();
    uint32_t local = 0;
    const uint64_t b0 = FILL ? bp_off[c] : 0ull;
    for (int j = 0; j < nvalid; j++) {
        const uint64_t k = first + (uint64_t)j;
        if ((h >> j) & 1u) {  // a record starts at op k
            if (j > 0) { r++; load_rec(); }
            T = 0;
            if (FILL && r < n_rec) rec_bp0[r] = b0 + local;
        }
        const uint32_t w = ops[k];
        const uint32_t code = op_code(w), len = op_len(w);
        if (k >= eo0 && k < eo1 && (code == OP_I || code == OP_D) && len > max_size) {
            if (FILL) {
                bp_end[b0 + local] = t_st + T;                                     // cur_tpos when the break op is met
                bp_next[b0 + local] = t_st + T + (code == OP_D ? (uint64_t)len : 0ull);  // pre_tpos after it
            }
            local++;
        }
        if (is_ref(code)) T += len;
        if (FILL && k + 1 == op_end && r < n_rec) rec_bp1[r] = b0 + local;
    }
    if (!FILL) cnt[c] = local;
}

// thread per record: its window range [wlo, whi) (one window more than it has break ops) and the windows themselves
__global__ void __launch_bounds__(128)
k_break_recs(uint32_t n_rec, RecInfo* __restrict__ recs, const uint64_t* __restrict__ rec_bp0, const uint64_t* __restrict__ rec_bp1,
             const uint64_t* __restrict__ bp_end, const uint64_t* __restrict__ bp_next, uint64_t* __restrict__ w_st,
             uint64_t* __restrict__ w_en, uint32_t* __restrict__ pair_cnt) {
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rec) return;
    const uint64_t B0 = rec_bp0[r], B1 = rec_bp1[r];
    if (B0 == ~0ull || B1 == ~0ull || B1 < B0) {  // a record without ops: the call fails in the strip check anyway
        recs[r].wlo = recs[r].whi = 0;
        pair_cnt[r] = 0;
        return;
    }
    const uint64_t nb = B1 - B0;
    const uint64_t wlo = B0 + r;  // every earlier record owns one window more than it has break ops
    const uint64_t t_st = recs[r].t_st, t_en = recs[r].t_en;
    for (uint64_t j = 0; j <= nb; j++) {
        w_st[wlo + j] = j ? bp_next[B0 + j - 1] : t_st;
        w_en[wlo + j] = (j < nb) ? bp_end[B0 + j] : t_en;
    }
    recs[r].wlo = (uint32_t)wlo;
    recs[r].whi = (uint32_t)(wlo + nb + 1);
    pair_cnt[r] = (uint32_t)(nb + 1);
}

void launch_break_scan(bool fill, const uint32_t* ops, const uint64_t* n_ops_dev, uint64_t n_ops_bound, const uint32_t* heads,
                       const Ctr* samples, const uint64_t* op_off, uint32_t n_rec, const RecInfo* recs, uint32_t max_size,
                       uint32_t* cnt, const uint64_t* bp_off, uint64_t* bp_end, uint64_t* bp_next, uint64_t* rec_bp0, uint64_t* rec_bp1,
                       cudaStream_t s) {
    const uint64_t chunks = (n_ops_bound + SAMPLE - 1) / SAMPLE;
    if (chunks == 0) return;
    const unsigned blocks = (unsigned)((chunks + 255) / 256);
    if (fill) k_break_scan<true><<<blocks, 256, 0, s>>>(ops, n_ops_dev, heads, samples, op_off, n_rec, recs, max_size, cnt, bp_off, bp_end, bp_next, rec_bp0, rec_bp1);
    else k_break_scan<false><<<blocks, 256, 0, s>>>(ops, n_ops_dev, heads, samples, op_off, n_rec, recs, max_size, cnt, bp_off, bp_end, bp_next, rec_bp0, rec_bp1);
}
void launch_break_recs(uint32_t n_rec, RecInfo* recs, const uint64_t* rec_bp0, const uint64_t* rec_bp1, const uint64_t* bp_end,
                       const uint64_t* bp_next, uint64_t* w_st, uint64_t* w_en, uint32_t* pair_cnt, cudaStream_t s) {
    if (n_rec == 0) return;
    k_break_recs<<<(n_rec + 127) / 128, 128, 0, s>>>(n_rec, recs, rec_bp0, rec_bp1, bp_end, bp_next, w_st, w_en, pair_cnt);
}

// Device scalars -> mapped pinned host memory with plain SM stores: the host reads them after a stream sync.  (A
// cudaMemcpyAsync would queue on the device->host DMA engine behind the bulk download of the previous slice.)
__global__ void k_publish(PublishArgs a) {
    if (threadIdx.x < (unsigned)a.n) {
        const int i = threadIdx.x;
        a.dst[a.slot[i]] = a.wide[i] ? *reinterpret_cast<const unsigned long long*>(a.src[i])
                                     : (unsigned long long)*reinterpret_cast<const uint32_t*>(a.src[i]);
        __threadfence_system();
    }
}
void launch_publish(const PublishArgs& a, cudaStream_t s) { k_publish<<<1, 32, 0, s>>>(a); }
void launch_win_check(const uint32_t* t_id, const uint64_t* st, const uint64_t* en, const uint32_t* row, uint32_t n_win,
                      uint32_t n_names, uint32_t* flags, cudaStream_t s) {
    if (n_win == 0) return;
    const unsigned blocks = (unsigned)std::min<uint64_t>(((uint64_t)n_win + 255) / 256, 148 * 8);
    k_win_check<<<blocks, 256, 0, s>>>(t_id, st, en, row, n_win, n_names, flags);
}
void launch_pair_count_bf(const RecInfo* recs, uint32_t n_rec, WinView win, uint32_t* pair_cnt, cudaStream_t s) {
    if (n_rec == 0) return;
    k_pair_count_bf<<<n_rec, 256, 0, s>>>(recs, n_rec, win, pair_cnt);
}
void launch_pair_fill_bf(const RecInfo* recs, const uint32_t* rec_rank, uint32_t n_rec, WinView win,
                         const uint64_t* pair_off, uint32_t* pair_win, cudaStream_t s) {
    if (n_rec == 0) return;
    k_pair_fill_bf<<<n_rec, 256, 0, s>>>(recs, rec_rank, n_rec, win, pair_off, pair_win);
}

}  // namespace rb
