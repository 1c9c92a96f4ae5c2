// paf_parse_kernels.cu — PAF text -> the device layout of a resident batch (rb_batch_upload_paf), the rules of
// paf_parse_core.cuh applied on the GPU:
//
//   k_paf_lines_count  per 64 KiB of text: '\n' count (16-byte loads, per-byte masks, popcount, warp sums) and, per 4 KiB
//                      tile, whether it holds any whitespace byte at all (also BED line starts: bed_parse_kernels.cu)
//   k_paf_scan_*       exclusive scans (reduce -> scan of the block sums -> scan down) of up to three u64 columns at once
//   k_paf_lines_fill   line start offsets: the newline of rank k starts line k + 1
//   k_paf_fields       one warp per line: tokens, the tag test of every extra token, the first cg payload, the numeric columns
//                      and the line's state (paf_parse_core.cuh: line_finish)
//   k_paf_pack         kept lines -> record columns (cols64 SoA, strand, cigar_off) and the q/t name bytes of each record
//   k_paf_copy_cg      the cg payloads -> the batch's CIGAR text (16 destination bytes per thread)
//
// Only the bytes of a line's first tokens are read one by one (by the whole warp at once: the lanes read the same address).  A
// long token — the cg payload of a whole-genome record is MBs, a cs tag as long — is searched for its end 512 bytes per warp
// step, and 4 KiB tiles that hold no whitespace at all (k_paf_lines_count's flags) are stepped over 32 at a time, so a
// megabyte of CIGAR costs its line a few dozen warp steps, whatever the line's length.
#include <algorithm>
#include <cstdint>

#include "bed_parse_core.cuh"
#include "paf_parse_core.cuh"
#include "rb_kernels.cuh"

namespace rb {

namespace {

constexpr int PP_THREADS = 256;
constexpr uint64_t PP_CHUNK = 64 * 1024;  // text bytes per k_paf_lines_* block
constexpr int PP_TILE_SHIFT = 12;         // 4 KiB whitespace tiles
constexpr int SCAN_ITEMS = 8;             // elements per thread of the scan kernels
constexpr uint64_t SCAN_CH = (uint64_t)PP_THREADS * SCAN_ITEMS;
constexpr unsigned FULL = 0xFFFFFFFFu;

// per-byte masks of 16 bytes: bit j = byte j is '\n' / is whitespace
__device__ __forceinline__ void masks16(const uint4 w, uint32_t& nl, uint32_t& ws) {
    nl = 0; ws = 0;
    const uint32_t wd[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
    for (int k = 0; k < 4; k++)
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const uint8_t c = (uint8_t)(wd[k] >> (8 * j));
            nl |= (uint32_t)(c == '\n') << (4 * k + j);
            ws |= (uint32_t)rbpp::is_ws(c) << (4 * k + j);
        }
}

__device__ __forceinline__ uint4 load16(const uint8_t* text, uint64_t pos, uint64_t n) {
    if (pos + 16 <= n) return *reinterpret_cast<const uint4*>(text + pos);
    uint8_t b[16];
#pragma unroll
    for (int j = 0; j < 16; j++) b[j] = pos + j < n ? text[pos + j] : (uint8_t)'x';  // (past the end: neither '\n' nor whitespace)
    uint4 w;
    w.x = b[0] | (b[1] << 8) | (b[2] << 16) | ((uint32_t)b[3] << 24);
    w.y = b[4] | (b[5] << 8) | (b[6] << 16) | ((uint32_t)b[7] << 24);
    w.z = b[8] | (b[9] << 8) | (b[10] << 16) | ((uint32_t)b[11] << 24);
    w.w = b[12] | (b[13] << 8) | (b[14] << 16) | ((uint32_t)b[15] << 24);
    return w;
}

__device__ __forceinline__ unsigned long long warp_min_u64(unsigned long long v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        const unsigned long long w = __shfl_xor_sync(FULL, v, o);
        v = w < v ? w : v;
    }
    return v;
}

// block-wide exclusive scan of one u64 per thread (PP_THREADS threads); returns the block total through `total`
__device__ __forceinline__ uint64_t block_excl_scan(uint64_t v, uint64_t* sh, uint64_t& total) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    uint64_t x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint64_t y = __shfl_up_sync(FULL, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) sh[w] = x;
    __syncthreads();
    if (w == 0) {
        uint64_t s = lane < PP_THREADS / 32 ? sh[lane] : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint64_t y = __shfl_up_sync(FULL, s, o);
            if (lane >= o) s += y;
        }
        if (lane < PP_THREADS / 32) sh[lane] = s;
    }
    __syncthreads();
    total = sh[PP_THREADS / 32 - 1];
    const uint64_t before = w ? sh[w - 1] : 0;
    __syncthreads();
    return before + x - v;
}

}  // namespace

// Line starts, for two definitions of a line (the template parameter):
//   LINES_PAF  a line ends at each '\n' (paf.rs lines()): the newline of rank k starts line k + 1, line 0 starts at 0; the count
//              pass also flags the 4 KiB tiles that hold any whitespace byte and reads the last byte of the text
//   LINES_BED  a line starts at a byte that is neither '\n' nor '\r' at offset 0 or right after one of them (bio's BED reader: a
//              run of line ends is one separator, there are no empty lines); start of rank k starts line k
enum : int { LINES_PAF = 0, LINES_BED = 1 };

// bit j: a mark at pos + j (LINES_PAF: a '\n'; LINES_BED: a line start), ws = whitespace bits (LINES_PAF only)
template <int MODE>
__device__ __forceinline__ uint32_t line_marks(const uint8_t* text, uint64_t pos, uint64_t n, uint32_t& ws) {
    uint32_t nl;
    const uint4 w = load16(text, pos, n);
    masks16(w, nl, ws);
    if (MODE == LINES_PAF) return nl;
    const uint32_t wd[4] = {w.x, w.y, w.z, w.w};
    uint32_t eol = 0;
#pragma unroll
    for (int k = 0; k < 4; k++)
#pragma unroll
        for (int j = 0; j < 4; j++) eol |= (uint32_t)rbbp::is_eol((uint8_t)(wd[k] >> (8 * j))) << (4 * k + j);
    const uint32_t prev_eol = pos == 0 || rbbp::is_eol(text[pos - 1]) ? 1u : 0u;
    uint32_t st = ~eol & ((eol << 1) | prev_eol) & 0xFFFFu;
    if (pos + 16 > n) st &= (1u << (n - pos)) - 1;  // (load16 pads with non-EOL bytes)
    return st;
}

template <int MODE>
__global__ void __launch_bounds__(PP_THREADS) k_paf_lines_count(const uint8_t* text, uint64_t n, uint64_t* chunk_cnt, uint8_t* tile_ws,
                                                             uint32_t* last_byte) {
    const uint64_t c0 = (uint64_t)blockIdx.x * PP_CHUNK;
    uint32_t cnt = 0;
    for (uint64_t t0 = c0; t0 < c0 + PP_CHUNK && t0 < n; t0 += PP_THREADS * 16) {
        const uint64_t pos = t0 + threadIdx.x * 16;
        uint32_t m = 0, ws = 0;
        if (pos < n) m = line_marks<MODE>(text, pos, n, ws);
        cnt += __popc(m);
        if (MODE == LINES_PAF) {
            const int any = __syncthreads_or(ws != 0);
            if (threadIdx.x == 0) tile_ws[t0 >> PP_TILE_SHIFT] = (uint8_t)any;
        }
    }
    cnt = __reduce_add_sync(FULL, cnt);
    __shared__ uint32_t sh[PP_THREADS / 32];
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t s = 0;
        for (int k = 0; k < PP_THREADS / 32; k++) s += sh[k];
        chunk_cnt[blockIdx.x] = s;
        if (MODE == LINES_PAF && n && c0 <= n - 1 && n - 1 < c0 + PP_CHUNK) *last_byte = text[n - 1];
    }
}

// chunk_off = exclusive scan of the chunk counts
template <int MODE>
__global__ void __launch_bounds__(PP_THREADS) k_paf_lines_fill(const uint8_t* text, uint64_t n, const uint64_t* chunk_off, uint64_t* line_start) {
    __shared__ uint64_t sh[PP_THREADS / 32];
    const uint64_t c0 = (uint64_t)blockIdx.x * PP_CHUNK;
    uint64_t carry = chunk_off[blockIdx.x];
    if (MODE == LINES_PAF && blockIdx.x == 0 && threadIdx.x == 0) line_start[0] = 0;
    for (uint64_t t0 = c0; t0 < c0 + PP_CHUNK && t0 < n; t0 += PP_THREADS * 16) {
        const uint64_t pos = t0 + threadIdx.x * 16;
        uint32_t m = 0, ws = 0;
        if (pos < n) m = line_marks<MODE>(text, pos, n, ws);
        uint64_t tot;
        uint64_t k = carry + block_excl_scan(__popc(m), sh, tot);
        while (m) {
            const int j = __ffs(m) - 1;
            m &= m - 1;
            if (MODE == LINES_PAF) line_start[++k] = pos + j + 1;
            else line_start[k++] = pos + j;
        }
        carry += tot;
    }
}

// exclusive scans of nv (<= 3) u64 columns: in[v][0 .. n) -> out[v][0 .. n], out[v][n] = the total
struct ScanCols {
    const uint64_t* in[3];
    uint64_t* out[3];
    int nv;
};

__global__ void __launch_bounds__(PP_THREADS) k_paf_scan_reduce(ScanCols c, uint64_t n, uint64_t* part, uint64_t nb) {
    __shared__ uint64_t sh[PP_THREADS / 32];
    const uint64_t i0 = (uint64_t)blockIdx.x * SCAN_CH + threadIdx.x * SCAN_ITEMS;
    for (int v = 0; v < c.nv; v++) {
        uint64_t s = 0;
#pragma unroll
        for (int k = 0; k < SCAN_ITEMS; k++)
            if (i0 + k < n) s += c.in[v][i0 + k];
        uint64_t tot;
        block_excl_scan(s, sh, tot);
        if (threadIdx.x == 0) part[v * nb + blockIdx.x] = tot;
    }
}

__global__ void __launch_bounds__(PP_THREADS) k_paf_scan_parts(ScanCols c, uint64_t n, uint64_t* part, uint64_t nb) {
    __shared__ uint64_t sh[PP_THREADS / 32];
    for (int v = 0; v < c.nv; v++) {
        uint64_t carry = 0;
        for (uint64_t b0 = 0; b0 < nb; b0 += PP_THREADS) {
            const uint64_t b = b0 + threadIdx.x;
            const uint64_t x = b < nb ? part[v * nb + b] : 0;
            uint64_t tot;
            const uint64_t ex = block_excl_scan(x, sh, tot);
            if (b < nb) part[v * nb + b] = carry + ex;
            carry += tot;
        }
        if (threadIdx.x == 0) c.out[v][n] = carry;
    }
}

__global__ void __launch_bounds__(PP_THREADS) k_paf_scan_down(ScanCols c, uint64_t n, const uint64_t* part, uint64_t nb) {
    __shared__ uint64_t sh[PP_THREADS / 32];
    const uint64_t i0 = (uint64_t)blockIdx.x * SCAN_CH + threadIdx.x * SCAN_ITEMS;
    for (int v = 0; v < c.nv; v++) {
        uint64_t x[SCAN_ITEMS], s = 0;
#pragma unroll
        for (int k = 0; k < SCAN_ITEMS; k++) {
            x[k] = i0 + k < n ? c.in[v][i0 + k] : 0;
            s += x[k];
        }
        uint64_t tot;
        uint64_t run = part[v * nb + blockIdx.x] + block_excl_scan(s, sh, tot);
#pragma unroll
        for (int k = 0; k < SCAN_ITEMS; k++)
            if (i0 + k < n) { c.out[v][i0 + k] = run; run += x[k]; }
    }
}

namespace {

// first position in [p, e) whose byte is (WS: whitespace / !WS: not whitespace), else e; every lane gets the answer.
// 32 bytes are tried by the whole warp in step (one address per load), then 512 bytes per step, 16 per lane; the whitespace
// search steps over 4 KiB tiles without any whitespace byte 32 tiles at a time.
template <bool WS>
__device__ uint64_t warp_find(const uint8_t* text, uint64_t p, uint64_t e, const uint8_t* tile_ws, int lane) {
    const uint64_t lim = e - p > 32 ? p + 32 : e;
    uint64_t q = p;
    for (; q < lim; q++)
        if (rbpp::is_ws(text[q]) == WS) return q;
    if (q >= e) return e;
    uint64_t base = q & ~15ull;
    const uint64_t last_tile = (e - 1) >> PP_TILE_SHIFT;
    while (base < e) {
        if (WS) {
            const uint64_t t0 = base >> PP_TILE_SHIFT;
            const bool stop = t0 + lane > last_tile || tile_ws[t0 + lane] != 0;
            const unsigned m = __ballot_sync(FULL, stop);
            if (m == 0) { base = (t0 + 32) << PP_TILE_SHIFT; continue; }
            const uint64_t tf = t0 + (uint64_t)(__ffs(m) - 1);
            if (tf > t0) base = tf << PP_TILE_SHIFT;
        }
        const uint64_t pos = base + (uint64_t)lane * 16;
        unsigned long long hit = ~0ull;
        if (pos < e) {
            uint32_t nl, ws;
            masks16(*reinterpret_cast<const uint4*>(text + pos), nl, ws);
            uint32_t m = WS ? ws : (~ws & 0xFFFFu);
            if (pos < q) m &= ~0u << (q - pos);
            if (m) {
                const uint64_t at = pos + (uint64_t)(__ffs(m) - 1);
                if (at < e) hit = at;
            }
        }
        hit = warp_min_u64(hit);
        if (hit != ~0ull) return hit;
        base += 512;
    }
    return e;
}

// offset of the first PAF_TAG match in the token [p, p + tn), tn if there is none
__device__ uint64_t warp_tag(const uint8_t* text, uint64_t p, uint64_t tn, int lane) {
    const uint8_t* tok = text + p;
    for (uint64_t a = 0; a < 8 && a + 5 <= tn; a++)
        if (rbpp::tag_at(tok, a, tn)) return a;
    for (uint64_t a0 = 8; a0 + 5 <= tn; a0 += 512) {
        unsigned long long hit = ~0ull;
        for (uint64_t a = a0 + (uint64_t)lane * 16; a < a0 + (uint64_t)lane * 16 + 16; a++)
            if (rbpp::tag_at(tok, a, tn)) { hit = a; break; }
        hit = warp_min_u64(hit);
        if (hit != ~0ull) return hit;
    }
    return tn;
}

}  // namespace

__global__ void __launch_bounds__(PP_THREADS) k_paf_fields(const uint8_t* text, const uint64_t* line_start, uint64_t n_lines,
                                                            const uint8_t* tile_ws, PafLineCols L, unsigned long long* first_panic) {
    const int lane = threadIdx.x & 31;
    const uint64_t warps = (uint64_t)gridDim.x * (PP_THREADS / 32);
    for (uint64_t i = (uint64_t)blockIdx.x * (PP_THREADS / 32) + (threadIdx.x >> 5); i < n_lines; i += warps) {
        const uint64_t b = line_start[i];
        uint64_t e = line_start[i + 1] - 1;
        if (e > b && text[e - 1] == '\r') e--;
        uint64_t tok_off[12], tok_len[12];
        uint32_t n_tok = 0;
        bool bad_tag = false, has_cg = false;
        uint64_t cg_off = 0, cg_len = 0;
        uint64_t p = b;
        for (;;) {
            p = warp_find<false>(text, p, e, tile_ws, lane);
            if (p >= e) break;
            const uint64_t q = warp_find<true>(text, p, e, tile_ws, lane);
            if (n_tok < 12) {
                tok_off[n_tok] = p; tok_len[n_tok] = q - p; n_tok++;
            } else {
                const uint64_t tn = q - p, m = warp_tag(text, p, tn, lane);
                if (m == tn) { bad_tag = true; break; }  // (the reference stops at the first bad tag)
                if (cg_len == 0 && text[p + m] == 'c' && text[p + m + 1] == 'g') { has_cg = true; cg_off = p + m + 5; cg_len = tn - (m + 5); }
            }
            p = q;
        }
        if (lane == 0) {
            rbpp::LineOut o;
            rbpp::line_finish(text, tok_off, tok_len, n_tok, bad_tag, has_cg, cg_off, cg_len, o);
            L.state[i] = o.state;
            const bool kept = o.state == rbpp::LS_OK;
            L.keep[i] = kept ? 1 : 0;
            L.cg_len[i] = kept ? o.cg_len : 0;
            L.name_len[i] = kept ? (uint64_t)o.qn_len + o.tn_len : 0;
            if (kept) {
#pragma unroll
                for (int k = 0; k < 7; k++) L.v[k * n_lines + i] = o.v[k];
                L.strand[i] = o.strand;
                L.qn_off[i] = o.qn_off; L.tn_off[i] = o.tn_off; L.cg_off[i] = o.cg_off;
                L.qn_len[i] = o.qn_len;
            }
            if (o.state >= rbpp::LS_FEW_COLUMNS) atomicMin(first_panic, ((unsigned long long)i << 8) | o.state);
        }
    }
}

// one thread per line: the kept ones become record rec_idx[i]
__global__ void __launch_bounds__(PP_THREADS) k_paf_pack(const uint8_t* text, uint64_t n_lines, PafLineCols L, const uint64_t* rec_idx,
                                                          const uint64_t* cg_pos, const uint64_t* name_pos, uint32_t n_rec, uint64_t* cols64,
                                                          uint8_t* strand, uint64_t* cigar_off, uint32_t* rec_line, uint8_t* names,
                                                          uint64_t* rec_name_off, uint32_t* rec_qlen) {
    const uint64_t i = (uint64_t)blockIdx.x * PP_THREADS + threadIdx.x;
    if (i == 0) { cigar_off[n_rec] = cg_pos[n_lines]; rec_name_off[n_rec] = name_pos[n_lines]; }
    if (i >= n_lines || !L.keep[i]) return;
    const uint64_t r = rec_idx[i];
#pragma unroll
    for (int k = 0; k < 7; k++) cols64[(uint64_t)k * n_rec + r] = L.v[k * n_lines + i];
    strand[r] = L.strand[i];
    cigar_off[r] = cg_pos[i];
    rec_line[r] = (uint32_t)i;
    uint8_t* dst = names + name_pos[i];
    const uint32_t ql = L.qn_len[i];
    const uint64_t tl = L.name_len[i] - ql;
    for (uint32_t k = 0; k < ql; k++) dst[k] = text[L.qn_off[i] + k];
    for (uint64_t k = 0; k < tl; k++) dst[ql + k] = text[L.tn_off[i] + k];
    rec_name_off[r] = name_pos[i];
    rec_qlen[r] = ql;
}

// destination bytes [16 t, 16 t + 16) of the packed CIGAR text (also the packed BED ids: rec_line nullptr, cg_off per row)
__global__ void __launch_bounds__(PP_THREADS) k_paf_copy_cg(const uint8_t* text, uint32_t n_rec, const uint64_t* cigar_off,
                                                             const uint32_t* rec_line, const uint64_t* cg_off, uint8_t* dst) {
    const uint64_t total = cigar_off[n_rec];
    const uint64_t pos0 = ((uint64_t)blockIdx.x * PP_THREADS + threadIdx.x) * 16;
    if (pos0 >= total) return;
    uint32_t lo = 0, hi = n_rec;  // last record whose payload starts at or before pos0
    while (hi - lo > 1) {
        const uint32_t mid = lo + (hi - lo) / 2;
        if (cigar_off[mid] <= pos0) lo = mid; else hi = mid;
    }
    uint32_t r = lo;
    uint8_t b[16];
#pragma unroll
    for (int j = 0; j < 16; j++) {
        const uint64_t pos = pos0 + j;
        if (pos >= total) { b[j] = '0'; continue; }  // (the tail padding of the text is '0' bytes)
        while (pos >= cigar_off[r + 1]) r++;
        b[j] = text[cg_off[rec_line ? rec_line[r] : r] + (pos - cigar_off[r])];
    }
    uint4 w;
    w.x = b[0] | (b[1] << 8) | (b[2] << 16) | ((uint32_t)b[3] << 24);
    w.y = b[4] | (b[5] << 8) | (b[6] << 16) | ((uint32_t)b[7] << 24);
    w.z = b[8] | (b[9] << 8) | (b[10] << 16) | ((uint32_t)b[11] << 24);
    w.w = b[12] | (b[13] << 8) | (b[14] << 16) | ((uint32_t)b[15] << 24);
    *reinterpret_cast<uint4*>(dst + pos0) = w;
}

uint64_t paf_chunks(uint64_t n) { return (n + PP_CHUNK - 1) / PP_CHUNK; }
uint64_t paf_tiles(uint64_t n) { return (n >> PP_TILE_SHIFT) + 1; }
uint64_t paf_scan_parts(uint64_t n) { return (n + SCAN_CH - 1) / SCAN_CH + 1; }

void launch_paf_lines_count(const uint8_t* text, uint64_t n, uint64_t* chunk_cnt, uint8_t* tile_ws, uint32_t* last_byte, cudaStream_t s) {
    if (n) k_paf_lines_count<LINES_PAF><<<(unsigned)paf_chunks(n), PP_THREADS, 0, s>>>(text, n, chunk_cnt, tile_ws, last_byte);
}
void launch_paf_lines_fill(const uint8_t* text, uint64_t n, const uint64_t* chunk_off, uint64_t* line_start, cudaStream_t s) {
    if (n) k_paf_lines_fill<LINES_PAF><<<(unsigned)paf_chunks(n), PP_THREADS, 0, s>>>(text, n, chunk_off, line_start);
}
void launch_bed_lines_count(const uint8_t* text, uint64_t n, uint64_t* chunk_cnt, cudaStream_t s) {
    if (n) k_paf_lines_count<LINES_BED><<<(unsigned)paf_chunks(n), PP_THREADS, 0, s>>>(text, n, chunk_cnt, nullptr, nullptr);
}
void launch_bed_lines_fill(const uint8_t* text, uint64_t n, const uint64_t* chunk_off, uint64_t* line_start, cudaStream_t s) {
    if (n) k_paf_lines_fill<LINES_BED><<<(unsigned)paf_chunks(n), PP_THREADS, 0, s>>>(text, n, chunk_off, line_start);
}
void launch_paf_scan(int nv, const uint64_t* const* in, uint64_t* const* out, uint64_t n, uint64_t* part, cudaStream_t s) {
    ScanCols c{};
    c.nv = nv;
    for (int v = 0; v < nv; v++) { c.in[v] = in[v]; c.out[v] = out[v]; }
    const uint64_t nb = (n + SCAN_CH - 1) / SCAN_CH;
    if (nb) k_paf_scan_reduce<<<(unsigned)nb, PP_THREADS, 0, s>>>(c, n, part, nb);
    k_paf_scan_parts<<<1, PP_THREADS, 0, s>>>(c, n, part, nb);
    if (nb) k_paf_scan_down<<<(unsigned)nb, PP_THREADS, 0, s>>>(c, n, part, nb);
}
void launch_paf_fields(const uint8_t* text, const uint64_t* line_start, uint64_t n_lines, const uint8_t* tile_ws, PafLineCols L,
                       unsigned long long* first_panic, cudaStream_t s) {
    if (!n_lines) return;
    const uint64_t blocks = std::min<uint64_t>((n_lines + PP_THREADS / 32 - 1) / (PP_THREADS / 32), 148ull * 64);
    k_paf_fields<<<(unsigned)blocks, PP_THREADS, 0, s>>>(text, line_start, n_lines, tile_ws, L, first_panic);
}
void launch_paf_pack(const uint8_t* text, uint64_t n_lines, PafLineCols L, const uint64_t* rec_idx, const uint64_t* cg_pos,
                     const uint64_t* name_pos, uint32_t n_rec, uint64_t* cols64, uint8_t* strand, uint64_t* cigar_off, uint32_t* rec_line,
                     uint8_t* names, uint64_t* rec_name_off, uint32_t* rec_qlen, cudaStream_t s) {
    const uint64_t blocks = (n_lines + PP_THREADS - 1) / PP_THREADS;
    k_paf_pack<<<(unsigned)(blocks ? blocks : 1), PP_THREADS, 0, s>>>(text, n_lines, L, rec_idx, cg_pos, name_pos, n_rec, cols64, strand,
                                                                      cigar_off, rec_line, names, rec_name_off, rec_qlen);
}
void launch_paf_copy_cg(const uint8_t* text, uint32_t n_rec, const uint64_t* cigar_off, const uint32_t* rec_line, const uint64_t* cg_off,
                        uint64_t cg_bytes, uint8_t* dst, cudaStream_t s) {
    const uint64_t threads = (cg_bytes + 15) / 16;
    if (threads) k_paf_copy_cg<<<(unsigned)((threads + PP_THREADS - 1) / PP_THREADS), PP_THREADS, 0, s>>>(text, n_rec, cigar_off, rec_line, cg_off, dst);
}

}  // namespace rb
