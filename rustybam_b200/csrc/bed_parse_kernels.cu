// bed_parse_kernels.cu — BED text -> the window tables of a resident batch (rb_batch_set_windows_bed), the rules of
// bed_parse_core.cuh applied on the GPU.  Line starts come from k_paf_lines_count / k_paf_lines_fill (LINES_BED) and every
// exclusive scan from launch_paf_scan (paf_parse_kernels.cu); then:
//
//   k_bed_names    the batch's name table -> an open-addressing hash table (u32 slots: name id + 1, linear probing)
//   k_bed_fields   one thread per line: comment, field count, st / en, field 1 and field 4 spans (bed_parse_core.cuh: bed_line);
//                  the first non-comment line by atomicMin on its index
//   k_bed_judge    one thread per line: parses against that line's field count, contig lookup (byte compares) -> kept
//   k_bed_compact  kept lines -> rows in file order (t_id, st, en, bed_row, line); max st for the sort key; (t_id, st) order check
//   CUB radix sort stable sort by (t_id, st) (one packed 64-bit key when t_id and st fit in it, else st then t_id), only when the
//                  rows are not in that order already; by t_id alone for the general layout
//   k_bed_gather   rows in sorted order -> the batch's w_* tables, and the id spans in that order
//   k_bed_cont     per contig, the range of its rows (cont_lo / cont_hi)
// The id bytes are copied by k_paf_copy_cg (16 destination bytes per thread) after a scan of their lengths.
// BED lines are short: one thread per line.  A megabyte-long column is correct, not fast.
#include <algorithm>
#include <cstdint>

#include <cub/device/device_radix_sort.cuh>

#include "bed_parse_core.cuh"
#include "rb_kernels.cuh"

namespace rb {

namespace {

constexpr int BP_THREADS = 256;

__device__ __forceinline__ uint64_t line_end(const uint8_t* text, uint64_t n, uint64_t a) {
    uint64_t b = a;
    while (b < n && !rbbp::is_eol(text[b])) b++;
    return b;
}

__device__ __forceinline__ bool bytes_eq(const uint8_t* x, const uint8_t* y, uint64_t n) {
    for (uint64_t k = 0; k < n; k++)
        if (x[k] != y[k]) return false;
    return true;
}

unsigned grid_for(uint64_t n) { return (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((n + BP_THREADS - 1) / BP_THREADS, 148ull * 64)); }

}  // namespace

// equal names keep the smallest id (what a host index built in id order finds)
__global__ void __launch_bounds__(BP_THREADS) k_bed_names(const uint8_t* names, const uint64_t* names_off, uint32_t n_names, uint32_t* table,
                                                          uint64_t mask) {
    for (uint64_t i = (uint64_t)blockIdx.x * BP_THREADS + threadIdx.x; i < n_names; i += (uint64_t)gridDim.x * BP_THREADS) {
        const uint64_t a = names_off[i], len = names_off[i + 1] - a;
        uint64_t h = rbbp::name_hash(names + a, len) & mask;
        for (;;) {
            const uint32_t cur = atomicCAS(&table[h], 0u, (uint32_t)i + 1);
            if (cur == 0) break;
            const uint64_t ja = names_off[cur - 1], jl = names_off[cur] - ja;
            if (jl == len && bytes_eq(names + ja, names + a, len)) { atomicMin(&table[h], (uint32_t)i + 1); break; }
            h = (h + 1) & mask;
        }
    }
}

__global__ void __launch_bounds__(BP_THREADS) k_bed_fields(const uint8_t* text, uint64_t n, uint64_t n_lines, BedLineCols L,
                                                           unsigned long long* first_row) {
    for (uint64_t i = (uint64_t)blockIdx.x * BP_THREADS + threadIdx.x; i < n_lines; i += (uint64_t)gridDim.x * BP_THREADS) {
        const uint64_t a = L.line_start[i];
        rbbp::BedLine o;
        rbbp::bed_line(text, a, line_end(text, n, a), o);
        L.n_fields[i] = o.n_fields;
        L.st[i] = o.st; L.en[i] = o.en;
        L.name_len[i] = o.name_len;
        L.id_off[i] = o.id_off; L.id_len[i] = o.id_len;
        L.nums_ok[i] = o.nums_ok ? 1 : 0;
        L.comment[i] = o.comment ? 1 : 0;
        if (!o.comment) atomicMin(first_row, (unsigned long long)i);
    }
}

__global__ void __launch_bounds__(BP_THREADS) k_bed_judge(const uint8_t* text, uint64_t n_lines, BedLineCols L, const unsigned long long* first_row,
                                                          const uint8_t* names, const uint64_t* names_off, const uint32_t* table, uint64_t mask,
                                                          unsigned long long* nf0_out) {
    const uint64_t f = *first_row;
    const uint64_t nf0 = f < n_lines ? L.n_fields[f] : 0;
    for (uint64_t i = (uint64_t)blockIdx.x * BP_THREADS + threadIdx.x; i < n_lines; i += (uint64_t)gridDim.x * BP_THREADS) {
        if (i == f) *nf0_out = nf0;
        rbbp::BedLine o;
        o.comment = L.comment[i] != 0; o.n_fields = L.n_fields[i]; o.nums_ok = L.nums_ok[i] != 0;
        const bool parses = rbbp::row_parses(o, nf0);
        uint32_t tid = ~0u;
        if (parses) {
            const uint8_t* name = text + L.line_start[i];
            const uint64_t len = L.name_len[i];
            uint64_t h = rbbp::name_hash(name, len) & mask;
            for (;;) {
                const uint32_t v = table[h];
                if (v == 0) break;
                const uint64_t ja = names_off[v - 1], jl = names_off[v] - ja;
                if (jl == len && bytes_eq(names + ja, name, len)) { tid = v - 1; break; }
                h = (h + 1) & mask;
            }
        }
        L.parses[i] = parses ? 1 : 0;
        L.kept[i] = tid != ~0u ? 1 : 0;
        L.tid[i] = tid;
    }
}

// row_idx / win_idx = exclusive scans of parses / kept
__global__ void __launch_bounds__(BP_THREADS) k_bed_compact(uint64_t n_lines, BedLineCols L, const uint64_t* row_idx, const uint64_t* win_idx,
                                                            BedRows R, unsigned long long* max_st) {
    unsigned long long m = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * BP_THREADS + threadIdx.x; i < n_lines; i += (uint64_t)gridDim.x * BP_THREADS) {
        if (!L.kept[i]) continue;
        const uint64_t k = win_idx[i];
        R.tid[k] = L.tid[i]; R.st[k] = L.st[i]; R.en[k] = L.en[i]; R.row[k] = (uint32_t)row_idx[i]; R.line[k] = i;
        m = L.st[i] > m ? L.st[i] : m;
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        const unsigned long long w = __shfl_xor_sync(0xFFFFFFFFu, m, o);
        m = w > m ? w : m;
    }
    if ((threadIdx.x & 31) == 0 && m) atomicMax(max_st, m);
}

__global__ void __launch_bounds__(BP_THREADS) k_bed_order(BedRows R, uint32_t n, uint32_t* unsorted) {
    uint32_t f = 0;
    for (uint64_t k = (uint64_t)blockIdx.x * BP_THREADS + threadIdx.x + 1; k < n; k += (uint64_t)gridDim.x * BP_THREADS)
        if (R.tid[k] < R.tid[k - 1] || (R.tid[k] == R.tid[k - 1] && R.st[k] < R.st[k - 1])) f = 1;
    if (__any_sync(0xFFFFFFFFu, f) && (threadIdx.x & 31) == 0) atomicOr(unsorted, 1u);
}

// sort keys: mode 0 = (t_id << sb) | st, mode 1 = st, mode 2 = t_id[perm[k]] (the second pass), mode 3 = t_id; vals = the identity
// (modes 0, 1, 3) or perm (mode 2)
__global__ void __launch_bounds__(BP_THREADS) k_bed_keys(int mode, BedRows R, uint32_t n, int sb, const uint32_t* perm, uint64_t* keys,
                                                         uint32_t* vals) {
    for (uint64_t k = (uint64_t)blockIdx.x * BP_THREADS + threadIdx.x; k < n; k += (uint64_t)gridDim.x * BP_THREADS) {
        const uint32_t j = mode == 2 ? perm[k] : (uint32_t)k;
        keys[k] = mode == 0 ? ((uint64_t)R.tid[k] << sb) | R.st[k] : mode == 1 ? R.st[k] : (uint64_t)R.tid[j];
        vals[k] = j;
    }
}

__global__ void __launch_bounds__(BP_THREADS) k_bed_gather(BedRows R, uint32_t n, const uint32_t* perm, const uint64_t* line_id_off,
                                                           const uint64_t* line_id_len, uint32_t* w_tid, uint64_t* w_st, uint64_t* w_en,
                                                           uint32_t* w_row, uint64_t* id_off, uint64_t* id_len) {
    for (uint64_t k = (uint64_t)blockIdx.x * BP_THREADS + threadIdx.x; k < n; k += (uint64_t)gridDim.x * BP_THREADS) {
        const uint32_t j = perm ? perm[k] : (uint32_t)k;
        w_tid[k] = R.tid[j]; w_st[k] = R.st[j]; w_en[k] = R.en[j]; w_row[k] = R.row[j];
        if (id_off) { id_off[k] = line_id_off[R.line[j]]; id_len[k] = line_id_len[R.line[j]]; }
    }
}

__global__ void __launch_bounds__(BP_THREADS) k_bed_cont(const uint32_t* w_tid, uint32_t n, uint32_t* cont_lo, uint32_t* cont_hi) {
    for (uint64_t k = (uint64_t)blockIdx.x * BP_THREADS + threadIdx.x; k < n; k += (uint64_t)gridDim.x * BP_THREADS) {
        const uint32_t t = w_tid[k];
        if (k == 0 || w_tid[k - 1] != t) cont_lo[t] = (uint32_t)k;
        if (k + 1 == n || w_tid[k + 1] != t) cont_hi[t] = (uint32_t)k + 1;
    }
}

uint64_t bed_name_slots(uint32_t n_names) {
    uint64_t s = 64;
    while (s < 2ull * n_names) s <<= 1;
    return s;
}

void launch_bed_names(const uint8_t* names, const uint64_t* names_off, uint32_t n_names, uint32_t* table, uint64_t slots, cudaStream_t s) {
    if (n_names) k_bed_names<<<grid_for(n_names), BP_THREADS, 0, s>>>(names, names_off, n_names, table, slots - 1);
}
void launch_bed_fields(const uint8_t* text, uint64_t n, uint64_t n_lines, BedLineCols L, unsigned long long* first_row, cudaStream_t s) {
    if (n_lines) k_bed_fields<<<grid_for(n_lines), BP_THREADS, 0, s>>>(text, n, n_lines, L, first_row);
}
void launch_bed_judge(const uint8_t* text, uint64_t n_lines, BedLineCols L, const unsigned long long* first_row, const uint8_t* names,
                      const uint64_t* names_off, const uint32_t* table, uint64_t slots, unsigned long long* nf0_out, cudaStream_t s) {
    if (n_lines) k_bed_judge<<<grid_for(n_lines), BP_THREADS, 0, s>>>(text, n_lines, L, first_row, names, names_off, table, slots - 1, nf0_out);
}
void launch_bed_compact(uint64_t n_lines, BedLineCols L, const uint64_t* row_idx, const uint64_t* win_idx, BedRows R, unsigned long long* max_st,
                        cudaStream_t s) {
    if (n_lines) k_bed_compact<<<grid_for(n_lines), BP_THREADS, 0, s>>>(n_lines, L, row_idx, win_idx, R, max_st);
}
void launch_bed_order(BedRows R, uint32_t n, uint32_t* unsorted, cudaStream_t s) {
    if (n > 1) k_bed_order<<<grid_for(n), BP_THREADS, 0, s>>>(R, n, unsorted);
}

// bytes of sort scratch for n rows: two key arrays, two value arrays, CUB's temporary storage
size_t bed_sort_scratch(uint32_t n) {
    size_t tmp = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tmp, (const uint64_t*)nullptr, (uint64_t*)nullptr, (const uint32_t*)nullptr, (uint32_t*)nullptr,
                                    n, 0, 64, (cudaStream_t)0);
    return 2 * ((size_t)n * 8 + 256) + 2 * ((size_t)n * 4 + 256) + tmp + 256;
}

// perm = the stable order of R's rows by (t_id, st) (by_tid_only: by t_id); tb / sb = bits of the largest t_id / st
cudaError_t launch_bed_sort(BedRows R, uint32_t n, int tb, int sb, bool by_tid_only, void* scratch, size_t scratch_bytes, uint32_t* perm,
                            cudaStream_t s) {
    auto up = [](size_t x) { return (x + 255) / 256 * 256; };
    uint8_t* p = static_cast<uint8_t*>(scratch);
    uint64_t* k0 = reinterpret_cast<uint64_t*>(p); p += up((size_t)n * 8);
    uint64_t* k1 = reinterpret_cast<uint64_t*>(p); p += up((size_t)n * 8);
    uint32_t* v0 = reinterpret_cast<uint32_t*>(p); p += up((size_t)n * 4);
    uint32_t* v1 = reinterpret_cast<uint32_t*>(p); p += up((size_t)n * 4);
    void* tmp = p;
    size_t tmp_bytes = scratch_bytes - (size_t)(p - static_cast<uint8_t*>(scratch));
    auto sort = [&](const uint64_t* kin, const uint32_t* vin, uint32_t* vout, int bits) {
        return cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, kin, k1, vin, vout, n, 0, std::max(bits, 1), s);
    };
    const unsigned g = grid_for(n);
    if (by_tid_only) {
        k_bed_keys<<<g, BP_THREADS, 0, s>>>(3, R, n, 0, nullptr, k0, v0);
        return sort(k0, v0, perm, tb);
    }
    if (tb + sb <= 64) {
        k_bed_keys<<<g, BP_THREADS, 0, s>>>(0, R, n, sb, nullptr, k0, v0);
        return sort(k0, v0, perm, tb + sb);
    }
    k_bed_keys<<<g, BP_THREADS, 0, s>>>(1, R, n, 0, nullptr, k0, v0);
    cudaError_t e = sort(k0, v0, v1, sb);
    if (e != cudaSuccess) return e;
    k_bed_keys<<<g, BP_THREADS, 0, s>>>(2, R, n, 0, v1, k0, v0);
    return sort(k0, v0, perm, tb);
}

void launch_bed_gather(BedRows R, uint32_t n, const uint32_t* perm, const uint64_t* line_id_off, const uint64_t* line_id_len, uint32_t* w_tid,
                       uint64_t* w_st, uint64_t* w_en, uint32_t* w_row, uint64_t* id_off, uint64_t* id_len, cudaStream_t s) {
    if (n) k_bed_gather<<<grid_for(n), BP_THREADS, 0, s>>>(R, n, perm, line_id_off, line_id_len, w_tid, w_st, w_en, w_row, id_off, id_len);
}
void launch_bed_cont(const uint32_t* w_tid, uint32_t n, uint32_t* cont_lo, uint32_t* cont_hi, cudaStream_t s) {
    if (n) k_bed_cont<<<grid_for(n), BP_THREADS, 0, s>>>(w_tid, n, cont_lo, cont_hi);
}

}  // namespace rb
