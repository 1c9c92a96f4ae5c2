// text_multi_kernels.cu — the device steps of rb_liftover_text on a multi-device context that are not parsing or lifting: the first
// '\n' of a device's byte range (the line fix-up, text_split.hpp), and the contig runs of a device's rows with their line offsets
// rebased into the merged output.
#include "rb_kernels.cuh"

namespace rb {

namespace {
constexpr int NL_THREADS = 256;
constexpr uint64_t NL_BLOCK_BYTES = (uint64_t)NL_THREADS * 16;

// 16 bytes per thread; a block whose bytes all lie behind a newline found already leaves at once, so a range whose first line is
// short costs a few blocks, not a pass over the range
__global__ void k_first_newline(const uint8_t* __restrict__ text, uint64_t n, unsigned long long* first) {
    const uint64_t b0 = (uint64_t)blockIdx.x * NL_BLOCK_BYTES;
    if (*reinterpret_cast<volatile unsigned long long*>(first) < b0) return;
    const uint64_t at = b0 + (uint64_t)threadIdx.x * 16;
    if (at >= n) return;
    const uint4 w = *reinterpret_cast<const uint4*>(text + at);  // (the buffer is 16-byte aligned and padded)
    const uint32_t v[4] = {w.x, w.y, w.z, w.w};
    for (int k = 0; k < 16; k++) {
        if (at + k >= n) return;
        if (((v[k >> 2] >> (8 * (k & 3))) & 0xFF) == '\n') { atomicMin(first, (unsigned long long)(at + k)); return; }
    }
}

__device__ __forceinline__ uint32_t row_rank(const uint32_t* rec_idx, uint32_t rec_base, const uint32_t* t_id, const uint32_t* rank_of,
                                             uint64_t i) {
    return rank_of[t_id[rec_idx[i] - rec_base]];
}

// rows are grouped by contig (emission order): the first row of a run stores its start, the last its end
__global__ void k_contig_runs(uint64_t n, const uint32_t* __restrict__ rec_idx, uint32_t rec_base, const uint32_t* __restrict__ t_id,
                              const uint32_t* __restrict__ rank_of, const uint64_t* __restrict__ line_off, uint64_t out_bytes,
                              uint64_t* __restrict__ runs, uint32_t n_ranks) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t r = row_rank(rec_idx, rec_base, t_id, rank_of, i);
    uint64_t* row_lo = runs; uint64_t* row_hi = runs + n_ranks; uint64_t* byte_lo = runs + 2 * (uint64_t)n_ranks;
    uint64_t* byte_hi = runs + 3 * (uint64_t)n_ranks;
    if (i == 0 || row_rank(rec_idx, rec_base, t_id, rank_of, i - 1) != r) {
        row_lo[r] = i;
        byte_lo[r] = line_off ? line_off[i] : 0;
    }
    if (i + 1 == n || row_rank(rec_idx, rec_base, t_id, rank_of, i + 1) != r) {
        row_hi[r] = i + 1;
        byte_hi[r] = line_off ? (i + 1 == n ? out_bytes : line_off[i + 1]) : 0;
    }
}

__global__ void k_rebase_runs(uint64_t n, const uint32_t* __restrict__ rec_idx, uint32_t rec_base, const uint32_t* __restrict__ t_id,
                              const uint32_t* __restrict__ rank_of, const unsigned long long* __restrict__ delta,
                              unsigned long long* __restrict__ line_off) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) line_off[i] += delta[row_rank(rec_idx, rec_base, t_id, rank_of, i)];
}
}  // namespace

void launch_first_newline(const uint8_t* text, uint64_t n, unsigned long long* first, cudaStream_t s) {
    if (n) k_first_newline<<<(unsigned)((n + NL_BLOCK_BYTES - 1) / NL_BLOCK_BYTES), NL_THREADS, 0, s>>>(text, n, first);
}
void launch_contig_runs(uint64_t n, const uint32_t* rec_idx, uint32_t rec_base, const uint32_t* t_id, const uint32_t* rank_of,
                        const uint64_t* line_off, uint64_t out_bytes, uint64_t* runs, uint32_t n_ranks, cudaStream_t s) {
    if (n) k_contig_runs<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(n, rec_idx, rec_base, t_id, rank_of, line_off, out_bytes, runs, n_ranks);
}
void launch_rebase_runs(uint64_t n, const uint32_t* rec_idx, uint32_t rec_base, const uint32_t* t_id, const uint32_t* rank_of,
                        const uint64_t* delta, uint64_t* line_off, cudaStream_t s) {
    if (n)
        k_rebase_runs<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(n, rec_idx, rec_base, t_id, rank_of,
                                                                  reinterpret_cast<const unsigned long long*>(delta),
                                                                  reinterpret_cast<unsigned long long*>(line_off));
}

}  // namespace rb
