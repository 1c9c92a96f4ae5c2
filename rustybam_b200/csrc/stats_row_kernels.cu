// stats_row_kernels.cu — the rows `rb stats --paf` prints for whole records (rb_stats_text), formatted on the device from a batch's
// resident columns, names and the Stats k_rec_prep left (mode 0).  Two passes: k_stats_row_len (one thread per record) and a CUB scan
// give every row its place; k_stats_rows composes a block's rows in shared memory — in the 16-byte phase of their place in the
// output, which is known before they are composed — and stores them with aligned 16-byte stores.  A row longer than the staging
// area (only names of kilobytes make one) is written straight to global memory by its thread: there is no row-length limit.
#include <cub/device/device_scan.cuh>

#include "rb_kernels.cuh"
#include "stats_row.cuh"

namespace rb {

namespace {
constexpr int SR_THREADS = 128;
constexpr uint32_t SR_STAGE = 20 * 1024;  // staging bytes of a block (~150 rows of ~130 bytes: one round at typical name lengths)

__device__ __forceinline__ StatsRow stats_row_of(const RecInput& in, const StatsDev& st, uint32_t i) {
    StatsRow r;
    r.id_bits[0] = __float_as_uint(st.id_m[i]); r.id_bits[1] = __float_as_uint(st.id_e[i]); r.id_bits[2] = __float_as_uint(st.id_a[i]);
    stats_row_digits(r);
    const uint32_t q = in.q_id[i], t = in.t_id[i];
    r.q_name = in.names + in.names_off[q]; r.q_name_len = (uint32_t)(in.names_off[q + 1] - in.names_off[q]);
    r.t_name = in.names + in.names_off[t]; r.t_name_len = (uint32_t)(in.names_off[t + 1] - in.names_off[t]);
    r.q_st = in.q_st[i]; r.q_en = in.q_en[i]; r.q_len = in.q_len[i];
    r.t_st = in.t_st[i]; r.t_en = in.t_en[i]; r.t_len = in.t_len[i];
    r.strand = in.strand[i];
    r.equal = st.equal[i]; r.diff = st.diff[i]; r.ins = st.ins[i]; r.del = st.del[i];
    r.ins_events = st.ins_ev[i]; r.del_events = st.del_ev[i]; r.matches = st.matches[i];
    return r;
}

// line_len[i] = bytes of row i; line_len[n] = 0 (the scan leaves the total there)
__global__ void __launch_bounds__(SR_THREADS, 4) k_stats_row_len(RecInput in, StatsDev st, unsigned long long* __restrict__ line_len) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < in.n_rec) line_len[i] = stats_row_len(stats_row_of(in, st, (uint32_t)i));
    else if (i == in.n_rec) line_len[i] = 0;
}

// Rounds over the block's rows: a round starts at the first row not written yet and composes every row that ends within SR_STAGE
// bytes of it (a run of consecutive rows), then the whole block stores the run.
__global__ void __launch_bounds__(SR_THREADS) k_stats_rows(RecInput in, StatsDev st, const uint64_t* __restrict__ line_off,
                                                           uint8_t* __restrict__ out, uint32_t qbed) {
    __shared__ __align__(16) uint8_t s_buf[SR_STAGE + 32];
    __shared__ unsigned long long s_next, s_end;
    const int tid = threadIdx.x;
    const uint64_t first = (uint64_t)blockIdx.x * SR_THREADS, i = first + (uint64_t)tid;
    const uint64_t blk_lo = line_off[first];
    const bool live = i < in.n_rec;
    const uint64_t my_lo = live ? line_off[i] - blk_lo : 0, my_len = live ? line_off[i + 1] - line_off[i] : 0;
    const bool is_long = live && my_len > SR_STAGE;
    bool done = !live || is_long, put_long = is_long;  // (a long row takes no part in the rounds: it goes out in the first one)
    for (;;) {
        if (tid == 0) { s_next = ~0ull; s_end = 0; }
        __syncthreads();
        if (!done) atomicMin(&s_next, (unsigned long long)my_lo);
        __syncthreads();
        const uint64_t base = s_next;
        const bool last = base == ~0ull;  // (block-uniform)
        const uint32_t ph = (uint32_t)((blk_lo + base) & 15u);  // s_buf[ph + k] holds out[blk_lo + base + k]
        const bool fits = !done && !last && my_lo + my_len <= base + SR_STAGE;
        if (fits || put_long) {  // (one call site: the composer is inlined once)
            stats_row_put(fits ? s_buf + ph + (my_lo - base) : out + blk_lo + my_lo, stats_row_of(in, st, (uint32_t)i), qbed != 0);
            if (fits) atomicMax(&s_end, (unsigned long long)(my_lo + my_len));
            done = true; put_long = false;
        }
        if (last) break;
        __syncthreads();
        const uint64_t g0 = blk_lo + base, g1 = blk_lo + s_end;
        const uint64_t a0 = (g0 + 15u) & ~15ull, a1 = g1 & ~15ull;
        const uint8_t* sb = s_buf + ph;
        if (a0 >= a1) {
            for (uint64_t g = g0 + tid; g < g1; g += SR_THREADS) out[g] = sb[g - g0];
        } else {
            for (uint64_t g = g0 + tid; g < a0; g += SR_THREADS) out[g] = sb[g - g0];
            for (uint64_t v = a0 + 16u * (uint64_t)tid; v < a1; v += 16u * SR_THREADS)
                *reinterpret_cast<uint4*>(out + v) = *reinterpret_cast<const uint4*>(sb + (v - g0));
            for (uint64_t g = a1 + tid; g < g1; g += SR_THREADS) out[g] = sb[g - g0];
        }
        __syncthreads();
    }
}
}  // namespace

void launch_stats_row_len(const RecInput& in, const StatsDev& st, uint64_t* line_off, cudaStream_t s) {
    const uint64_t n = (uint64_t)in.n_rec + 1;
    k_stats_row_len<<<(unsigned)((n + SR_THREADS - 1) / SR_THREADS), SR_THREADS, 0, s>>>(in, st, reinterpret_cast<unsigned long long*>(line_off));
}
cudaError_t launch_stats_row_scan(uint64_t* line_off, uint32_t n_rec, void* tmp, size_t& tmp_bytes, cudaStream_t s) {
    return cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, line_off, (uint64_t)n_rec + 1, s);
}
void launch_stats_rows(const RecInput& in, const StatsDev& st, const uint64_t* line_off, uint8_t* out, bool qbed, cudaStream_t s) {
    if (in.n_rec)
        k_stats_rows<<<(unsigned)((in.n_rec + SR_THREADS - 1) / SR_THREADS), SR_THREADS, 0, s>>>(in, st, line_off, out, qbed ? 1u : 0u);
}

}  // namespace rb
