// rbcuda.cu — C ABI (include/rbcuda.h) over the sm_100a kernels: context, HBM / pinned buffer
// pools, and the upload -> tokenise -> scan -> join -> lift -> serialise -> download pipeline.
// There is NO CPU implementation behind these entry points: without a compute-capability-10
// device they fail with RB_ERR_NO_DEVICE.
#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include <sys/mman.h>

#include "../../include/rbcuda.h"
#include "name_intern.hpp"
#include "paf_parse_core.cuh"
#include "rb_kernels.cuh"
#include "rec_core.cuh"
#include "text_split.hpp"
#include "trim_rounds.hpp"

using namespace rb;

namespace {

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = n + n / 8 + 256;  // head-room so that steady-state calls never reallocate
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) { (void)cudaGetLastError(); want = n; e = cudaMalloc(&p, want); }
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

void* big_pinned_alloc(size_t n);
void big_pinned_free(void* q, size_t n);
constexpr size_t BIG_PIN_MIN = 64ull << 20;

// pinned staging area owned by a batch: the record columns are gathered here on the host and leave by
// asynchronous DMA (the caller's column arrays may share pages with a buffer it page-locked, which the driver rejects).
// Small for whole-genome records; millions of short records (rb stats --paf behind rb liftover: 81 B per record) make it
// hundreds of MB, which cudaHostAlloc page-locks at ~2.3 GB/s — those sizes take the mapped + registered route (big_pinned_alloc)
struct PinBuf {
    uint8_t* p = nullptr;
    size_t cap = 0;
    bool mapped = false;
    cudaError_t ensure(size_t n) {
        if (n <= cap) return cudaSuccess;
        release();
        size_t want = n + n / 4 + 4096;
        if (want >= BIG_PIN_MIN && !getenv("RB_PIN_HOSTALLOC")) {
            want = (want + 4095) / 4096 * 4096;
            p = static_cast<uint8_t*>(big_pinned_alloc(want));
            mapped = p != nullptr;
        }
        if (!p) {
            const cudaError_t e = cudaHostAlloc(reinterpret_cast<void**>(&p), want, cudaHostAllocDefault);
            if (e != cudaSuccess) { p = nullptr; return e; }
        }
        cap = want;
        return cudaSuccess;
    }
    void release() {
        if (p) { if (mapped) big_pinned_free(p, cap); else cudaFreeHost(p); }
        p = nullptr; cap = 0; mapped = false;
    }
};

struct PinnedBlock {
    void* p = nullptr;
    size_t cap = 0;
    bool in_use = false;
    bool mapped = false;  // big_pinned_alloc (mmap + cudaHostRegister) instead of cudaHostAlloc
};

// Page-locked host memory for the large output blocks.  cudaHostAlloc locks pages at ~2.3 GB/s (16 GiB: 7.1 s — the driver
// faults them in one by one), which made the first rb_liftover of a process that returns C5's 17.6 GB take 12 s.  An anonymous
// mapping first-touched by a few host threads and then registered takes 0.6 s for 16 GiB and copies at the same
// 55 GB/s (tools/pin_bench.cu, profiles/r02_pin_bench.json).  Portable: every device of a multi-device context copies into it.
void* big_pinned_alloc(size_t n) {
    void* q = mmap(nullptr, n, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
    if (q == MAP_FAILED) return nullptr;
    madvise(q, n, MADV_HUGEPAGE);
    unsigned nthr = std::thread::hardware_concurrency();
    nthr = nthr < 1 ? 1 : (nthr > 16 ? 16 : nthr);
    {
        std::vector<std::thread> th;
        uint8_t* b = static_cast<uint8_t*>(q);
        for (unsigned t = 0; t < nthr; t++)
            th.emplace_back([=] {
                const size_t lo = n / nthr * t, hi = (t + 1 == nthr) ? n : n / nthr * (t + 1);
                for (size_t i = lo; i < hi; i += 4096) b[i] = 0;
            });
        for (auto& x : th) x.join();
    }
    // ONE registration for the whole block: the library's copies into it (2-D ones among them) may start and end anywhere, and a
    // copy must not span two registrations.  If the driver refuses a range this large the caller falls back to cudaHostAlloc.
    if (cudaHostRegister(q, n, cudaHostRegisterPortable) != cudaSuccess) {
        (void)cudaGetLastError();
        munmap(q, n);
        return nullptr;
    }
    return q;
}
void big_pinned_free(void* q, size_t n) {
    cudaHostUnregister(q);
    munmap(q, n);
}
void pinned_block_free(PinnedBlock* b) {
    if (!b->p) return;
    if (b->mapped) big_pinned_free(b->p, b->cap);
    else cudaFreeHost(b->p);
    b->p = nullptr;
}

struct KEvent {
    const char* name;
    cudaEvent_t a, b;
};

}  // namespace

struct rb_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = true;
    std::string err;
    bool profiling = false;
    int lift_mode = RB_LIFT_SEARCH;
    bool fused_emit = true;       // line scan + serialiser in one kernel (k_emit) where the rows are short; RB_NO_FUSED_EMIT=1 disables
    bool invert = false;          // the call in progress is a --qbed liftover
    bool stats_text = false;      // the call in progress wants RB_WANT_STATS_TEXT rows
    std::vector<KEvent> pending;
    std::vector<cudaEvent_t> ev_pool;
    std::vector<rb_kernel_time> times;
    std::vector<PinnedBlock*> pinned;
    rb_batch* scratch = nullptr;  // reused by rb_liftover / rb_stats
    rb_batch* slice[2] = {nullptr, nullptr};  // ping-pong work areas of the sliced rb_liftover
    cudaStream_t copy_stream = nullptr;        // device -> host copies of finished slices
    cudaStream_t up_stream = nullptr;          // host -> device copies of the next slice
    cudaStream_t upload_on = nullptr;          // stream upload_cigar / upload_columns enqueue on (nullptr: `stream`)
    cudaEvent_t ev_up[2] = {nullptr, nullptr};
    cudaEvent_t ev_done[2] = {nullptr, nullptr}, ev_d2h[2] = {nullptr, nullptr};
    cudaEvent_t ev_win = nullptr, ev_wfirst = nullptr;
    uint64_t slice_min_bytes = 16ull << 20;  // rb_ctx_set_slicing (0 = off)
    DevBuf scalars;               // small device scalars
    void* h_scalars = nullptr;    // pinned, mapped mirror (kernels store into it: k_publish)
    void* h_scalars_dev = nullptr;  // its device-side address
    std::vector<rb_ctx*> peers;     // multi-device context (rb_ctx_create with n_devices > 1): one context per further device
    uint64_t err_rec = UINT64_MAX;  // the caller's record index of the error map_err reported last
    uint64_t multi_min_bytes = 8ull << 20;  // smaller calls stay on the first device (RB_MULTI_MIN_BYTES overrides)
};

struct rb_batch {
    uint32_t n_rec = 0, n_win = 0, n_names = 0;
    uint64_t n_bytes = 0, n_tiles = 0, ops_bound = 0;
    bool general = false;  // BED rows not (sorted, monotone `en`, file order == sorted order): brute-force join
    std::vector<uint64_t> h_cigar_off;
    // host staging of the asynchronous uploads (must stay alive until the stream has consumed it)
    std::vector<uint32_t> h_clo, h_chi, h_orig;
    PinBuf stage;   // pinned copies of the record columns
    PinBuf wstage;  // pinned copies of the contig ranges of the window table
    struct { std::vector<uint64_t> st, en, off; std::vector<uint32_t> row; std::vector<uint8_t> ids; } h_gen;
    bool busy = false;         // uploads of this batch may still be in flight
    bool file_order = false;   // emission order = file order (break-paf) instead of contig by contig
    bool invert = false;       // liftover --qbed: the uploaded columns are swapped, the ops get inverted after tokenising
    bool win_pending = false;  // the window check kernel's verdict has not been read yet
    rb_batch* wsrc = nullptr;  // the batch that holds the window tables (nullptr: this one) — slices share their parent's
    uint32_t rec_base = 0;     // slices: index of this batch's record 0 in the caller's arrays
    uint64_t byte_base = 0;    // slices: output bytes emitted before this batch (added to line_off)
    bool default_ids = false;  // rb_windows.ids_off == NULL: window id = "{t_name}:{st+1}-{en}" (bed.rs:150-153)
    // inputs
    DevBuf text_raw, cigar_off, cols64, strand, ids32, names, names_off, rec_order, rec_rank;
    DevBuf w_st, w_en, w_ids_off, w_ids, w_bed_row, w_tid, cont_lo, cont_hi;
    // intermediates
    DevBuf ops, tile_state, heads, samples, blk_state, blk_agg, blk_pre, op_off, recs, pair_cnt, pair_off;
    DevBuf tile_first, head_pos, seg_state, seg_agg, seg_pre;  // fused tokeniser + sample scan (k_tok_scan): per-tile tables
    bool have_samples = false;  // run_tok already left the samples (run_scan without boundary resolution has nothing to do)
    DevBuf pair_res, line_len, line_off, out_idx, pair_win, ln_state, ln_agg, ln_pre, half_s, half_e, plans, orig_idx;
    DevBuf bp_cnt, bp_off, bp_end, bp_next, rec_bp;  // break-paf: break ops per chunk, their scan, piece boundaries
    DevBuf trim_qp, trim_wp, trim_ap, trim_views, trim_sel, trim_out, trim_drop;  // trim-paf: per-op query / score prefixes, record views, one round's pairs
    bool trim_has_drop = false, trim_ready = false;   // trim_ready: between rb_trim_paf_begin and rb_trim_paf_end
    std::vector<uint32_t> trim_perm;                   // name-sorted position -> the caller's record index
    int trim_scores[3] = {1, 1, 1};
    int trim_policy = 0;
    uint64_t trim_max_score = 1, trim_n_ops = 0;
    uint32_t trim_groups = 0;
    size_t trim_o[4] = {0, 0, 0, 0};                   // offsets of sel / keys / round state / group offsets inside trim_sel
    // outputs (device)
    DevBuf out_text, out_line_off, out_num, out_stats;
    DevBuf blk_flags, emit_totals;  // k_emit: per-block "left to k_serialise" flags, {bytes, rows, overflow, deferred blocks}
    bool stats_text = false;        // the rows in out_text are `rb stats --paf` rows (RB_WANT_STATS_TEXT)
    uint64_t row_stride = 0;        // rows between the columns of out_num / out_stats (n_out, or the pair count when k_emit wrote them)
    rb_summary sum{};
    bool have_lift = false, have_stats = false, with_stats = false;
    uint32_t want = 0;
    uint64_t stats_n = 0;
    // rb_batch_upload_paf: the name table handed out through rb_paf_info; rb_batch_records: its pinned copy of the records
    std::vector<uint8_t> h_names;
    std::vector<uint64_t> h_names_off;
    PinBuf rec_out;
    PinBuf win_out;  // rb_batch_windows: its pinned copy of the window tables
};

namespace {

// device scalar slots
enum { SC_TICKET_TOK = 0, SC_TICKET_SMP = 1, SC_TICKET_LNS = 2, SC_MISC = 3, SC_ERR_TOK = 4 /*u64*/, SC_ERR_REC = 6 /*u64*/, SC_WINFLAGS = 8, SC_WORDS = 12 };

int fail(rb_ctx* c, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (c) c->err = buf;
    return code;
}
#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            (void)cudaGetLastError();                                                              \
            return fail(ctx, e_ == cudaErrorMemoryAllocation ? RB_ERR_OOM : RB_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(e_)); \
        }                                                                                          \
    } while (0)

size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// host -> device copy of a caller buffer, cut at absolute 1 GiB-aligned source addresses (see rb_host_register)
cudaError_t h2d_copy(void* dst, const void* src, size_t n, cudaStream_t s) {
    const uint64_t G = 1ull << 30;
    uint64_t a = reinterpret_cast<uintptr_t>(src);
    uint8_t* d = static_cast<uint8_t*>(dst);
    while (n) {
        const uint64_t e = (a / G + 1) * G;
        const size_t len = (size_t)std::min<uint64_t>(n, e - a);
        const cudaError_t rc = cudaMemcpyAsync(d, reinterpret_cast<const void*>(a), len, cudaMemcpyHostToDevice, s);
        if (rc != cudaSuccess) return rc;
        a += len; d += len; n -= len;
    }
    return cudaSuccess;
}

PinnedBlock* pinned_get(rb_ctx* ctx, size_t n) {
    PinnedBlock* best = nullptr;
    for (PinnedBlock* b : ctx->pinned)
        if (!b->in_use && b->cap >= n && (!best || b->cap < best->cap)) best = b;
    if (!best) {
        // drop the largest idle block that is too small, so the pool does not grow without bound
        for (size_t i = 0; i < ctx->pinned.size(); i++)
            if (!ctx->pinned[i]->in_use) {
                pinned_block_free(ctx->pinned[i]);
                delete ctx->pinned[i];
                ctx->pinned.erase(ctx->pinned.begin() + (long)i);
                break;
            }
        best = new PinnedBlock();
        size_t want = n + n / 8 + 4096;
        if (want >= BIG_PIN_MIN && !getenv("RB_PIN_HOSTALLOC")) {
            want = (want + 4095) / 4096 * 4096;
            best->p = big_pinned_alloc(want);
            best->mapped = best->p != nullptr;
        }
        if (!best->p && cudaHostAlloc(&best->p, want, cudaHostAllocPortable) != cudaSuccess) {  // (portable: every device of a multi-device context copies into it)
            (void)cudaGetLastError();
            delete best;
            return nullptr;
        }
        best->cap = want;
        ctx->pinned.push_back(best);
    }
    best->in_use = true;
    return best;
}

// ---- per-kernel CUDA-event timing ----
struct KScope {
    rb_ctx* ctx;
    KEvent ev{};
    bool on;
    KScope(rb_ctx* c, const char* name) : ctx(c), on(c->profiling) {
        if (!on) return;
        auto get = [&]() {
            cudaEvent_t e;
            if (!ctx->ev_pool.empty()) { e = ctx->ev_pool.back(); ctx->ev_pool.pop_back(); }
            else cudaEventCreate(&e);
            return e;
        };
        ev.name = name; ev.a = get(); ev.b = get();
        cudaEventRecord(ev.a, ctx->stream);
    }
    ~KScope() {
        if (!on) return;
        cudaEventRecord(ev.b, ctx->stream);
        ctx->pending.push_back(ev);
    }
};
void flush_times(rb_ctx* ctx) {  // call after a stream sync
    for (KEvent& k : ctx->pending) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, k.a, k.b) != cudaSuccess) (void)cudaGetLastError();
        rb_kernel_time* slot = nullptr;
        for (auto& t : ctx->times)
            if (strcmp(t.name, k.name) == 0) slot = &t;
        if (!slot) {
            rb_kernel_time t{};
            strncpy(t.name, k.name, sizeof t.name - 1);
            ctx->times.push_back(t);
            slot = &ctx->times.back();
        }
        slot->launches++;
        slot->ms += ms;
        ctx->ev_pool.push_back(k.a);
        ctx->ev_pool.push_back(k.b);
    }
    ctx->pending.clear();
}

// queue "copy these device scalars into ctx->h_scalars[slot]" (u64 slots) on the context's stream
struct Publisher {
    PublishArgs a{};
    explicit Publisher(rb_ctx* ctx) { a.dst = reinterpret_cast<unsigned long long*>(ctx->h_scalars_dev); a.n = 0; }
    Publisher& u64(int slot, const void* src) { a.src[a.n] = src; a.slot[a.n] = (uint8_t)slot; a.wide[a.n] = 1; a.n++; return *this; }
    Publisher& u32(int slot, const void* src) { a.src[a.n] = src; a.slot[a.n] = (uint8_t)slot; a.wide[a.n] = 0; a.n++; return *this; }
    void go(cudaStream_t s) { launch_publish(a, s); }
};

int map_err(rb_ctx* ctx, rb_batch* b, uint64_t e_tok, uint64_t e_rec) {
    uint64_t best_rec = UINT64_MAX;
    uint32_t code = 0;
    if (e_tok != UINT64_MAX) {
        const uint64_t pos = e_tok >> 8;
        auto it = std::upper_bound(b->h_cigar_off.begin(), b->h_cigar_off.end(), pos);
        best_rec = (uint64_t)(it - b->h_cigar_off.begin()) - 1;
        code = (uint32_t)(e_tok & 0xFF);
    }
    if (e_rec != UINT64_MAX && (e_rec >> 8) < best_rec) {
        best_rec = e_rec >> 8;
        code = (uint32_t)(e_rec & 0xFF);
    }
    if (best_rec == UINT64_MAX) return RB_OK;
    best_rec = (!b->h_orig.empty() && best_rec < b->h_orig.size()) ? b->h_orig[best_rec] : best_rec + b->rec_base;  // the caller's record index
    ctx->err_rec = best_rec;
    switch (code) {
        case RE_CIGAR_PARSE: return fail(ctx, RB_ERR_REF_CIGAR_PARSE, "record %llu: Unable to parse cigar string (reference panics, paf.rs:399)", (unsigned long long)best_rec);
        case RE_INTEGRITY: return fail(ctx, RB_ERR_REF_INTEGRITY, "record %llu: CIGAR does not match the record's spans (check_integrity().unwrap(), paf.rs:70)", (unsigned long long)best_rec);
        case RE_STRIP_PANIC: return fail(ctx, RB_ERR_REF_STRIP, "record %llu: remove_trailing_indels panics in the reference (empty / leading-deletion / all-indel CIGAR)", (unsigned long long)best_rec);
        case RE_INDEX_PANIC: return fail(ctx, RB_ERR_REF_INDEX, "record %llu: Problem getting index in cigar (liftover.rs:31-49)", (unsigned long long)best_rec);
        default: return fail(ctx, RB_ERR_UNSUPPORTED, "record %llu: op length >= 2^28 or per-record sums >= 2^32", (unsigned long long)best_rec);
    }
}

RecInput rec_input(const rb_batch* b) {
    RecInput in{};
    const uint64_t* c = b->cols64.as<uint64_t>();
    const size_t n = b->n_rec;
    in.cigar_off = b->cigar_off.as<uint64_t>();
    in.q_len = c + 0 * n; in.q_st = c + 1 * n; in.q_en = c + 2 * n; in.t_len = c + 3 * n;
    in.t_st = c + 4 * n; in.t_en = c + 5 * n; in.mapq = c + 6 * n;
    in.strand = b->strand.as<uint8_t>();
    in.q_id = b->ids32.as<uint32_t>(); in.t_id = b->ids32.as<uint32_t>() + n;
    in.names_off = b->names_off.as<uint64_t>(); in.names = b->names.as<uint8_t>();
    in.n_rec = b->n_rec;
    in.no_text = b->invert ? 1u : 0u;
    return in;
}
WinView win_view(const rb_batch* self) {
    const rb_batch* b = self->wsrc ? self->wsrc : self;
    WinView w{};
    if (b->n_win == 0) return w;
    w.st = b->w_st.as<uint64_t>(); w.en = b->w_en.as<uint64_t>(); w.en_pm = w.en;
    w.ids_off = b->default_ids ? nullptr : b->w_ids_off.as<uint64_t>(); w.ids = b->default_ids ? nullptr : b->w_ids.as<uint8_t>();
    w.bed_row = b->w_bed_row.as<uint32_t>();
    w.cont_lo = b->cont_lo.as<uint32_t>(); w.cont_hi = b->cont_hi.as<uint32_t>();
    w.pair_win = nullptr;
    w.general = b->general ? 1u : 0u;
    return w;
}
StatsDev stats_view(const rb_batch* b, uint64_t n) {
    StatsDev s{};
    uint32_t* p = b->out_stats.as<uint32_t>();
    s.equal = p; s.diff = p + n; s.ins = p + 2 * n; s.del = p + 3 * n; s.ins_ev = p + 4 * n; s.del_ev = p + 5 * n;
    s.matches = p + 6 * n;
    s.id_m = reinterpret_cast<float*>(p + 7 * n); s.id_e = reinterpret_cast<float*>(p + 8 * n);
    s.id_a = reinterpret_cast<float*>(p + 9 * n);
    return s;
}
NumDev num_view(const rb_batch* b, uint64_t n) {
    NumDev d{};
    uint64_t* p = b->out_num.as<uint64_t>();
    d.q_st = p; d.q_en = p + n; d.t_st = p + 2 * n; d.t_en = p + 3 * n; d.nmatch = p + 4 * n; d.aln_len = p + 5 * n;
    d.rec_idx = reinterpret_cast<uint32_t*>(p + 6 * n);
    d.win_idx = d.rec_idx + n;
    return d;
}

// The pinned output of a call.  Rows block: a 64-byte front, the text, (rows + 1) line offsets and the numeric columns (6 x u64,
// then 2 x u32 per row: 56 B).  Stats block: the 10 columns of rb_stats_out (40 B per row).  Columns sit `cap` rows apart.
struct RowsOut {
    PinnedBlock *blk = nullptr, *sblk = nullptr;
    uint64_t cap = 0;
    size_t cap_text = 0;  // text bytes the rows block has room for
    size_t o_loff = 0, o_num = 0;
    bool text = false, num = false;

    int reserve(rb_ctx* ctx, uint64_t cap_rows, size_t text_bytes, uint32_t want, bool with_stats) {
        text = (want & (RB_WANT_TEXT | RB_WANT_STATS_TEXT)) != 0;  // (stats rows are the text)
        num = (want & RB_WANT_NUMERIC) != 0;
        cap = cap_rows;
        const size_t loff = text ? align_up((cap + 1) * 8, 64) : 0, nums = num ? align_up(cap * 56, 64) : 0;
        const size_t need = 64 + (text ? align_up(text_bytes + 1, 64) : 0) + loff + nums;
        blk = pinned_get(ctx, need);
        if (!blk) return fail(ctx, RB_ERR_OOM, "pinned allocation of %zu bytes failed", need);
        o_loff = 64 + (blk->cap - 64 - loff - nums) / 64 * 64;  // the text gets every byte the block has beyond the tables
        o_num = o_loff + loff;
        cap_text = text ? o_loff - 128 : 0;
        return with_stats ? reserve_stats(ctx, cap_rows) : RB_OK;
    }
    int reserve_stats(rb_ctx* ctx, uint64_t cap_rows) {
        cap = cap_rows;
        const size_t need = (size_t)cap * 40 + 64;
        sblk = pinned_get(ctx, need);
        if (!sblk) { release(); return fail(ctx, RB_ERR_OOM, "pinned allocation of %zu bytes failed", need); }
        return RB_OK;
    }
    // enqueue on `s`: rows [row_lo, row_lo + n_rows) of batch b (text bytes [byte_lo, byte_lo + n_bytes)) -> output rows from at_row
    // (text from at_byte).  The line offsets travel as they are on the device: rebasing them is the caller's.
    int copy_rows(rb_ctx* ctx, const rb_batch* b, uint64_t row_lo, uint64_t n_rows, uint64_t byte_lo, uint64_t n_bytes, uint64_t at_row,
                  uint64_t at_byte, cudaStream_t s) const {
        // device columns: row_stride apart after a liftover (0: n_out); without a rows block, rb_batch_stats' one row per record
        const uint64_t sk = !blk ? b->n_rec : b->row_stride ? b->row_stride : b->sum.n_out;
        uint8_t* base = blk ? static_cast<uint8_t*>(blk->p) : nullptr;
        if (text) {
            if (n_bytes) CU(cudaMemcpyAsync(base + 64 + at_byte, b->out_text.as<uint8_t>() + byte_lo, n_bytes, cudaMemcpyDeviceToHost, s));
            if (n_rows)
                CU(cudaMemcpyAsync(reinterpret_cast<uint64_t*>(base + o_loff) + at_row, b->out_line_off.as<uint64_t>() + row_lo, n_rows * 8,
                                   cudaMemcpyDeviceToHost, s));
        }
        if (!n_rows) return RB_OK;
        if (num) {  // one strided copy per table
            uint64_t* dn = reinterpret_cast<uint64_t*>(base + o_num);
            const uint64_t* sp = b->out_num.as<uint64_t>();
            CU(cudaMemcpy2DAsync(dn + at_row, cap * 8, sp + row_lo, sk * 8, n_rows * 8, 6, cudaMemcpyDeviceToHost, s));
            CU(cudaMemcpy2DAsync(reinterpret_cast<uint32_t*>(dn + 6 * cap) + at_row, cap * 4, reinterpret_cast<const uint32_t*>(sp + 6 * sk) + row_lo,
                                 sk * 4, n_rows * 4, 2, cudaMemcpyDeviceToHost, s));
        }
        if (sblk)
            CU(cudaMemcpy2DAsync(static_cast<uint32_t*>(sblk->p) + at_row, cap * 4, b->out_stats.as<uint32_t>() + row_lo, sk * 4, n_rows * 4, 10,
                                 cudaMemcpyDeviceToHost, s));
        return RB_OK;
    }
    // the caller's views, once every copy has landed (out / stats: nullable)
    void finish(rb_lift_out* out, rb_stats_out* stats, uint64_t n_rows, uint64_t n_bytes, uint64_t n_pairs) const {
        const uint64_t c = cap;
        if (out) {
            memset(out, 0, sizeof *out);
            out->n_out = n_rows; out->paf_nbytes = n_bytes; out->n_pairs = n_pairs; out->_owner = blk;
            uint8_t* base = static_cast<uint8_t*>(blk->p);
            if (text) {
                out->paf_text = base + 64;
                out->line_off = reinterpret_cast<uint64_t*>(base + o_loff);
                out->line_off[n_rows] = n_bytes;
                out->paf_text[n_bytes] = 0;
            }
            if (num) {
                uint64_t* p = reinterpret_cast<uint64_t*>(base + o_num);
                out->q_st = p; out->q_en = p + c; out->t_st = p + 2 * c; out->t_en = p + 3 * c; out->nmatch = p + 4 * c; out->aln_len = p + 5 * c;
                out->rec_idx = reinterpret_cast<uint32_t*>(p + 6 * c);
                out->win_idx = out->rec_idx + c;
            }
        }
        if (stats) {
            uint32_t* p = static_cast<uint32_t*>(sblk->p);
            memset(stats, 0, sizeof *stats);
            stats->n = n_rows;
            stats->equal = p; stats->diff = p + c; stats->ins = p + 2 * c; stats->del = p + 3 * c; stats->ins_events = p + 4 * c;
            stats->del_events = p + 5 * c; stats->matches = p + 6 * c;
            stats->id_by_matches = reinterpret_cast<float*>(p + 7 * c); stats->id_by_events = reinterpret_cast<float*>(p + 8 * c);
            stats->id_by_all = reinterpret_cast<float*>(p + 9 * c);
            stats->_owner = sblk;
        }
    }
    void release() {
        if (blk) blk->in_use = false;
        if (sblk) sblk->in_use = false;
        blk = sblk = nullptr;
    }
};

// RB_TOKSCAN=1 in the environment: tokeniser and sample scan as ONE kernel (k_tok_scan) instead of k_tokenise + k_samples.
// Parity-clean but opt-in: measured at C4 it takes 0.83 ms against 0.22 + 0.32 ms — a tile is 4 KB of text (~1 500 ops), so
// 32 700 tiles queue behind one another in the 64-byte-payload look-back, whose frontier moves 32 tiles per ~0.8 us round.
bool tok_scan_enabled() {
    static const bool on = getenv("RB_TOKSCAN") != nullptr;
    return on;
}

// tokenise + record offsets (shared by liftover and stats)
int run_tok(rb_ctx* ctx, rb_batch* b) {
    cudaStream_t s = ctx->stream;
    uint32_t* sc = ctx->scalars.as<uint32_t>();
    CU(cudaMemsetAsync(sc, 0, 4 * sizeof(uint32_t), s));
    CU(cudaMemsetAsync(sc + SC_ERR_TOK, 0xFF, 4 * sizeof(uint32_t), s));
    CU(cudaMemsetAsync(b->tile_state.p, 0, b->n_tiles * 8, s));
    CU(cudaMemsetAsync(b->heads.p, 0, (b->ops_bound / SAMPLE + 2) * 4, s));
    CU(cudaMemsetAsync(b->blk_state.p, 0, (b->ops_bound / SMP_OPS + 2) * 4, s));
    ErrSlots err{reinterpret_cast<unsigned long long*>(sc + SC_ERR_TOK), reinterpret_cast<unsigned long long*>(sc + SC_ERR_REC)};
    const uint8_t* text = b->text_raw.as<uint8_t>() + TEXT_FRONT_PAD;
    b->have_samples = !b->invert && tok_scan_enabled();
    if (b->have_samples) {  // tokeniser + sampled segmented scan in one pass over the text
        CU(cudaMemsetAsync(b->tile_first.p, 0xFF, b->n_tiles * 4, s));
        CU(cudaMemsetAsync(b->seg_state.p, 0, b->n_tiles * 4, s));
        KScope k(ctx, "k_tok_scan");
        launch_tok_scan(text, b->n_tiles, b->cigar_off.as<uint64_t>(), b->n_rec, b->ops.as<uint32_t>(), b->tile_state.as<unsigned long long>(),
                        sc + SC_TICKET_TOK, err, sc + SC_MISC, b->tile_first.as<uint32_t>(), b->head_pos.as<uint64_t>(), b->samples.as<Ctr>(),
                        b->seg_state.as<uint32_t>(), b->seg_agg.as<ScanPayload>(), b->seg_pre.as<ScanPayload>(), s);
    } else {
        KScope k(ctx, "k_tokenise");
        launch_tokenise(text, b->n_tiles, b->ops.as<uint32_t>(), b->tile_state.as<unsigned long long>(), sc + SC_TICKET_TOK, err,
                        sc + SC_MISC, s);
    }
    {
        KScope k(ctx, "k_rec_ops");
        launch_rec_ops(text, b->cigar_off.as<uint64_t>(), b->n_rec, b->tile_state.as<unsigned long long>(), b->op_off.as<uint64_t>(),
                       b->heads.as<uint32_t>(), err, s);
    }
    if (b->invert) {  // --qbed: query and target change roles (the columns were swapped at upload)
        KScope k(ctx, "k_invert_ops");
        launch_invert_ops(b->ops.as<uint32_t>(), b->op_off.as<uint64_t>(), b->n_rec, b->strand.as<uint8_t>(), b->ops_bound, s);
    }
    CU(cudaGetLastError());
    return RB_OK;
}

// sampled segmented scan of the prefix counters; `la` != nullptr: fused with the window-boundary resolution (fast path)
int run_scan(rb_ctx* ctx, rb_batch* b, const LiftArgs* la, bool no_subs = false) {
    cudaStream_t s = ctx->stream;
    uint32_t* sc = ctx->scalars.as<uint32_t>();
    if (!la && b->have_samples) return RB_OK;  // k_tok_scan wrote them
    {
        KScope k(ctx, la ? "k_scan_lift" : "k_samples");
        launch_scan_lift(la != nullptr, b->ops.as<uint32_t>(), b->op_off.as<uint64_t>() + b->n_rec, b->ops_bound, b->heads.as<uint32_t>(),
                         b->samples.as<Ctr>(), b->blk_state.as<uint32_t>(), b->blk_agg.as<ScanPayload>(), b->blk_pre.as<ScanPayload>(),
                         sc + SC_TICKET_SMP, la ? *la : LiftArgs{}, s, no_subs && !la);
    }
    CU(cudaGetLastError());
    return RB_OK;
}

}  // namespace

// =================================================================================================
extern "C" {

const char* rb_version(void) { return "rbcuda 0.1 (sm_100a)"; }

// Page-locks [ptr, ptr + nbytes) in pieces of <= 1 GiB (a single cudaHostRegister of tens of GB can fail where the
// pieces succeed); rb_host_unregister undoes all pieces of that call.
static constexpr uint64_t REG_PIECE = 1ull << 30;
static std::mutex g_reg_mu;
static std::vector<std::pair<void*, std::vector<void*>>> g_reg;  // base pointer -> registered pieces

int rb_host_register(void* ptr, uint64_t nbytes) {
    if (!ptr || !nbytes) return RB_ERR_BAD_ARG;
    // pieces are cut at absolute 1 GiB-aligned addresses: no page is registered twice, and h2d_copy() below cuts its
    // transfers at the same addresses (one copy must not span two registrations)
    std::vector<void*> done;
    const uint64_t a0 = reinterpret_cast<uintptr_t>(ptr), a1 = a0 + nbytes;
    for (uint64_t a = a0; a < a1;) {
        uint64_t e = (a / REG_PIECE + 1) * REG_PIECE;
        if (e > a1) e = a1;
        if (cudaHostRegister(reinterpret_cast<void*>(a), e - a, cudaHostRegisterDefault) != cudaSuccess) {
            (void)cudaGetLastError();
            for (void* q : done) cudaHostUnregister(q);
            return RB_ERR_CUDA;
        }
        done.push_back(reinterpret_cast<void*>(a));
        a = e;
    }
    std::lock_guard<std::mutex> lk(g_reg_mu);
    g_reg.emplace_back(ptr, std::move(done));
    return RB_OK;
}
int rb_host_unregister(void* ptr) {
    if (!ptr) return RB_ERR_BAD_ARG;
    std::vector<void*> pieces;
    {
        std::lock_guard<std::mutex> lk(g_reg_mu);
        for (size_t i = 0; i < g_reg.size(); i++)
            if (g_reg[i].first == ptr) { pieces = std::move(g_reg[i].second); g_reg.erase(g_reg.begin() + (long)i); break; }
    }
    if (pieces.empty()) return RB_ERR_BAD_ARG;
    int rc = RB_OK;
    for (void* q : pieces)
        if (cudaHostUnregister(q) != cudaSuccess) { (void)cudaGetLastError(); rc = RB_ERR_CUDA; }
    return rc;
}

static rb_ctx* ctx_create_one(int dev, int* status) {
    auto set = [&](int s) { if (status) *status = s; };
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) {
        (void)cudaGetLastError();
        set(RB_ERR_NO_DEVICE);
        return nullptr;
    }
    cudaDeviceProp prop{};
    if (dev < 0 || dev >= count || cudaGetDeviceProperties(&prop, dev) != cudaSuccess || prop.major != 10) {
        (void)cudaGetLastError();
        set(RB_ERR_NO_DEVICE);  // kernels are compiled for sm_100a only; there is no fallback
        return nullptr;
    }
    rb_ctx* ctx = new rb_ctx();
    ctx->device = dev;
    ctx->fused_emit = getenv("RB_NO_FUSED_EMIT") == nullptr;
    if (const char* e = getenv("RB_MULTI_MIN_BYTES")) ctx->multi_min_bytes = strtoull(e, nullptr, 10);
    cudaSetDevice(dev);
    if (init_kernel_attrs() != 0 || cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess ||
        ctx->scalars.ensure(SC_WORDS * 4) != cudaSuccess || cudaHostAlloc(&ctx->h_scalars, 256, cudaHostAllocMapped) != cudaSuccess ||
        cudaHostGetDevicePointer(&ctx->h_scalars_dev, ctx->h_scalars, 0) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->ev_win, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->ev_wfirst, cudaEventDisableTiming) != cudaSuccess) {
        (void)cudaGetLastError();
        delete ctx;
        set(RB_ERR_CUDA);
        return nullptr;
    }
    set(RB_OK);
    return ctx;
}

// device_ids[0 .. n_devices): the GPUs of this context (NULL / 0: device 0).  With more than one, rb_liftover and rb_stats
// partition the records over them (contiguous runs of the emission order, balanced on CIGAR bytes; one host thread and
// stream set per device; no exchange between the devices) and merge the rows into ONE output in the reference's emission
// order; every other call runs on the first device.  The same id may be listed twice (two contexts on one GPU).
rb_ctx* rb_ctx_create(const int* device_ids, int n_devices, int* status) {
    const int dev0 = (device_ids && n_devices > 0) ? device_ids[0] : 0;
    rb_ctx* ctx = ctx_create_one(dev0, status);
    if (!ctx) return nullptr;
    for (int i = 1; device_ids && i < n_devices; i++) {
        rb_ctx* p = ctx_create_one(device_ids[i], status);
        if (!p) {
            rb_ctx_destroy(ctx);
            return nullptr;
        }
        ctx->peers.push_back(p);
    }
    cudaSetDevice(dev0);
    return ctx;
}

void rb_batch_free(rb_ctx* ctx, rb_batch* b) {
    if (!b) return;
    if (ctx) cudaSetDevice(ctx->device);
    if (ctx && b->busy) cudaStreamSynchronize(ctx->stream);
    DevBuf* all[] = {&b->text_raw, &b->cigar_off, &b->cols64, &b->strand, &b->ids32, &b->names, &b->names_off, &b->rec_order,
                     &b->rec_rank, &b->w_st, &b->w_en, &b->w_ids_off, &b->w_ids, &b->w_bed_row, &b->w_tid, &b->cont_lo, &b->cont_hi, &b->ops,
                     &b->tile_state, &b->heads, &b->samples, &b->blk_state, &b->blk_agg, &b->blk_pre, &b->op_off, &b->recs,
                     &b->pair_cnt, &b->pair_off, &b->pair_res, &b->line_len, &b->line_off, &b->out_idx, &b->pair_win, &b->ln_state,
                     &b->ln_agg, &b->ln_pre, &b->half_s, &b->half_e, &b->plans, &b->orig_idx, &b->bp_cnt, &b->bp_off, &b->bp_end, &b->bp_next, &b->rec_bp, &b->trim_qp, &b->trim_wp, &b->trim_ap, &b->trim_views,
                     &b->trim_sel, &b->trim_out, &b->trim_drop, &b->tile_first, &b->head_pos, &b->seg_state, &b->seg_agg, &b->seg_pre, &b->out_text, &b->out_line_off, &b->out_num, &b->out_stats, &b->blk_flags, &b->emit_totals};
    for (DevBuf* d : all) d->release();
    b->stage.release();
    b->wstage.release();
    b->rec_out.release();
    delete b;
}

void rb_ctx_destroy(rb_ctx* ctx) {
    if (!ctx) return;
    for (rb_ctx* p : ctx->peers) rb_ctx_destroy(p);
    ctx->peers.clear();
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
    if (ctx->up_stream) cudaStreamSynchronize(ctx->up_stream);
    if (ctx->scratch) rb_batch_free(ctx, ctx->scratch);
    for (int k = 0; k < 2; k++) {
        if (ctx->slice[k]) rb_batch_free(ctx, ctx->slice[k]);
        if (ctx->ev_done[k]) cudaEventDestroy(ctx->ev_done[k]);
        if (ctx->ev_d2h[k]) cudaEventDestroy(ctx->ev_d2h[k]);
    }
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->up_stream) cudaStreamDestroy(ctx->up_stream);
    for (int k = 0; k < 2; k++) if (ctx->ev_up[k]) cudaEventDestroy(ctx->ev_up[k]);
    if (ctx->ev_win) cudaEventDestroy(ctx->ev_win);
    if (ctx->ev_wfirst) cudaEventDestroy(ctx->ev_wfirst);
    for (PinnedBlock* b : ctx->pinned) { pinned_block_free(b); delete b; }
    for (cudaEvent_t e : ctx->ev_pool) cudaEventDestroy(e);
    ctx->scalars.release();
    if (ctx->h_scalars) cudaFreeHost(ctx->h_scalars);
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

const char* rb_last_error(const rb_ctx* ctx) { return ctx ? ctx->err.c_str() : "no context (no usable sm_100 device?)"; }

int rb_ctx_set_stream(rb_ctx* ctx, void* cuda_stream) {
    if (!ctx) return RB_ERR_BAD_ARG;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    if (cuda_stream) {
        ctx->stream = (cudaStream_t)cuda_stream;
        ctx->own_stream = false;
    } else {
        ctx->own_stream = true;
        if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) return fail(ctx, RB_ERR_CUDA, "cudaStreamCreate");
    }
    return RB_OK;
}

int rb_ctx_set_slicing(rb_ctx* ctx, uint64_t min_slice_bytes) {
    if (!ctx) return RB_ERR_BAD_ARG;
    ctx->slice_min_bytes = min_slice_bytes;
    return RB_OK;
}

int rb_ctx_set_lift_mode(rb_ctx* ctx, int mode) {
    if (!ctx || (mode != RB_LIFT_SEARCH && mode != RB_LIFT_STREAM)) return RB_ERR_BAD_ARG;
    ctx->lift_mode = mode;
    return RB_OK;
}

int rb_ctx_set_profiling(rb_ctx* ctx, int on) {
    if (!ctx) return RB_ERR_BAD_ARG;
    ctx->profiling = on != 0;
    return RB_OK;
}

int rb_ctx_kernel_times(rb_ctx* ctx, rb_kernel_time* out, int cap, int reset) {
    if (!ctx) return 0;
    int n = 0;
    for (auto& t : ctx->times) {
        if (n < cap && out) out[n] = t;
        n++;
    }
    if (reset) ctx->times.clear();
    return n;
}

int rb_sort_windows(uint32_t n_win, const uint32_t* t_id, const uint64_t* st, uint32_t* perm_out) {
    if (n_win && (!t_id || !st || !perm_out)) return RB_ERR_BAD_ARG;
    for (uint32_t i = 0; i < n_win; i++) perm_out[i] = i;
    std::stable_sort(perm_out, perm_out + n_win, [&](uint32_t a, uint32_t b) {
        if (t_id[a] != t_id[b]) return t_id[a] < t_id[b];
        return st[a] < st[b];
    });
    return RB_OK;
}

// -------------------------------------------------------------------------------------------------
// Host -> HBM.  Everything is enqueued on the context's stream without a host synchronisation: the big CIGAR
// copy goes first so that the host-side checks of the window table (3 M rows at 1 kb windows) run while the DMA
// engine is busy.  Host staging that must outlive the call lives in the batch.
// records [r0, r1) of R: the CIGAR text, the one big copy — issued before any host-side work
// Which records of the caller's arrays a batch holds: a run [r0, r0 + n), or the list idx[0..n) (slices of a PAF whose
// file order is not the emission order: the list is in emission order and is gathered run by run).
struct RecSel {
    const uint32_t* idx;
    uint32_t r0, n;
    uint32_t at(uint32_t i) const { return idx ? idx[i] : r0 + i; }
};

// n_bytes of CIGAR text: the tokeniser's tiles and op bound; returns the bytes text_raw holds behind its front pad (the text, then
// '0' up to the end of the last tile and 32 more)
static size_t text_layout(rb_batch* b, uint64_t n_bytes) {
    b->n_bytes = n_bytes;
    b->n_tiles = b->n_bytes / TOK_TILE + 1;
    b->ops_bound = b->n_bytes / 2 + 1;
    return b->n_tiles * (size_t)TOK_TILE + 32;
}

static int upload_cigar(rb_ctx* ctx, rb_batch* b, const rb_records* R, RecSel sel) {
    cudaStream_t s = ctx->upload_on ? ctx->upload_on : ctx->stream;
    if (!R || (R->n_rec && (!R->cigar_off || !R->q_len || !R->q_st || !R->q_en || !R->t_len || !R->t_st || !R->t_en || !R->mapq ||
                            !R->strand || !R->q_id || !R->t_id || !R->names_off)) ||
        (R->cigar_nbytes && !R->cigar))
        return fail(ctx, RB_ERR_BAD_ARG, "rb_records: null column");
    if (R->n_rec && (R->cigar_off[0] != 0 || R->cigar_off[R->n_rec] != R->cigar_nbytes)) return fail(ctx, RB_ERR_BAD_ARG, "cigar_off must span [0, cigar_nbytes]");
    if (!R->n_rec && R->cigar_nbytes) return fail(ctx, RB_ERR_BAD_ARG, "cigar_off must span [0, cigar_nbytes]");
    const uint32_t n = sel.n;
    if (b->busy) { CU(cudaStreamSynchronize(s)); b->busy = false; }  // the previous call's copies read the staging below
    // runs of consecutive records -> one copy each; h_cigar_off = offsets inside the batch's own text
    b->h_cigar_off.resize((size_t)n + 1);
    b->h_cigar_off[0] = 0;
    for (uint32_t i = 0; i < n; i++) {
        const uint32_t r = sel.at(i);
        if (r >= R->n_rec || R->cigar_off[r] > R->cigar_off[r + 1] || R->cigar_off[r + 1] > R->cigar_nbytes)
            return fail(ctx, RB_ERR_BAD_ARG, "cigar_off not monotone at record %u", r);
        b->h_cigar_off[i + 1] = b->h_cigar_off[i] + (R->cigar_off[r + 1] - R->cigar_off[r]);
    }
    b->n_rec = n; b->n_names = R->n_names;
    b->rec_base = sel.idx ? 0 : sel.r0; b->byte_base = 0;
    b->invert = ctx->invert;
    b->have_lift = b->have_stats = false;
    const size_t padded = text_layout(b, b->h_cigar_off[n]);
    CU(b->text_raw.ensure(TEXT_FRONT_PAD + padded));
    uint8_t* raw = b->text_raw.as<uint8_t>();
    CU(cudaMemsetAsync(raw, 0xFF, TEXT_FRONT_PAD, s));
    for (uint32_t i = 0; i < n;) {
        uint32_t j = i;
        while (j + 1 < n && sel.at(j + 1) == sel.at(j) + 1) j++;
        const uint64_t src0 = R->cigar_off[sel.at(i)], src1 = R->cigar_off[sel.at(j) + 1];
        if (src1 > src0)
            CU(h2d_copy(raw + TEXT_FRONT_PAD + b->h_cigar_off[i], R->cigar + src0, src1 - src0, s));
        i = j + 1;
    }
    CU(cudaMemsetAsync(raw + TEXT_FRONT_PAD + b->n_bytes, '0', padded - b->n_bytes, s));
    b->busy = true;
    return RB_OK;
}

// step 1a (host only): argument checks, device buffers, contig ranges
static int windows_prepare(rb_ctx* ctx, rb_batch* b, const rb_records* R, const rb_windows* W) {
    b->n_win = W ? W->n_win : 0;
    b->wsrc = nullptr;
    b->general = false; b->default_ids = false; b->win_pending = false;
    if (!(W && W->n_win)) return RB_OK;
    const uint32_t nw = W->n_win;
    if (!W->t_id || !W->st || !W->en || !W->bed_row || (W->ids_off && !W->ids)) return fail(ctx, RB_ERR_BAD_ARG, "rb_windows: null column");
    b->default_ids = (W->ids_off == nullptr);
    CU(b->w_st.ensure((size_t)nw * 8)); CU(b->w_en.ensure((size_t)nw * 8)); CU(b->w_bed_row.ensure((size_t)nw * 4));
    CU(b->w_tid.ensure((size_t)nw * 4));
    CU(b->cont_lo.ensure((size_t)(R->n_names + 1) * 4)); CU(b->cont_hi.ensure((size_t)(R->n_names + 1) * 4));
    // contig ranges: t_id is sorted (verified on the device; an unsorted table only yields ranges nobody will use)
    b->h_clo.assign(R->n_names + 1, 0); b->h_chi.assign(R->n_names + 1, 0);
    const uint32_t* tid = W->t_id;
    uint32_t i = 0;
    while (i < nw) {  // gallop from contig to contig: O(contigs * log n_win) host reads
        const uint32_t t = tid[i];
        const uint32_t j = (uint32_t)(std::upper_bound(tid + i, tid + nw, t) - tid);
        if (t < R->n_names) { b->h_clo[t] = i; b->h_chi[t] = j; }
        i = j > i ? j : i + 1;
    }
    return RB_OK;
}

// step 1b: rows [lo, hi) of the caller's (sorted) tables -> the same rows of the device tables
static int windows_upload_rows(rb_ctx* ctx, rb_batch* b, const rb_windows* W, uint32_t lo, uint32_t hi, cudaStream_t s) {
    if (hi <= lo) return RB_OK;
    const size_t n = hi - lo;
    CU(h2d_copy(b->w_tid.as<uint32_t>() + lo, W->t_id + lo, n * 4, s));
    CU(h2d_copy(b->w_st.as<uint64_t>() + lo, W->st + lo, n * 8, s));
    CU(h2d_copy(b->w_en.as<uint64_t>() + lo, W->en + lo, n * 8, s));
    CU(h2d_copy(b->w_bed_row.as<uint32_t>() + lo, W->bed_row + lo, n * 4, s));
    b->busy = true;
    return RB_OK;
}

// step 1c: what every kernel that touches windows needs besides the rows: contig ranges and (if given) the ids
static int windows_upload_aux(rb_ctx* ctx, rb_batch* b, const rb_records* R, const rb_windows* W, cudaStream_t s) {
    if (!b->n_win) return RB_OK;
    const uint32_t nw = b->n_win;
    if (!b->default_ids) {
        const uint64_t ids_bytes = W->ids_off[nw];
        CU(b->w_ids_off.ensure((size_t)(nw + 1) * 8)); CU(b->w_ids.ensure(ids_bytes + 8));
        CU(h2d_copy(b->w_ids_off.p, W->ids_off, (size_t)(nw + 1) * 8, s));
        if (ids_bytes) CU(h2d_copy(b->w_ids.p, W->ids, ids_bytes, s));
    }
    const size_t cbytes = (size_t)(R->n_names + 1) * 4;
    CU(b->wstage.ensure(2 * cbytes));
    memcpy(b->wstage.p, b->h_clo.data(), cbytes);
    memcpy(b->wstage.p + cbytes, b->h_chi.data(), cbytes);
    CU(cudaMemcpyAsync(b->cont_lo.p, b->wstage.p, cbytes, cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(b->cont_hi.p, b->wstage.p + cbytes, cbytes, cudaMemcpyHostToDevice, s));
    b->busy = true;
    return RB_OK;
}

// step 1d: check kernel over the whole table (all rows must have been enqueued on `s` or on streams `s` waits for);
// its verdict is read by upload_windows_end.  The host never walks the table (3 M rows at 1 kb windows = 75 MB of host
// reads); it only binary-searches t_id for the contig ranges.
static int windows_check(rb_ctx* ctx, rb_batch* b, const rb_records* R, cudaStream_t s) {
    if (!b->n_win) return RB_OK;
    uint32_t* sc = ctx->scalars.as<uint32_t>();
    CU(cudaMemsetAsync(sc + SC_WINFLAGS, 0, 4, s));
    launch_win_check(b->w_tid.as<uint32_t>(), b->w_st.as<uint64_t>(), b->w_en.as<uint64_t>(), b->w_bed_row.as<uint32_t>(), b->n_win,
                     R->n_names, sc + SC_WINFLAGS, s);
    PublishArgs a{};
    a.dst = reinterpret_cast<unsigned long long*>(ctx->h_scalars_dev);
    a.src[0] = sc + SC_WINFLAGS; a.slot[0] = 16; a.wide[0] = 0; a.n = 1;
    launch_publish(a, s);
    CU(cudaEventRecord(ctx->ev_win, s));
    b->win_pending = true;
    return RB_OK;
}

// The window tables, step 1 for the single-batch path: everything on the context's stream
static int upload_windows_begin(rb_ctx* ctx, rb_batch* b, const rb_records* R, const rb_windows* W) {
    cudaStream_t s = ctx->stream;
    int rc = windows_prepare(ctx, b, R, W);
    if (rc == RB_OK) rc = windows_upload_rows(ctx, b, W, 0, b->n_win, s);
    if (rc == RB_OK) rc = windows_check(ctx, b, R, s);
    if (rc == RB_OK) rc = windows_upload_aux(ctx, b, R, W, s);
    return rc;
}

// step 2: wait for the verdict of the check kernel; the rare general layout (BED rows whose file order is not the
// sorted order, or nested rows) re-uploads the tables in BED file order per contig (Q5)
static int upload_windows_end(rb_ctx* ctx, rb_batch* b, const rb_records* R, const rb_windows* W) {
    if (!b->win_pending) return RB_OK;
    b->win_pending = false;
    cudaStream_t s = ctx->stream;
    CU(cudaEventSynchronize(ctx->ev_win));
    const uint32_t flags = (uint32_t)reinterpret_cast<volatile uint64_t*>(ctx->h_scalars)[16];
    if (flags & 1u) return fail(ctx, RB_ERR_BAD_ARG, "windows must be sorted by (t_id, st) with t_id < n_names (see rb_sort_windows)");
    b->general = (flags & 2u) != 0;
    if (!b->general) return RB_OK;
    const uint32_t nw = W->n_win;
    std::vector<uint32_t> perm(nw);
    for (uint32_t i = 0; i < nw; i++) perm[i] = i;
    std::stable_sort(perm.begin(), perm.end(), [&](uint32_t a, uint32_t c) {
        if (W->t_id[a] != W->t_id[c]) return W->t_id[a] < W->t_id[c];
        return W->bed_row[a] < W->bed_row[c];
    });
    auto& g = b->h_gen;
    g.st.resize(nw); g.en.resize(nw); g.row.resize(nw);
    for (uint32_t i = 0; i < nw; i++) {
        const uint32_t j = perm[i];
        g.st[i] = W->st[j]; g.en[i] = W->en[j]; g.row[i] = W->bed_row[j];
    }
    CU(cudaMemcpyAsync(b->w_st.p, g.st.data(), (size_t)nw * 8, cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(b->w_en.p, g.en.data(), (size_t)nw * 8, cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(b->w_bed_row.p, g.row.data(), (size_t)nw * 4, cudaMemcpyHostToDevice, s));
    if (!b->default_ids) {
        g.off.resize(nw + 1);
        g.off[0] = 0;
        for (uint32_t i = 0; i < nw; i++) g.off[i + 1] = g.off[i] + (W->ids_off[perm[i] + 1] - W->ids_off[perm[i]]);
        g.ids.resize(g.off[nw] + 1);
        for (uint32_t i = 0; i < nw; i++) {
            const uint32_t j = perm[i];
            memcpy(g.ids.data() + g.off[i], W->ids + W->ids_off[j], W->ids_off[j + 1] - W->ids_off[j]);
        }
        CU(cudaMemcpyAsync(b->w_ids_off.p, g.off.data(), (size_t)(nw + 1) * 8, cudaMemcpyHostToDevice, s));
        if (g.off[nw]) CU(cudaMemcpyAsync(b->w_ids.p, g.ids.data(), g.off[nw], cudaMemcpyHostToDevice, s));
    }
    b->busy = true;
    (void)R;
    return RB_OK;
}

// device buffers for n records (columns, emission order, and what the kernels of every later call write); text_layout first
static int ensure_rec_buffers(rb_ctx* ctx, rb_batch* b, uint32_t n) {
    CU(b->cigar_off.ensure((size_t)(n + 1) * 8));
    CU(b->cols64.ensure((size_t)n * 7 * 8 + 8));
    CU(b->strand.ensure(n + 8));
    CU(b->ids32.ensure((size_t)n * 2 * 4 + 8));
    CU(b->rec_order.ensure((size_t)n * 4 + 8));
    CU(b->rec_rank.ensure((size_t)n * 4 + 8));
    CU(b->ops.ensure(b->ops_bound * 4 + 64));
    CU(b->tile_state.ensure(b->n_tiles * 8));
    if (tok_scan_enabled()) {
        CU(b->tile_first.ensure(b->n_tiles * 4));
        CU(b->head_pos.ensure((size_t)(n + 1) * 8));
        CU(b->seg_state.ensure(b->n_tiles * 4));
        CU(b->seg_agg.ensure(b->n_tiles * sizeof(ScanPayload)));
        CU(b->seg_pre.ensure(b->n_tiles * sizeof(ScanPayload)));
    }
    CU(b->heads.ensure((b->ops_bound / SAMPLE + 2) * 4));
    CU(b->samples.ensure((b->ops_bound / SAMPLE + 2) * SUBS * sizeof(Ctr)));
    const size_t smp_blocks = b->ops_bound / SMP_OPS + 2;
    CU(b->blk_state.ensure(smp_blocks * 4));
    CU(b->blk_agg.ensure(smp_blocks * sizeof(ScanPayload)));
    CU(b->blk_pre.ensure(smp_blocks * sizeof(ScanPayload)));
    CU(b->op_off.ensure((size_t)(n + 1) * 8));
    CU(b->recs.ensure((size_t)n * sizeof(RecInfo) + 8));
    CU(b->pair_cnt.ensure((size_t)n * 4 + 8));
    CU(b->pair_off.ensure((size_t)(n + 1) * 8));
    return RB_OK;
}

// emission order (liftover.rs:151-164): contigs by first appearance of t_name, records in file order inside (file_order: the
// identity); order[k] = the record emitted k-th, rank = its inverse.  contig_rank (nullable): the contigs' ranks by first appearance
// in a larger file these records are part of (rb_liftover_text: one device's share), in place of their first appearance here.
static void emission_ranks(const uint32_t* tid, uint32_t n, uint32_t n_names, bool file_order, const uint32_t* contig_rank, uint32_t* order,
                           uint32_t* rank) {
    std::vector<int64_t> first(contig_rank ? 0 : n_names, -1);
    std::vector<uint32_t> cnt(contig_rank ? n_names : 0, 0);
    std::vector<uint32_t> grp(n);
    for (uint32_t i = 0; i < n; i++) {
        if (contig_rank) {
            grp[i] = contig_rank[tid[i]];
        } else {
            int64_t& f = first[tid[i]];
            if (f < 0) { f = (int64_t)cnt.size(); cnt.push_back(0); }
            grp[i] = (uint32_t)f;
        }
        cnt[grp[i]]++;
    }
    std::vector<uint32_t> start(cnt.size() + 1, 0);
    for (size_t g = 0; g < cnt.size(); g++) start[g + 1] = start[g] + cnt[g];
    for (uint32_t i = 0; i < n; i++) {
        const uint32_t k = file_order ? i : start[grp[i]]++;
        order[k] = i;
        rank[i] = k;
    }
}

// records [r0, r1) of R: numeric columns, names, emission order (small)
static int upload_columns(rb_ctx* ctx, rb_batch* b, const rb_records* R, RecSel sel) {
    cudaStream_t s = ctx->upload_on ? ctx->upload_on : ctx->stream;
    const uint32_t n = sel.n;
    for (uint32_t i = 0; i < n; i++) {
        const uint32_t r = sel.at(i);
        if (R->q_id[r] >= R->n_names || R->t_id[r] >= R->n_names) return fail(ctx, RB_ERR_BAD_ARG, "name id out of range at record %u", r);
    }
    int rc = ensure_rec_buffers(ctx, b, n);
    if (rc != RB_OK) return rc;
    CU(b->names_off.ensure((size_t)(R->n_names + 1) * 8));
    const uint64_t names_bytes = R->n_names ? R->names_off[R->n_names] : 0;
    CU(b->names.ensure(names_bytes + 8));


    // gather every small column into the batch's pinned staging area, then one asynchronous copy each
    const uint64_t* cols[7] = {R->q_len, R->q_st, R->q_en, R->t_len, R->t_st, R->t_en, R->mapq};
    const size_t nn = R->n_names;
    const size_t o_off = 0, o_cols = o_off + align_up((size_t)(n + 1) * 8, 64), o_qid = o_cols + align_up((size_t)n * 7 * 8, 64),
                 o_tid = o_qid + align_up((size_t)n * 4, 64), o_strand = o_tid + align_up((size_t)n * 4, 64),
                 o_noff = o_strand + align_up((size_t)n, 64), o_names = o_noff + align_up((nn + 1) * 8, 64),
                 o_order = o_names + align_up(names_bytes + 1, 64), o_rank = o_order + align_up((size_t)n * 4, 64),
                 o_orig = o_rank + align_up((size_t)n * 4, 64), o_end = o_orig + align_up((size_t)n * 4, 64);
    CU(b->stage.ensure(o_end));
    uint8_t* sp = b->stage.p;
    uint64_t* s_off = reinterpret_cast<uint64_t*>(sp + o_off);
    uint64_t* s_cols = reinterpret_cast<uint64_t*>(sp + o_cols);
    uint32_t* s_qid = reinterpret_cast<uint32_t*>(sp + o_qid);
    uint32_t* s_tid = reinterpret_cast<uint32_t*>(sp + o_tid);
    uint8_t* s_strand = sp + o_strand;
    uint32_t* s_orig = reinterpret_cast<uint32_t*>(sp + o_orig);
    memcpy(s_off, b->h_cigar_off.data(), (size_t)(n + 1) * 8);
    b->h_orig.clear();
    if (sel.idx) {
        b->h_orig.assign(sel.idx, sel.idx + n);
        for (uint32_t i = 0; i < n; i++) {
            const uint32_t r = sel.idx[i];
            for (int k = 0; k < 7; k++) s_cols[(size_t)k * n + i] = cols[k][r];
            s_strand[i] = R->strand[r]; s_qid[i] = R->q_id[r]; s_tid[i] = R->t_id[r]; s_orig[i] = r;
        }
        CU(b->orig_idx.ensure((size_t)n * 4 + 8));
        if (n) CU(cudaMemcpyAsync(b->orig_idx.p, s_orig, (size_t)n * 4, cudaMemcpyHostToDevice, s));
    } else if (n) {
        for (int k = 0; k < 7; k++) memcpy(s_cols + (size_t)k * n, cols[k] + sel.r0, (size_t)n * 8);
        memcpy(s_strand, R->strand + sel.r0, n);
        memcpy(s_qid, R->q_id + sel.r0, (size_t)n * 4);
        memcpy(s_tid, R->t_id + sel.r0, (size_t)n * 4);
    }
    const uint32_t* h_tid = s_tid;
    CU(cudaMemcpyAsync(b->cigar_off.p, s_off, (size_t)(n + 1) * 8, cudaMemcpyHostToDevice, s));
    if (n) {
        CU(cudaMemcpyAsync(b->cols64.p, s_cols, (size_t)n * 7 * 8, cudaMemcpyHostToDevice, s));
        CU(cudaMemcpyAsync(b->strand.p, s_strand, n, cudaMemcpyHostToDevice, s));
        CU(cudaMemcpyAsync(b->ids32.as<uint32_t>(), s_qid, (size_t)n * 4, cudaMemcpyHostToDevice, s));
        CU(cudaMemcpyAsync(b->ids32.as<uint32_t>() + n, s_tid, (size_t)n * 4, cudaMemcpyHostToDevice, s));
    }
    if (nn) {
        memcpy(sp + o_noff, R->names_off, (nn + 1) * 8);
        if (names_bytes) memcpy(sp + o_names, R->names, names_bytes);
        CU(cudaMemcpyAsync(b->names_off.p, sp + o_noff, (nn + 1) * 8, cudaMemcpyHostToDevice, s));
        if (names_bytes) CU(cudaMemcpyAsync(b->names.p, sp + o_names, names_bytes, cudaMemcpyHostToDevice, s));
    }
    uint32_t* s_order = reinterpret_cast<uint32_t*>(sp + o_order);
    uint32_t* s_rank = reinterpret_cast<uint32_t*>(sp + o_rank);

    emission_ranks(h_tid, n, R->n_names, b->file_order, nullptr, s_order, s_rank);
    if (n) {
        CU(cudaMemcpyAsync(b->rec_order.p, s_order, (size_t)n * 4, cudaMemcpyHostToDevice, s));
        CU(cudaMemcpyAsync(b->rec_rank.p, s_rank, (size_t)n * 4, cudaMemcpyHostToDevice, s));
    }
    b->sum = rb_summary{};
    b->sum.cigar_bytes = b->n_bytes;
    return RB_OK;
}

static int upload_into_impl(rb_ctx* ctx, rb_batch* b, const rb_records* R, const rb_windows* W) {
    const RecSel all{nullptr, 0, R ? R->n_rec : 0};
    int rc = upload_cigar(ctx, b, R, all);  // validates R
    if (rc == RB_OK) rc = upload_windows_begin(ctx, b, R, W);
    if (rc == RB_OK) rc = upload_columns(ctx, b, R, all);
    if (rc == RB_OK) rc = upload_windows_end(ctx, b, R, W);
    return rc;
}

static int upload_into(rb_ctx* ctx, rb_batch* b, const rb_records* R, const rb_windows* W) {
    const int rc = upload_into_impl(ctx, b, R, W);
    if (rc != RB_OK && b->busy) {  // copies out of the caller's buffers may be in flight: do not hand them back early
        cudaStreamSynchronize(ctx->stream);
        b->busy = false;
    }
    return rc;
}

rb_batch* rb_batch_upload(rb_ctx* ctx, const rb_records* recs, const rb_windows* wins, int* status) {
    auto set = [&](int s) { if (status) *status = s; };
    if (!ctx) { set(RB_ERR_NO_DEVICE); return nullptr; }
    cudaSetDevice(ctx->device);
    rb_batch* b = new rb_batch();
    int rc = upload_into(ctx, b, recs, wins);
    if (rc == RB_OK && cudaStreamSynchronize(ctx->stream) != cudaSuccess) {  // the caller may reuse its buffers after this call
        (void)cudaGetLastError();
        rc = fail(ctx, RB_ERR_CUDA, "upload failed");
    }
    b->busy = false;
    set(rc);
    if (rc != RB_OK) { rb_batch_free(ctx, b); return nullptr; }
    return b;
}

int rb_batch_stats(rb_ctx* ctx, rb_batch* b, rb_summary* summary) {
    if (!ctx || !b) return RB_ERR_BAD_ARG;
    cudaSetDevice(ctx->device);
    cudaStream_t s = ctx->stream;
    int rc = run_tok(ctx, b);
    if (rc != RB_OK) return rc;
    rc = run_scan(ctx, b, nullptr);
    if (rc != RB_OK) return rc;
    uint32_t* sc = ctx->scalars.as<uint32_t>();
    ErrSlots err{reinterpret_cast<unsigned long long*>(sc + SC_ERR_TOK), reinterpret_cast<unsigned long long*>(sc + SC_ERR_REC)};
    CU(b->out_stats.ensure((size_t)b->n_rec * 40 + 64));
    {
        KScope k(ctx, "k_rec_prep");
        launch_rec_prep(0, rec_input(b), b->op_off.as<uint64_t>(), b->ops.as<uint32_t>(), b->samples.as<Ctr>(), WinView{},
                        b->recs.as<RecInfo>(), b->pair_cnt.as<uint32_t>(), stats_view(b, b->n_rec), err, s);
    }
    volatile uint64_t* hs = reinterpret_cast<volatile uint64_t*>(ctx->h_scalars);
    Publisher(ctx).u64(0, sc + SC_ERR_TOK).u64(1, sc + SC_ERR_REC).u64(2, b->op_off.as<uint64_t>() + b->n_rec).u32(3, sc + SC_MISC).go(s);
    CU(cudaStreamSynchronize(s));
    b->busy = false;  // every upload of this batch has been consumed
    if ((uint32_t)hs[3] & 1u) {  // clips present: validate their placement like rust-htslib does
        launch_check_clips(b->ops.as<uint32_t>(), b->op_off.as<uint64_t>(), b->n_rec, err, s);
        Publisher(ctx).u64(0, sc + SC_ERR_TOK).u64(1, sc + SC_ERR_REC).go(s);
        CU(cudaStreamSynchronize(s));
    }
    flush_times(ctx);
    CU(cudaGetLastError());
    rc = map_err(ctx, b, hs[0], hs[1]);
    if (rc != RB_OK) return rc;
    b->sum.n_ops = hs[2];
    b->have_stats = true; b->stats_n = b->n_rec;
    if (summary) *summary = b->sum;
    return RB_OK;
}

// plan -> lift (or combine) -> line scan -> [host: output sizes] -> serialise; shared by liftover and break-paf
enum : int { TAIL_SEARCH = 0, TAIL_COMBINE = 1, TAIL_WHOLE = 2, TAIL_TRIM = 3 };  // who fills PairRes: k_lift, k_combine, k_whole_rows (rb invert), k_trim_rows (rb trim-paf)
static int lift_tail(rb_ctx* ctx, rb_batch* b, WinView win, int policy, int tail, uint32_t want, int with_stats, uint64_t P,
                     uint64_t n_ops, rb_summary* summary) {
    cudaStream_t s = ctx->stream;
    uint32_t* sc = ctx->scalars.as<uint32_t>();
    ErrSlots err{reinterpret_cast<unsigned long long*>(sc + SC_ERR_TOK), reinterpret_cast<unsigned long long*>(sc + SC_ERR_REC)};
    volatile uint64_t* hs = reinterpret_cast<volatile uint64_t*>(ctx->h_scalars);
    const uint32_t n = b->n_rec;
    int rc = RB_OK;
    CU(b->plans.ensure((P / LIFT_THREADS + 2) * sizeof(LiftPlan)));
    // Short rows (the usual tiling-window call): lift + line scan + serialiser in ONE kernel, k_emit.  Blocks of 128 pairs that
    // belong to one record and fit its staging area are lifted there, out of shared memory (PLAN_FAST); k_lift only sees the rest.
    const bool stats_text = b->stats_text && (tail == TAIL_SEARCH || tail == TAIL_COMBINE);  // (rows of ~130 bytes whatever the CIGARs are)
    const bool fused = ctx->fused_emit && (tail == TAIL_SEARCH || tail == TAIL_COMBINE) && P > 0 && (stats_text || b->n_bytes / P <= 1024);
    if (b->stats_text && !fused && P > 0) return fail(ctx, RB_ERR_UNSUPPORTED, "RB_WANT_STATS_TEXT needs the fused emit kernel (rb_liftover / rb_batch_liftover)");
    // wide windows (the rule k_samples uses for its sub-samples): no block of the call fits k_emit's staging area bar the odd short
    // record, so none is marked — k_lift<false> lifts everything and k_emit runs with the smaller shared-memory footprint
    const bool wide = P > 0 && n_ops > 64ull * P && !getenv("RB_NO_WIDE");
    const bool fast_lift = fused && tail == TAIL_SEARCH && policy == RB_POLICY_RIGHTMOST && !wide && !getenv("RB_NO_FAST_LIFT");
    if (tail == TAIL_SEARCH || tail == TAIL_COMBINE) {
        KScope k(ctx, "k_lift_plan");
        launch_lift_plan(P, b->pair_off.as<uint64_t>(), b->rec_order.as<uint32_t>(), n, b->recs.as<RecInfo>(), b->samples.as<Ctr>(), win,
                         b->plans.as<LiftPlan>(), s, fast_lift);
    }
    if (tail == TAIL_TRIM) {
        KScope k(ctx, "k_trim_rows");
        launch_trim_rows(n, b->recs.as<RecInfo>(), b->trim_views.as<TrimView>(), b->ops.as<uint32_t>(), b->samples.as<Ctr>(),
                         b->trim_has_drop ? b->trim_drop.as<uint8_t>() : nullptr, b->pair_res.as<PairRes>(), b->line_len.as<uint32_t>(),
                         b->pair_off.as<uint64_t>(), b->plans.as<LiftPlan>(), s);
    } else if (tail == TAIL_WHOLE) {
        KScope k(ctx, "k_whole_rows");
        launch_whole_rows(n, b->recs.as<RecInfo>(), b->pair_res.as<PairRes>(), b->line_len.as<uint32_t>(), b->pair_off.as<uint64_t>(),
                          b->plans.as<LiftPlan>(), s);
    } else if (tail == TAIL_COMBINE) {
        KScope k(ctx, "k_combine");
        launch_combine(P, b->pair_off.as<uint64_t>(), b->rec_order.as<uint32_t>(), n, b->recs.as<RecInfo>(), b->ops.as<uint32_t>(), win,
                       b->names_off.as<uint64_t>(), b->half_s.as<HalfS>(), b->half_e.as<HalfE>(), b->pair_res.as<PairRes>(),
                       b->line_len.as<uint32_t>(), err, s);
    } else {
        KScope k(ctx, "k_lift");
        launch_lift(P, b->pair_off.as<uint64_t>(), b->rec_order.as<uint32_t>(), n, b->recs.as<RecInfo>(), b->ops.as<uint32_t>(),
                    b->samples.as<Ctr>(), win, b->names_off.as<uint64_t>(), policy, b->plans.as<LiftPlan>(), b->pair_res.as<PairRes>(),
                    b->line_len.as<uint32_t>(), err, s, fast_lift, wide);
    }
    // Short rows (the usual tiling-window call): line scan + serialiser in ONE kernel, k_emit — no per-pair offsets in HBM, no
    // second pass over the results.  The sizes are known only afterwards, so the text buffer is sized from an estimate (or
    // kept from the call before); a buffer that turns out too small is grown to the exact size and the kernel runs again.
    if (fused) {
        const uint64_t nblk = (P + SER_LINES - 1) / SER_LINES;
        b->want = want;
        b->with_stats = with_stats != 0;
        b->row_stride = P;
        CU(b->blk_flags.ensure(nblk * 4 + 64));
        CU(b->emit_totals.ensure(64));
        CU(b->line_off.ensure((P + 1) * 8 + 64));
        CU(b->out_idx.ensure((P + 1) * 8 + 64));
        if (want & RB_WANT_TEXT) {
            const uint64_t est = stats_text ? P * 220 + 4096 : b->n_bytes + P * 160 + 4096;
            if (b->out_text.cap < est + 64) CU(b->out_text.ensure(est + 64));
            CU(b->out_line_off.ensure((P + 1) * 8 + 64));
        }
        if (want & RB_WANT_NUMERIC) CU(b->out_num.ensure(P * (6 * 8 + 2 * 4) + 64));
        if (with_stats) CU(b->out_stats.ensure(P * 40 + 64));
        unsigned long long* tot = b->emit_totals.as<unsigned long long>();
        uint64_t out_bytes = 0, n_out = 0, deferred = 0;
        unsigned long long* lb_bytes = b->ln_agg.as<unsigned long long>();  // one look-back word per block each
        unsigned long long* lb_rows = b->ln_pre.as<unsigned long long>();
        for (int attempt = 0;; attempt++) {
            CU(cudaMemsetAsync(tot, 0, 32, s));
            CU(cudaMemsetAsync(lb_bytes, 0, (nblk + 1) * 8, s));
            CU(cudaMemsetAsync(lb_rows, 0, (nblk + 1) * 8, s));
            {
                KScope k(ctx, "k_emit");
                launch_emit(P, b->pair_off.as<uint64_t>(), b->rec_order.as<uint32_t>(), n, b->recs.as<RecInfo>(), b->ops.as<uint32_t>(),
                            b->samples.as<Ctr>(), b->text_raw.as<uint8_t>() + TEXT_FRONT_PAD, win, b->names_off.as<uint64_t>(), b->names.as<uint8_t>(),
                            b->plans.as<LiftPlan>(), b->pair_res.as<PairRes>(), b->line_len.as<uint32_t>(), b->line_off.as<uint64_t>(),
                            b->out_idx.as<uint64_t>(), b->blk_flags.as<uint32_t>(),
                            (want & RB_WANT_TEXT) ? b->out_text.as<uint8_t>() : nullptr, (want & RB_WANT_TEXT) ? b->out_text.cap - 64 : 0,
                            (want & RB_WANT_TEXT) ? b->out_line_off.as<uint64_t>() : nullptr,
                            (want & RB_WANT_NUMERIC) ? num_view(b, P) : NumDev{}, with_stats ? stats_view(b, P) : StatsDev{}, b->byte_base,
                            b->rec_base, b->h_orig.empty() ? nullptr : b->orig_idx.as<uint32_t>(), lb_bytes, lb_rows, sc + SC_TICKET_LNS,
                            tot, err, s, stats_text, wide && !fast_lift);
            }
            Publisher(ctx).u64(0, sc + SC_ERR_TOK).u64(1, sc + SC_ERR_REC).u64(5, tot).u64(6, tot + 1).u64(7, tot + 2).u64(8, tot + 3).go(s);
            CU(cudaStreamSynchronize(s));
            rc = map_err(ctx, b, hs[0], hs[1]);
            if (rc != RB_OK) { flush_times(ctx); return rc; }
            out_bytes = hs[5]; n_out = hs[6]; deferred = hs[8];
            if (!hs[7]) break;
            if (attempt) return fail(ctx, RB_ERR_CUDA, "k_emit: the text does not fit a buffer of its own size");
            CU(b->out_text.ensure(out_bytes + 64));  // exact now
            CU(cudaMemsetAsync(sc + SC_TICKET_LNS, 0, 4, s));
        }
        if (deferred && stats_text) return fail(ctx, RB_ERR_UNSUPPORTED, "RB_WANT_STATS_TEXT: a row longer than 2 KB (names of ~1 KB?)");
        if (deferred && (want & RB_WANT_TEXT)) {  // blocks holding a line > 2 KB: warp-per-line path of the serialiser
            KScope k(ctx, "k_serialise");
            launch_serialise(P, b->pair_off.as<uint64_t>(), b->rec_order.as<uint32_t>(), n, b->recs.as<RecInfo>(), b->ops.as<uint32_t>(),
                             b->text_raw.as<uint8_t>() + TEXT_FRONT_PAD, win, b->names_off.as<uint64_t>(), b->names.as<uint8_t>(),
                             b->plans.as<LiftPlan>(), b->pair_res.as<PairRes>(), b->line_off.as<uint64_t>(), b->out_idx.as<uint64_t>(),
                             b->out_text.as<uint8_t>(), b->out_line_off.as<uint64_t>(),
                             (want & RB_WANT_NUMERIC) ? num_view(b, P) : NumDev{}, with_stats ? stats_view(b, P) : StatsDev{}, b->byte_base,
                             b->rec_base, b->h_orig.empty() ? nullptr : b->orig_idx.as<uint32_t>(), (uint32_t)SER_LINES, 0u, s,
                             b->blk_flags.as<uint32_t>());
        }
        CU(cudaGetLastError());
        if (ctx->profiling) { CU(cudaStreamSynchronize(s)); flush_times(ctx); }
        b->sum.n_ops = n_ops; b->sum.n_pairs = P; b->sum.n_out = n_out; b->sum.out_bytes = out_bytes;
        b->have_lift = true; b->stats_n = n_out;
        if (summary) *summary = b->sum;
        return RB_OK;
    }
    {
        KScope k(ctx, "k_scan_lines");
        launch_scan_lines(b->line_len.as<uint32_t>(), P, b->line_off.as<uint64_t>(), b->out_idx.as<uint64_t>(),
                          b->ln_state.as<uint32_t>(), b->ln_agg.as<ulonglong2>(), b->ln_pre.as<ulonglong2>(), sc + SC_TICKET_LNS, s);
    }
    Publisher(ctx).u64(0, sc + SC_ERR_TOK).u64(1, sc + SC_ERR_REC).u64(5, b->line_off.as<uint64_t>() + P).u64(6, b->out_idx.as<uint64_t>() + P).go(s);
    CU(cudaStreamSynchronize(s));
    rc = map_err(ctx, b, hs[0], hs[1]);
    if (rc != RB_OK) { flush_times(ctx); return rc; }
    const uint64_t out_bytes = hs[5], n_out = hs[6];

    b->want = want;
    b->row_stride = n_out;
    if (want & RB_WANT_TEXT) {
        CU(b->out_text.ensure(out_bytes + 64));
        CU(b->out_line_off.ensure((n_out + 1) * 8 + 64));
    }
    if (want & RB_WANT_NUMERIC) CU(b->out_num.ensure(n_out * (6 * 8 + 2 * 4) + 64));
    b->with_stats = with_stats != 0;
    if (with_stats) CU(b->out_stats.ensure(n_out * 40 + 64));
    // few, long rows (e.g. 100 kb windows: ~4 KB per row): 8 rows per block instead of 128, so the warp-per-line path
    // has enough blocks to fill the GPU
    // (whole-record rows of rb invert: 4 per block, a warp each)
    const uint32_t ser_group = (n_out && out_bytes / n_out > 1536 && P / SER_LINES < 4 * 148) ? (tail == TAIL_WHOLE ? 4u : 8u)
                                                                                               : (uint32_t)SER_LINES;
    // in that regime the long verbatim runs of input text inside the rows (whole-record rows, early rows, wide windows) are
    // copied by the whole grid (k_copy_mid) instead of one warp per row; blocks per row are capped so that a call with
    // many rows and no long run pays one empty block per row
    uint64_t max_rec_bytes = 0;
    // (whole-record-like rows — trim-paf, break-paf — or rows that are long on average; 100 kb windows over ~16 ops/kb make 4 KB
    // rows with hardly any run above the threshold, and the extra launch would cost them 2 %)
    const uint32_t defer_big = (ser_group != (uint32_t)SER_LINES && (want & RB_WANT_TEXT) && tail != TAIL_WHOLE && !b->invert &&
                                (tail == TAIL_TRIM || win.from_record || out_bytes / n_out >= MID_BIG)) ? 1u : 0u;
    if (defer_big)
        for (size_t i = 0; i + 1 < b->h_cigar_off.size(); i++) max_rec_bytes = std::max(max_rec_bytes, b->h_cigar_off[i + 1] - b->h_cigar_off[i]);
    {
        KScope k(ctx, "k_serialise");
        launch_serialise(P, b->pair_off.as<uint64_t>(), b->rec_order.as<uint32_t>(), n, b->recs.as<RecInfo>(), b->ops.as<uint32_t>(),
                         b->text_raw.as<uint8_t>() + TEXT_FRONT_PAD, win, b->names_off.as<uint64_t>(), b->names.as<uint8_t>(),
                         b->plans.as<LiftPlan>(), b->pair_res.as<PairRes>(),
                         b->line_off.as<uint64_t>(), b->out_idx.as<uint64_t>(), (want & RB_WANT_TEXT) ? b->out_text.as<uint8_t>() : nullptr,
                         (want & RB_WANT_TEXT) ? b->out_line_off.as<uint64_t>() : nullptr,
                         (want & RB_WANT_NUMERIC) ? num_view(b, n_out) : NumDev{}, with_stats ? stats_view(b, n_out) : StatsDev{},
                         b->byte_base, b->rec_base, b->h_orig.empty() ? nullptr : b->orig_idx.as<uint32_t>(), ser_group, defer_big, s);
    }
    if (defer_big) {
        KScope k(ctx, "k_copy_mid");
        launch_copy_mid(P, b->pair_off.as<uint64_t>(), b->rec_order.as<uint32_t>(), n, b->recs.as<RecInfo>(), b->pair_res.as<PairRes>(),
                        b->line_off.as<uint64_t>(), b->text_raw.as<uint8_t>() + TEXT_FRONT_PAD, b->out_text.as<uint8_t>(),
                        (uint32_t)std::min<uint64_t>((max_rec_bytes + 65535) / 65536, std::max<uint64_t>(1, 8192 / std::max<uint64_t>(P, 1))), s);
    }
    if (tail == TAIL_WHOLE && (want & RB_WANT_TEXT)) {
        KScope k(ctx, "k_whole_text");
        launch_whole_text(b->ops.as<uint32_t>(), b->op_off.as<uint64_t>(), n, b->recs.as<RecInfo>(), b->samples.as<Ctr>(),
                          b->line_off.as<uint64_t>(), b->out_text.as<uint8_t>(), b->ops_bound, s);
    }
    if (P == 0 && (want & RB_WANT_TEXT)) CU(cudaMemsetAsync(b->out_line_off.p, 0, 8, s));
    CU(cudaGetLastError());
    if (ctx->profiling) { CU(cudaStreamSynchronize(s)); flush_times(ctx); }
    b->sum.n_ops = n_ops; b->sum.n_pairs = P; b->sum.n_out = n_out; b->sum.out_bytes = out_bytes;
    b->have_lift = true; b->stats_n = n_out;
    if (summary) *summary = b->sum;
    return RB_OK;
}

int rb_batch_liftover(rb_ctx* ctx, rb_batch* b, int policy, uint32_t want, int with_stats, rb_summary* summary) {
    if (!ctx || !b) return RB_ERR_BAD_ARG;
    if (policy != RB_POLICY_RIGHTMOST && policy != RB_POLICY_EARLY_EXIT) return fail(ctx, RB_ERR_BAD_ARG, "unknown policy %d", policy);
    if ((want & RB_WANT_STATS_TEXT) && (want & RB_WANT_TEXT)) return fail(ctx, RB_ERR_BAD_ARG, "RB_WANT_STATS_TEXT and RB_WANT_TEXT exclude each other");
    b->stats_text = ctx->stats_text || (want & RB_WANT_STATS_TEXT);
    if (want & RB_WANT_STATS_TEXT) want = (want & ~RB_WANT_STATS_TEXT) | RB_WANT_TEXT;  // from here on the rows are "the text"
    cudaSetDevice(ctx->device);
    cudaStream_t s = ctx->stream;
    b->have_lift = false;
    int rc = run_tok(ctx, b);
    if (rc != RB_OK) return rc;
    uint32_t* sc = ctx->scalars.as<uint32_t>();
    ErrSlots err{reinterpret_cast<unsigned long long*>(sc + SC_ERR_TOK), reinterpret_cast<unsigned long long*>(sc + SC_ERR_REC)};
    WinView win = win_view(b);
    const rb_batch* wb = b->wsrc ? b->wsrc : b;  // holder of the window tables
    const uint32_t n = b->n_rec;
    {   // phase A: indel strip + window join (needs the ops only)
        KScope k(ctx, "k_rec_prep");
        launch_rec_prep(1, rec_input(b), b->op_off.as<uint64_t>(), b->ops.as<uint32_t>(), nullptr, win, b->recs.as<RecInfo>(),
                        b->pair_cnt.as<uint32_t>(), StatsDev{}, err, s);
    }
    if (wb->general && wb->n_win) {
        KScope k(ctx, "k_pair_count_bf");
        launch_pair_count_bf(b->recs.as<RecInfo>(), n, win, b->pair_cnt.as<uint32_t>(), s);
    }
    {
        KScope k(ctx, "k_pair_scan");
        launch_pair_scan(b->pair_cnt.as<uint32_t>(), b->rec_order.as<uint32_t>(), n, b->pair_off.as<uint64_t>(), s);
    }
    volatile uint64_t* hs = reinterpret_cast<volatile uint64_t*>(ctx->h_scalars);
    Publisher(ctx).u64(0, sc + SC_ERR_TOK).u64(1, sc + SC_ERR_REC).u64(2, b->op_off.as<uint64_t>() + n).u32(3, sc + SC_MISC)
        .u64(4, b->pair_off.as<uint64_t>() + n).go(s);
    CU(cudaStreamSynchronize(s));
    b->busy = false;  // every upload of this batch has been consumed
    if ((uint32_t)hs[3] & 1u) {
        launch_check_clips(b->ops.as<uint32_t>(), b->op_off.as<uint64_t>(), n, err, s);
        Publisher(ctx).u64(0, sc + SC_ERR_TOK).u64(1, sc + SC_ERR_REC).go(s);
        CU(cudaStreamSynchronize(s));
    }
    // CIGAR parse errors end the call here; strip panics wait for the integrity check of phase B so that the
    // error of the FIRST failing record is reported, whatever its kind
    rc = map_err(ctx, b, hs[0], UINT64_MAX);
    if (rc != RB_OK) { flush_times(ctx); return rc; }
    const uint64_t n_ops = hs[2], P = hs[4];
    // RB_LIFT_SEARCH (default): sampled scan, then one search per pair out of staged shared memory (k_lift).
    // RB_LIFT_STREAM (sorted BED + right-most policy only): the scan resolves the window boundaries itself
    // (k_scan_lift + k_combine) — no per-pair search at all, cost independent of the window count.
    const bool fused = ctx->lift_mode == RB_LIFT_STREAM && !wb->general && policy == RB_POLICY_RIGHTMOST && P > 0;

    CU(b->pair_res.ensure(P * sizeof(PairRes) + 64));
    CU(b->line_len.ensure(P * 4 + 64));
    CU(b->line_off.ensure((P + 1) * 8 + 64));
    CU(b->out_idx.ensure((P + 1) * 8 + 64));
    const size_t ln_blocks = P / (size_t)SER_LINES + 4;  // k_emit looks back over blocks of SER_LINES pairs (k_scan_lines needs fewer)
    CU(b->ln_state.ensure(ln_blocks * 4));
    CU(b->ln_agg.ensure(ln_blocks * 16));
    CU(b->ln_pre.ensure(ln_blocks * 16));
    CU(cudaMemsetAsync(b->ln_state.p, 0, ln_blocks * 4, s));
    if (fused) {
        CU(b->half_s.ensure(P * sizeof(HalfS) + 64));
        CU(b->half_e.ensure(P * sizeof(HalfE) + 64));
        LiftArgs la{b->recs.as<RecInfo>(), b->op_off.as<uint64_t>(), n, b->rec_rank.as<uint32_t>(), b->pair_off.as<uint64_t>(),
                    win.st, win.en, b->half_s.as<HalfS>(), b->half_e.as<HalfE>()};
        rc = run_scan(ctx, b, &la);
    } else {
        // wide windows (more than 64 ops per pair: one boundary per ~30 ops or fewer): the per-8-op sub-samples would serve a
        // few percent of the chunks and cost k_samples three quarters of its stores — absolute samples only, the boundary
        // walks of k_lift start at the chunk (<= 31 ops instead of <= 7).  RB_SUBS=1 / 0 in the environment forces either form.
        static const char* subs_env = getenv("RB_SUBS");
        const bool no_subs = subs_env ? subs_env[0] == '0' : (P > 0 && n_ops > 64ull * P);
        rc = run_scan(ctx, b, nullptr, no_subs);
    }
    if (rc != RB_OK) return rc;
    {   // phase B: integrity, RF_SLOW, counters of the stripped op range
        KScope k(ctx, "k_rec_prep");
        launch_rec_prep(2, rec_input(b), b->op_off.as<uint64_t>(), b->ops.as<uint32_t>(), b->samples.as<Ctr>(), win,
                        b->recs.as<RecInfo>(), b->pair_cnt.as<uint32_t>(), StatsDev{}, err, s);
    }
    if (wb->general && P) {
        CU(b->pair_win.ensure(P * 4 + 64));
        KScope k(ctx, "k_pair_fill_bf");
        launch_pair_fill_bf(b->recs.as<RecInfo>(), b->rec_rank.as<uint32_t>(), n, win, b->pair_off.as<uint64_t>(),
                            b->pair_win.as<uint32_t>(), s);
        win.pair_win = b->pair_win.as<uint32_t>();
    }
    return lift_tail(ctx, b, win, policy, fused ? TAIL_COMBINE : TAIL_SEARCH, want, with_stats, P, n_ops, summary);
}

// `rb break-paf` on a resident batch (uploaded WITHOUT windows): every record is cut at its insertions / deletions
// longer than max_size (liftover.rs:182-226); rows come out in FILE order, record by record (main.rs:271-281).
int rb_batch_break(rb_ctx* ctx, rb_batch* b, uint32_t max_size, int policy, uint32_t want, int with_stats, rb_summary* summary) {
    if (!ctx || !b) return RB_ERR_BAD_ARG;
    if (policy != RB_POLICY_RIGHTMOST && policy != RB_POLICY_EARLY_EXIT) return fail(ctx, RB_ERR_BAD_ARG, "unknown policy %d", policy);
    if (b->wsrc || b->n_win) return fail(ctx, RB_ERR_BAD_ARG, "rb_batch_break wants a batch uploaded without windows");
    if (want & RB_WANT_STATS_TEXT) return fail(ctx, RB_ERR_BAD_ARG, "RB_WANT_STATS_TEXT is an rb_liftover mode");
    b->stats_text = false;
    cudaSetDevice(ctx->device);
    cudaStream_t s = ctx->stream;
    b->have_lift = false;
    int rc = run_tok(ctx, b);
    if (rc != RB_OK) return rc;
    uint32_t* sc = ctx->scalars.as<uint32_t>();
    ErrSlots err{reinterpret_cast<unsigned long long*>(sc + SC_ERR_TOK), reinterpret_cast<unsigned long long*>(sc + SC_ERR_REC)};
    const uint32_t n = b->n_rec;
    {   // phase A without windows: the indel strip only
        KScope k(ctx, "k_rec_prep");
        launch_rec_prep(1, rec_input(b), b->op_off.as<uint64_t>(), b->ops.as<uint32_t>(), nullptr, WinView{}, b->recs.as<RecInfo>(),
                        b->pair_cnt.as<uint32_t>(), StatsDev{}, err, s);
    }
    rc = run_scan(ctx, b, nullptr);
    if (rc != RB_OK) return rc;
    {
        KScope k(ctx, "k_rec_prep");
        launch_rec_prep(2, rec_input(b), b->op_off.as<uint64_t>(), b->ops.as<uint32_t>(), b->samples.as<Ctr>(), WinView{},
                        b->recs.as<RecInfo>(), b->pair_cnt.as<uint32_t>(), StatsDev{}, err, s);
    }
    // count the break ops per 32-op chunk, scan
    const uint64_t n_chunks = b->ops_bound / SAMPLE + 1;
    CU(b->bp_cnt.ensure(n_chunks * 4 + 64));
    CU(b->bp_off.ensure((n_chunks + 1) * 8 + 64));
    CU(b->out_idx.ensure((n_chunks + 1) * 8 + 64));  // second output of the generic scan kernel (unused here)
    CU(cudaMemsetAsync(b->bp_cnt.p, 0, n_chunks * 4, s));
    const size_t ln_blocks0 = n_chunks / ((size_t)LNS_THREADS * 4) + 2;
    CU(b->ln_state.ensure(ln_blocks0 * 4)); CU(b->ln_agg.ensure(ln_blocks0 * 16)); CU(b->ln_pre.ensure(ln_blocks0 * 16));
    CU(cudaMemsetAsync(b->ln_state.p, 0, ln_blocks0 * 4, s));
    {
        KScope k(ctx, "k_break_scan");
        launch_break_scan(false, b->ops.as<uint32_t>(), b->op_off.as<uint64_t>() + n, b->ops_bound, b->heads.as<uint32_t>(),
                          b->samples.as<Ctr>(), b->op_off.as<uint64_t>(), n, b->recs.as<RecInfo>(), max_size, b->bp_cnt.as<uint32_t>(),
                          nullptr, nullptr, nullptr, nullptr, nullptr, s);
    }
    {
        KScope k(ctx, "k_scan_lines");
        launch_scan_lines(b->bp_cnt.as<uint32_t>(), n_chunks, b->bp_off.as<uint64_t>(), b->out_idx.as<uint64_t>(), b->ln_state.as<uint32_t>(),
                          b->ln_agg.as<ulonglong2>(), b->ln_pre.as<ulonglong2>(), sc + SC_TICKET_LNS, s);
    }
    volatile uint64_t* hs = reinterpret_cast<volatile uint64_t*>(ctx->h_scalars);
    Publisher(ctx).u64(0, sc + SC_ERR_TOK).u64(1, sc + SC_ERR_REC).u64(2, b->op_off.as<uint64_t>() + n).u32(3, sc + SC_MISC)
        .u64(4, b->bp_off.as<uint64_t>() + n_chunks).go(s);
    CU(cudaStreamSynchronize(s));
    b->busy = false;
    if ((uint32_t)hs[3] & 1u) {
        launch_check_clips(b->ops.as<uint32_t>(), b->op_off.as<uint64_t>(), n, err, s);
        Publisher(ctx).u64(0, sc + SC_ERR_TOK).u64(1, sc + SC_ERR_REC).go(s);
        CU(cudaStreamSynchronize(s));
    }
    rc = map_err(ctx, b, hs[0], hs[1]);  // parse, integrity and strip panics of ANY record end the call (the reference
    if (rc != RB_OK) { flush_times(ctx); return rc; }  // loads and strips every record before it prints the first row)
    const uint64_t n_ops = hs[2], total_bp = hs[4];
    const uint64_t P = total_bp + n;
    if (P > 0xFFFFFFFFull) return fail(ctx, RB_ERR_UNSUPPORTED, "more than 2^32 pieces");

    // fill pass -> per-record window ranges + the window table (in the batch's own window buffers)
    CU(b->bp_end.ensure(total_bp * 8 + 64)); CU(b->bp_next.ensure(total_bp * 8 + 64));
    CU(b->rec_bp.ensure((size_t)n * 16 + 64));
    CU(b->w_st.ensure(P * 8 + 64)); CU(b->w_en.ensure(P * 8 + 64));
    CU(cudaMemsetAsync(b->rec_bp.p, 0xFF, (size_t)n * 16, s));
    uint64_t* rec_bp0 = b->rec_bp.as<uint64_t>();
    uint64_t* rec_bp1 = rec_bp0 + n;
    {
        KScope k(ctx, "k_break_scan");
        launch_break_scan(true, b->ops.as<uint32_t>(), b->op_off.as<uint64_t>() + n, b->ops_bound, b->heads.as<uint32_t>(),
                          b->samples.as<Ctr>(), b->op_off.as<uint64_t>(), n, b->recs.as<RecInfo>(), max_size, b->bp_cnt.as<uint32_t>(),
                          b->bp_off.as<uint64_t>(), b->bp_end.as<uint64_t>(), b->bp_next.as<uint64_t>(), rec_bp0, rec_bp1, s);
    }
    {
        KScope k(ctx, "k_break_recs");
        launch_break_recs(n, b->recs.as<RecInfo>(), rec_bp0, rec_bp1, b->bp_end.as<uint64_t>(), b->bp_next.as<uint64_t>(),
                          b->w_st.as<uint64_t>(), b->w_en.as<uint64_t>(), b->pair_cnt.as<uint32_t>(), s);
    }
    {
        KScope k(ctx, "k_pair_scan");  // rec_order is the identity for this batch (file order)
        launch_pair_scan(b->pair_cnt.as<uint32_t>(), b->rec_order.as<uint32_t>(), n, b->pair_off.as<uint64_t>(), s);
    }
    WinView win{};
    win.st = b->w_st.as<uint64_t>(); win.en = b->w_en.as<uint64_t>(); win.en_pm = win.en;
    win.from_record = 1u;
    CU(b->pair_res.ensure(P * sizeof(PairRes) + 64));
    CU(b->line_len.ensure(P * 4 + 64));
    CU(b->line_off.ensure((P + 1) * 8 + 64));
    CU(b->out_idx.ensure((P + 1) * 8 + 64));
    const size_t ln_blocks = P / (size_t)SER_LINES + 4;  // k_emit looks back over blocks of SER_LINES pairs (k_scan_lines needs fewer)
    CU(b->ln_state.ensure(ln_blocks * 4)); CU(b->ln_agg.ensure(ln_blocks * 16)); CU(b->ln_pre.ensure(ln_blocks * 16));
    CU(cudaMemsetAsync(b->ln_state.p, 0, ln_blocks * 4, s));
    CU(cudaMemsetAsync(sc + SC_TICKET_LNS, 0, 4, s));  // the line scan reuses the ticket of the break-op scan
    return lift_tail(ctx, b, win, policy, TAIL_SEARCH, want, with_stats, P, n_ops, summary);
}

// `rb invert` on a batch uploaded by rb_invert (columns swapped, ctx->invert set): tokenise + invert the ops, counters and
// integrity of every record, then one whole-record row each
static int batch_invert(rb_ctx* ctx, rb_batch* b, uint32_t want, rb_summary* summary) {
    if (!ctx || !b) return RB_ERR_BAD_ARG;
    if (!b->invert) return fail(ctx, RB_ERR_BAD_ARG, "batch_invert wants a batch uploaded by rb_invert");
    if (b->wsrc || b->n_win) return fail(ctx, RB_ERR_BAD_ARG, "batch_invert wants a batch uploaded without windows");
    if (want & RB_WANT_STATS_TEXT) return fail(ctx, RB_ERR_BAD_ARG, "RB_WANT_STATS_TEXT is an rb_liftover mode");
    b->stats_text = false;
    cudaSetDevice(ctx->device);
    cudaStream_t s = ctx->stream;
    b->have_lift = false;
    int rc = run_tok(ctx, b);
    if (rc != RB_OK) return rc;
    rc = run_scan(ctx, b, nullptr);
    if (rc != RB_OK) return rc;
    uint32_t* sc = ctx->scalars.as<uint32_t>();
    ErrSlots err{reinterpret_cast<unsigned long long*>(sc + SC_ERR_TOK), reinterpret_cast<unsigned long long*>(sc + SC_ERR_REC)};
    const uint32_t n = b->n_rec;
    CU(b->out_stats.ensure((size_t)n * 40 + 64));
    {
        KScope k(ctx, "k_rec_prep");
        launch_rec_prep(0, rec_input(b), b->op_off.as<uint64_t>(), b->ops.as<uint32_t>(), b->samples.as<Ctr>(), WinView{},
                        b->recs.as<RecInfo>(), b->pair_cnt.as<uint32_t>(), stats_view(b, n), err, s);
    }
    volatile uint64_t* hs = reinterpret_cast<volatile uint64_t*>(ctx->h_scalars);
    Publisher(ctx).u64(0, sc + SC_ERR_TOK).u64(1, sc + SC_ERR_REC).u64(2, b->op_off.as<uint64_t>() + n).u32(3, sc + SC_MISC).go(s);
    CU(cudaStreamSynchronize(s));
    b->busy = false;
    if ((uint32_t)hs[3] & 1u) {
        launch_check_clips(b->ops.as<uint32_t>(), b->op_off.as<uint64_t>(), n, err, s);
        Publisher(ctx).u64(0, sc + SC_ERR_TOK).u64(1, sc + SC_ERR_REC).go(s);
        CU(cudaStreamSynchronize(s));
    }
    rc = map_err(ctx, b, hs[0], hs[1]);
    if (rc != RB_OK) { flush_times(ctx); return rc; }
    const uint64_t n_ops = hs[2], P = n;
    CU(b->pair_res.ensure(P * sizeof(PairRes) + 64));
    CU(b->line_len.ensure(P * 4 + 64));
    CU(b->line_off.ensure((P + 1) * 8 + 64));
    CU(b->out_idx.ensure((P + 1) * 8 + 64));
    CU(b->plans.ensure((P / LIFT_THREADS + 2) * sizeof(LiftPlan)));
    const size_t ln_blocks = P / (size_t)SER_LINES + 4;  // k_emit looks back over blocks of SER_LINES pairs (k_scan_lines needs fewer)
    CU(b->ln_state.ensure(ln_blocks * 4)); CU(b->ln_agg.ensure(ln_blocks * 16)); CU(b->ln_pre.ensure(ln_blocks * 16));
    CU(cudaMemsetAsync(b->ln_state.p, 0, ln_blocks * 4, s));
    WinView win{};
    win.from_record = 1u;  // a row's id is its record's (empty)
    return lift_tail(ctx, b, win, RB_POLICY_RIGHTMOST, TAIL_WHOLE, want, 0, P, n_ops, summary);
}

// the copies of a download have been enqueued on the context's stream (rc: unless that failed): wait for them
static int download_wait(rb_ctx* ctx, RowsOut& rows, int rc) {
    if (rc == RB_OK && cudaStreamSynchronize(ctx->stream) != cudaSuccess) {
        (void)cudaGetLastError();
        rc = fail(ctx, RB_ERR_CUDA, "cudaStreamSynchronize(ctx->stream) after the device -> host copies failed");
    }
    if (rc != RB_OK) rows.release();
    return rc;
}

int rb_batch_download_stats(rb_ctx* ctx, rb_batch* b, rb_stats_out* st) {
    if (!ctx || !b || !st) return RB_ERR_BAD_ARG;
    if (!b->have_stats) return fail(ctx, RB_ERR_BAD_ARG, "rb_batch_stats has not run on this batch");
    cudaSetDevice(ctx->device);
    memset(st, 0, sizeof *st);
    RowsOut rows;
    int rc = rows.reserve_stats(ctx, b->n_rec);
    if (rc == RB_OK) rc = rows.copy_rows(ctx, b, 0, b->n_rec, 0, 0, 0, 0, ctx->stream);
    rc = download_wait(ctx, rows, rc);
    if (rc == RB_OK) rows.finish(nullptr, st, b->n_rec, 0, 0);
    return rc;
}

int rb_batch_download_lift(rb_ctx* ctx, rb_batch* b, uint32_t want, rb_lift_out* out, rb_stats_out* st) {
    if (!ctx || !b || !out) return RB_ERR_BAD_ARG;
    if (!b->have_lift) return fail(ctx, RB_ERR_BAD_ARG, "rb_batch_liftover has not run on this batch");
    if (st && !b->with_stats) return fail(ctx, RB_ERR_BAD_ARG, "rb_batch_liftover ran without stats");
    if (want & RB_WANT_STATS_TEXT) {
        if (!b->stats_text) return fail(ctx, RB_ERR_BAD_ARG, "rb_batch_liftover did not run with RB_WANT_STATS_TEXT");
        want = (want & ~RB_WANT_STATS_TEXT) | RB_WANT_TEXT;
    }
    if (want & ~b->want) return fail(ctx, RB_ERR_BAD_ARG, "rb_batch_liftover did not materialise the requested outputs");
    cudaSetDevice(ctx->device);
    memset(out, 0, sizeof *out);
    const uint64_t n = b->sum.n_out, nb = b->sum.out_bytes;
    RowsOut rows;
    int rc = rows.reserve(ctx, n, nb, want, st != nullptr);
    if (rc == RB_OK) rc = rows.copy_rows(ctx, b, 0, n, 0, nb, 0, 0, ctx->stream);
    rc = download_wait(ctx, rows, rc);
    if (rc == RB_OK) rows.finish(out, st, n, nb, b->sum.n_pairs);
    return rc;
}

void rb_free_lift_out(rb_ctx*, rb_lift_out* out) {
    if (!out) return;
    if (out->_owner) reinterpret_cast<PinnedBlock*>(out->_owner)->in_use = false;
    memset(out, 0, sizeof *out);
}
void rb_free_stats_out(rb_ctx*, rb_stats_out* st) {
    if (!st) return;
    if (st->_owner) reinterpret_cast<PinnedBlock*>(st->_owner)->in_use = false;
    memset(st, 0, sizeof *st);
}

// ---- BGZF inflate (myio.rs:41-64: the `.bgz` reader) ----------------------------------------------
// One table row per block from a hop over the headers (RFC 1952 + the 'BC' extra field of the SAM spec, 4.1); false if
// `p` is not a well-formed series of BGZF blocks.  starts (nullable): where each row's block begins in `p`.
static bool bgzf_blocks(const uint8_t* p, uint64_t n, std::vector<BgzfBlock>& blocks, uint64_t& total, std::vector<uint64_t>* starts = nullptr) {
    uint64_t pos = 0;
    total = 0;
    while (pos < n) {
        if (n - pos < 18 || p[pos] != 0x1f || p[pos + 1] != 0x8b || p[pos + 2] != 8 || !(p[pos + 3] & 4)) return false;
        const uint64_t xlen = p[pos + 10] | ((uint64_t)p[pos + 11] << 8);
        uint64_t x = pos + 12, bsize = 0;
        const uint64_t xend = x + xlen;
        if (xend > n) return false;
        while (x + 4 <= xend) {
            const uint64_t slen = p[x + 2] | ((uint64_t)p[x + 3] << 8);
            if (p[x] == 'B' && p[x + 1] == 'C' && slen == 2 && x + 6 <= xend) bsize = (uint64_t)(p[x + 4] | (p[x + 5] << 8)) + 1;
            x += 4 + slen;
        }
        if (bsize == 0 || pos + bsize > n || bsize < xlen + 20) return false;
        auto le32 = [&](uint64_t at) { return (uint32_t)p[at] | ((uint32_t)p[at + 1] << 8) | ((uint32_t)p[at + 2] << 16) | ((uint32_t)p[at + 3] << 24); };
        BgzfBlock b{};
        b.cdata = xend; b.clen = (uint32_t)(bsize - xlen - 20); b.out_off = total;
        b.crc = le32(pos + bsize - 8); b.out_len = le32(pos + bsize - 4);
        if (b.out_len > 65536u) return false;  // (the format's bound; keeps a block's output offsets in 32 bits)
        if (b.out_len) {                       // (the empty end-of-file marker block has nothing to inflate)
            blocks.push_back(b);
            if (starts) starts->push_back(pos);
        }
        total += b.out_len;
        pos += bsize;
    }
    return true;
}
int rb_is_bgzf(const uint8_t* data, uint64_t nbytes) {
    return data && nbytes >= 18 && data[0] == 0x1f && data[1] == 0x8b && data[2] == 8 && (data[3] & 4) && data[12] == 'B' && data[13] == 'C';
}
// The inflate step: block table, compressed bytes -> HBM, k_inflate_bgzf, CRC-32 / ISIZE verdict.  On RB_OK `out` holds the
// `total` inflated bytes followed by `pad` bytes of head-room (the stream has been synchronised).  block_base: blocks of the file in
// front of `bgzf` (a share of a larger file), for the block numbers of the messages.
static int inflate_to_device(rb_ctx* ctx, const uint8_t* bgzf, uint64_t nbytes, DevBuf& out, uint64_t& total, size_t pad,
                             uint64_t block_base = 0) {
    std::vector<BgzfBlock> blocks;
    total = 0;
    if (!bgzf_blocks(bgzf, nbytes, blocks, total)) return fail(ctx, RB_ERR_BAD_ARG, "rb_inflate_bgzf: not a well-formed series of BGZF blocks");
    if (blocks.size() > 0xFFFFFFF0ull) return fail(ctx, RB_ERR_UNSUPPORTED, "rb_inflate_bgzf: more than 2^32 blocks");
    if (total == 0) return out.ensure(pad + 64) == cudaSuccess ? RB_OK : fail(ctx, RB_ERR_OOM, "rb_inflate_bgzf: device memory");
    cudaStream_t s = ctx->stream;
    DevBuf d_comp, d_blk, d_err;
    auto release = [&] { d_comp.release(); d_blk.release(); d_err.release(); };
    if (d_comp.ensure(nbytes + 64) != cudaSuccess || d_blk.ensure(blocks.size() * sizeof(BgzfBlock)) != cudaSuccess ||
        out.ensure(total + pad + 64) != cudaSuccess || d_err.ensure(8) != cudaSuccess) {
        (void)cudaGetLastError();
        release();
        return fail(ctx, RB_ERR_OOM, "rb_inflate_bgzf: device memory for %llu + %llu bytes", (unsigned long long)nbytes, (unsigned long long)total);
    }
    unsigned long long h_err = ~0ull;
    cudaError_t e = h2d_copy(d_comp.p, bgzf, nbytes, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_blk.p, blocks.data(), blocks.size() * sizeof(BgzfBlock), cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaMemsetAsync(d_err.p, 0xFF, 8, s);
    if (e == cudaSuccess) {
        KScope k(ctx, "k_inflate_bgzf");
        launch_inflate_bgzf(d_comp.as<uint8_t>(), d_blk.as<BgzfBlock>(), (uint32_t)blocks.size(), out.as<uint8_t>(), d_err.as<unsigned long long>(), s);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(&h_err, d_err.p, 8, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    flush_times(ctx);
    release();
    if (e != cudaSuccess) { (void)cudaGetLastError(); return fail(ctx, RB_ERR_CUDA, "rb_inflate_bgzf: %s", cudaGetErrorString(e)); }
    if (h_err != ~0ull)
        return fail(ctx, RB_ERR_BAD_ARG, "rb_inflate_bgzf: corrupt DEFLATE data in block %llu (code %u)", (unsigned long long)((h_err >> 8) + block_base), (unsigned)(h_err & 0xFF));
    return RB_OK;
}
int rb_inflate_bgzf(rb_ctx* ctx, const uint8_t* bgzf, uint64_t nbytes, uint8_t** text, uint64_t* text_nbytes) {
    if (!ctx) return RB_ERR_NO_DEVICE;
    if (!text || !text_nbytes || (!bgzf && nbytes)) return fail(ctx, RB_ERR_BAD_ARG, "rb_inflate_bgzf: null argument");
    *text = nullptr; *text_nbytes = 0;
    cudaSetDevice(ctx->device);
    DevBuf d_out;
    uint64_t total = 0;
    int rc = inflate_to_device(ctx, bgzf, nbytes, d_out, total, 0);
    PinnedBlock* blk = nullptr;
    if (rc == RB_OK) {
        blk = pinned_get(ctx, (size_t)total + 64);
        if (!blk) rc = fail(ctx, RB_ERR_OOM, "rb_inflate_bgzf: %llu bytes of pinned host memory", (unsigned long long)total);
    }
    if (rc == RB_OK && total) {
        cudaError_t e = cudaMemcpyAsync(blk->p, d_out.p, total, cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) {
            (void)cudaGetLastError();
            blk->in_use = false;
            rc = fail(ctx, RB_ERR_CUDA, "rb_inflate_bgzf: %s", cudaGetErrorString(e));
        }
    }
    d_out.release();
    if (rc != RB_OK) return rc;
    *text = static_cast<uint8_t*>(blk->p);
    *text_nbytes = total;
    return RB_OK;
}
void rb_free_text(rb_ctx* ctx, uint8_t* text) {
    if (!ctx || !text) return;
    for (PinnedBlock* b : ctx->pinned)
        if (b->p == text) b->in_use = false;
}

// ---- PAF text on the device (rb_batch_upload_paf; kernels in paf_parse_kernels.cu) -----------------------------------------
// text -> HBM (or BGZF -> inflated in HBM) -> line starts -> per-line fields -> scans -> the batch's columns and CIGAR text, byte
// for byte what upload_cigar + upload_columns build from the host reader's records.  The name bytes of the records come back and
// are interned here with the host reader's loop (name_intern.hpp); ids, names and the emission order go up again.  The text and
// every per-line table are freed before the call returns: the peak is about twice the text, during the call only.
struct DevScratch {  // device buffers of one call, released on every way out
    std::vector<DevBuf*> bufs;
    ~DevScratch() { for (DevBuf* d : bufs) d->release(); }
};

constexpr size_t TEXT_PAD = 4096;  // (16-byte loads of the last bytes)

// the call's input -> text in HBM (`who` names the call in the messages)
static int text_to_device(rb_ctx* ctx, const uint8_t* data, uint64_t nbytes, DevBuf& d_text, uint64_t& n, const char* who) {
    n = 0;
    if (rb_is_bgzf(data, nbytes)) return inflate_to_device(ctx, data, nbytes, d_text, n, TEXT_PAD);
    if (nbytes >= 2 && data[0] == 0x1f && data[1] == 0x8b) return fail(ctx, RB_ERR_BAD_ARG, "%s: a plain gzip stream (not BGZF); inflate it first", who);
    n = nbytes;
    CU(d_text.ensure(n + TEXT_PAD));
    if (n) CU(h2d_copy(d_text.p, data, n, ctx->stream));
    return RB_OK;
}

// What the device parse of one text leaves for the host steps: counts, the first panic, the records' name bytes, then their ids.
struct PafParsed {
    uint64_t text_bytes = 0, n_lines = 0, cg_bytes = 0, panic = ~0ull;  // panic: (0-based line << 8) | LS_* of the first one
    uint32_t n_rec = 0;
    std::vector<uint64_t> noff;   // record r's names: bytes [noff[r], noff[r + 1]) of `names`, the query name's qlen[r] first
    std::vector<uint32_t> qlen;
    std::vector<char> names;
    std::vector<uint32_t> ids;    // q ids, then t ids (paf_intern)
};

static int paf_panic(rb_ctx* ctx, uint64_t panic, uint64_t line_base) {
    const unsigned long long line = (panic >> 8) + 1 + line_base;
    switch ((uint32_t)(panic & 0xFF)) {
        case rbpp::LS_FEW_COLUMNS: return fail(ctx, RB_ERR_REF_PAF_PARSE, "line %llu: assertion failed: t.len() >= 12", line);
        case rbpp::LS_BAD_TAG: return fail(ctx, RB_ERR_REF_PAF_PARSE, "line %llu: assertion failed: PAF_TAG.is_match(token)", line);
        default: return fail(ctx, RB_ERR_REF_CIGAR_PARSE, "line %llu: Unable to parse cigar string.", line);
    }
}

// steps 1 - 3 of rb_batch_upload_paf on n bytes of text in HBM (16-byte aligned, TEXT_PAD bytes of head-room): lines, fields, scans,
// the batch's columns and CIGAR text, the name bytes to the host.  A panic is left in p.panic (nothing is packed then).
static int paf_parse_text(rb_ctx* ctx, rb_batch* b, const uint8_t* text, uint64_t n, PafParsed& p) {
    cudaStream_t s = ctx->stream;
    uint32_t* sc = ctx->scalars.as<uint32_t>();
    volatile uint64_t* hs = reinterpret_cast<volatile uint64_t*>(ctx->h_scalars);
    DevBuf d_chunk, d_tws, d_part, d_lines, d_cols, d_rec;
    DevScratch scratch{{&d_chunk, &d_tws, &d_part, &d_lines, &d_cols, &d_rec}};
    p.text_bytes = n;
    // 1. line starts: newline counts per 64 KiB, their scan, the starts; a last line without a terminator ends at n + 1 - 1
    uint64_t n_lines = 0;
    if (n) {
        const uint64_t nc = paf_chunks(n);
        CU(d_chunk.ensure((2 * nc + 2) * 8));
        CU(d_tws.ensure(paf_tiles(n) + 64));
        CU(d_part.ensure(paf_scan_parts(nc) * 8));
        uint64_t* cnt = d_chunk.as<uint64_t>();
        uint64_t* off = cnt + nc;
        CU(cudaMemsetAsync(sc + SC_MISC, 0, 4, s));
        {
            KScope k(ctx, "k_paf_lines_count");
            launch_paf_lines_count(text, n, cnt, d_tws.as<uint8_t>(), sc + SC_MISC, s);
        }
        {
            KScope k(ctx, "k_paf_scan");
            const uint64_t* in[1] = {cnt};
            uint64_t* out[1] = {off};
            launch_paf_scan(1, in, out, nc, d_part.as<uint64_t>(), s);
        }
        Publisher(ctx).u64(0, off + nc).u32(1, sc + SC_MISC).go(s);
        CU(cudaStreamSynchronize(s));
        n_lines = hs[0] + ((uint8_t)hs[1] != '\n' ? 1 : 0);
        if (n_lines > 0xFFFFFFFFull) return fail(ctx, RB_ERR_REF_PAF_PARSE, "more than 2^32 lines");
        CU(d_lines.ensure((n_lines + 2) * 8));
        {
            KScope k(ctx, "k_paf_lines_fill");
            launch_paf_lines_fill(text, n, off, d_lines.as<uint64_t>(), s);
        }
        if (n_lines > hs[0]) {
            const uint64_t end = n + 1;  // (pageable source: the copy is staged before the call returns)
            CU(cudaMemcpyAsync(d_lines.as<uint64_t>() + n_lines, &end, 8, cudaMemcpyHostToDevice, s));
        }
    }
    // 2. per-line fields, first panic, scans of (kept, cg bytes, name bytes)
    const uint64_t nl = n_lines;
    size_t o = 0;
    auto carve = [&](size_t bytes) { const size_t at = o; o += align_up(bytes, 256); return at; };
    const size_t o_state = carve(nl + 8), o_keep = carve(nl * 8), o_cgl = carve(nl * 8), o_nml = carve(nl * 8), o_v = carve(nl * 56),
                 o_strand = carve(nl + 8), o_qo = carve(nl * 8), o_to = carve(nl * 8), o_co = carve(nl * 8), o_ql = carve(nl * 4),
                 o_s0 = carve((nl + 1) * 8), o_s1 = carve((nl + 1) * 8), o_s2 = carve((nl + 1) * 8);
    CU(d_cols.ensure(o + 256));
    CU(d_part.ensure(3 * paf_scan_parts(nl) * 8));
    uint8_t* cb = d_cols.as<uint8_t>();
    PafLineCols L{};
    L.state = cb + o_state; L.keep = reinterpret_cast<uint64_t*>(cb + o_keep); L.cg_len = reinterpret_cast<uint64_t*>(cb + o_cgl);
    L.name_len = reinterpret_cast<uint64_t*>(cb + o_nml); L.v = reinterpret_cast<uint64_t*>(cb + o_v); L.strand = cb + o_strand;
    L.qn_off = reinterpret_cast<uint64_t*>(cb + o_qo); L.tn_off = reinterpret_cast<uint64_t*>(cb + o_to);
    L.cg_off = reinterpret_cast<uint64_t*>(cb + o_co); L.qn_len = reinterpret_cast<uint32_t*>(cb + o_ql);
    uint64_t* rec_idx = reinterpret_cast<uint64_t*>(cb + o_s0);
    uint64_t* cg_pos = reinterpret_cast<uint64_t*>(cb + o_s1);
    uint64_t* name_pos = reinterpret_cast<uint64_t*>(cb + o_s2);
    CU(cudaMemsetAsync(sc + SC_ERR_TOK, 0xFF, 8, s));
    {
        KScope k(ctx, "k_paf_fields");
        launch_paf_fields(text, d_lines.as<uint64_t>(), nl, d_tws.as<uint8_t>(), L, reinterpret_cast<unsigned long long*>(sc + SC_ERR_TOK), s);
    }
    {
        KScope k(ctx, "k_paf_scan");
        const uint64_t* in[3] = {L.keep, L.cg_len, L.name_len};
        uint64_t* out[3] = {rec_idx, cg_pos, name_pos};
        launch_paf_scan(3, in, out, nl, d_part.as<uint64_t>(), s);
    }
    Publisher(ctx).u64(0, sc + SC_ERR_TOK).u64(1, rec_idx + nl).u64(2, cg_pos + nl).u64(3, name_pos + nl).go(s);
    CU(cudaStreamSynchronize(s));
    CU(cudaGetLastError());
    const uint64_t n_rec64 = hs[1], cg_bytes = hs[2], name_bytes = hs[3];
    p.n_lines = nl;
    p.panic = hs[0];
    if (p.panic != ~0ull) { flush_times(ctx); return RB_OK; }
    const uint32_t n_rec = (uint32_t)n_rec64;
    p.n_rec = n_rec; p.cg_bytes = cg_bytes;
    // 3. the batch's columns and CIGAR text
    b->n_rec = n_rec;
    b->rec_base = 0; b->byte_base = 0;
    b->h_orig.clear();  // (a batch reused from rb_liftover may still map its rows to another call's records)
    b->invert = false;
    b->have_lift = b->have_stats = false;
    const size_t padded = text_layout(b, cg_bytes);
    CU(b->text_raw.ensure(TEXT_FRONT_PAD + padded));
    int rc = ensure_rec_buffers(ctx, b, n_rec);
    if (rc != RB_OK) return rc;
    const size_t r_line = 0, r_noff = align_up((size_t)n_rec * 4 + 8, 256), r_qlen = r_noff + align_up(((size_t)n_rec + 1) * 8, 256),
                 r_names = r_qlen + align_up((size_t)n_rec * 4 + 8, 256);
    CU(d_rec.ensure(r_names + name_bytes + 64));
    uint8_t* rb = d_rec.as<uint8_t>();
    {
        KScope k(ctx, "k_paf_pack");
        launch_paf_pack(text, nl, L, rec_idx, cg_pos, name_pos, n_rec, b->cols64.as<uint64_t>(), b->strand.as<uint8_t>(),
                        b->cigar_off.as<uint64_t>(), reinterpret_cast<uint32_t*>(rb + r_line), rb + r_names,
                        reinterpret_cast<uint64_t*>(rb + r_noff), reinterpret_cast<uint32_t*>(rb + r_qlen), s);
    }
    uint8_t* raw = b->text_raw.as<uint8_t>();
    CU(cudaMemsetAsync(raw, 0xFF, TEXT_FRONT_PAD, s));
    {
        KScope k(ctx, "k_paf_copy_cg");
        launch_paf_copy_cg(text, n_rec, b->cigar_off.as<uint64_t>(), reinterpret_cast<const uint32_t*>(rb + r_line), L.cg_off, cg_bytes,
                           raw + TEXT_FRONT_PAD, s);
    }
    const uint64_t tail0 = align_up(cg_bytes, 16);  // (k_paf_copy_cg wrote '0' up to here)
    CU(cudaMemsetAsync(raw + TEXT_FRONT_PAD + tail0, '0', padded - tail0, s));
    // 4. the names back to the host (interned by paf_intern)
    b->h_cigar_off.resize((size_t)n_rec + 1);
    p.noff.resize((size_t)n_rec + 1);
    p.qlen.resize(n_rec);
    p.names.resize(name_bytes + 1);
    CU(cudaMemcpyAsync(b->h_cigar_off.data(), b->cigar_off.p, ((size_t)n_rec + 1) * 8, cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpyAsync(p.noff.data(), rb + r_noff, ((size_t)n_rec + 1) * 8, cudaMemcpyDeviceToHost, s));
    if (n_rec) CU(cudaMemcpyAsync(p.qlen.data(), rb + r_qlen, (size_t)n_rec * 4, cudaMemcpyDeviceToHost, s));
    if (name_bytes) CU(cudaMemcpyAsync(p.names.data(), rb + r_names, name_bytes, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    flush_times(ctx);
    return RB_OK;
}

// ids by first appearance, with the host reader's loop; `index` / names / names_off carry the table from one call to the next, so
// the shares of one file interned in file order get the ids the whole file gets
static void paf_intern(PafParsed& p, std::unordered_map<std::string, uint32_t>& index, std::vector<uint8_t>& names,
                       std::vector<uint64_t>& names_off) {
    const uint32_t n_rec = p.n_rec;
    const char* nb = p.names.data();
    p.ids.resize((size_t)n_rec * 2);
    rbn::intern_record_names(
        n_rec, [&](size_t r) { return std::make_pair(nb + p.noff[r], (size_t)p.qlen[r]); },
        [&](size_t r) { return std::make_pair(nb + p.noff[r] + p.qlen[r], (size_t)(p.noff[r + 1] - p.noff[r] - p.qlen[r])); },
        [&](const char* q, size_t len) {
            const auto ins = index.emplace(std::string(q, len), (uint32_t)(names_off.size() - 1));
            if (ins.second) {
                names.insert(names.end(), q, q + len);
                names_off.push_back(names.size());
            }
            return ins.first->second;
        },
        p.ids.data(), p.ids.data() + n_rec);
}

// step 5: ids, the name table and the emission order up to the batch (asynchronous: b->busy)
static int paf_upload_names(rb_ctx* ctx, rb_batch* b, const PafParsed& p, const uint8_t* names, const uint64_t* names_off, uint32_t n_names,
                            const uint32_t* contig_rank) {
    cudaStream_t s = ctx->stream;
    const uint32_t n_rec = p.n_rec;
    const uint64_t tbl_bytes = names_off[n_names];
    b->n_names = n_names;
    CU(b->names_off.ensure(((size_t)n_names + 1) * 8));
    CU(b->names.ensure(tbl_bytes + 8));
    const size_t s_ids = 0, s_noff = align_up((size_t)n_rec * 8, 64), s_names = s_noff + align_up(((size_t)n_names + 1) * 8, 64),
                 s_order = s_names + align_up(tbl_bytes + 1, 64), s_rank = s_order + align_up((size_t)n_rec * 4, 64),
                 s_end = s_rank + align_up((size_t)n_rec * 4, 64);
    CU(b->stage.ensure(s_end));
    uint8_t* sp = b->stage.p;
    memcpy(sp + s_ids, p.ids.data(), (size_t)n_rec * 8);
    memcpy(sp + s_noff, names_off, ((size_t)n_names + 1) * 8);
    if (tbl_bytes) memcpy(sp + s_names, names, tbl_bytes);
    emission_ranks(p.ids.data() + n_rec, n_rec, n_names, b->file_order, contig_rank, reinterpret_cast<uint32_t*>(sp + s_order),
                   reinterpret_cast<uint32_t*>(sp + s_rank));
    if (n_rec) {
        CU(cudaMemcpyAsync(b->ids32.p, sp + s_ids, (size_t)n_rec * 8, cudaMemcpyHostToDevice, s));
        CU(cudaMemcpyAsync(b->rec_order.p, sp + s_order, (size_t)n_rec * 4, cudaMemcpyHostToDevice, s));
        CU(cudaMemcpyAsync(b->rec_rank.p, sp + s_rank, (size_t)n_rec * 4, cudaMemcpyHostToDevice, s));
    }
    CU(cudaMemcpyAsync(b->names_off.p, sp + s_noff, ((size_t)n_names + 1) * 8, cudaMemcpyHostToDevice, s));
    if (tbl_bytes) CU(cudaMemcpyAsync(b->names.p, sp + s_names, tbl_bytes, cudaMemcpyHostToDevice, s));
    b->busy = true;
    b->sum = rb_summary{};
    b->sum.cigar_bytes = b->n_bytes;
    return RB_OK;
}

static void paf_fill_info(rb_paf_info* info, uint64_t text_bytes, uint64_t n_lines, uint64_t n_rec, const std::vector<uint8_t>& names,
                          const std::vector<uint64_t>& names_off, uint64_t cg_bytes) {
    if (!info) return;
    info->text_bytes = text_bytes; info->n_lines = n_lines; info->skipped = n_lines - n_rec;
    info->n_rec = (uint32_t)n_rec; info->n_names = (uint32_t)(names_off.size() - 1);
    info->names = names.empty() ? nullptr : names.data();
    info->names_off = names_off.data();
    info->cigar_bytes = cg_bytes;
}

static int paf_upload_into(rb_ctx* ctx, rb_batch* b, const uint8_t* data, uint64_t nbytes, rb_paf_info* info) {
    DevBuf d_text;
    DevScratch scratch{{&d_text}};
    uint64_t n = 0;
    int rc = text_to_device(ctx, data, nbytes, d_text, n, "rb_batch_upload_paf");
    if (rc != RB_OK) return rc;
    PafParsed p;
    rc = paf_parse_text(ctx, b, d_text.as<uint8_t>(), n, p);
    d_text.release();  // (before the host work: the text is not needed any more)
    if (rc != RB_OK) return rc;
    if (p.panic != ~0ull) return paf_panic(ctx, p.panic, 0);
    std::unordered_map<std::string, uint32_t> index;
    b->h_names.clear();
    b->h_names_off.assign(1, 0);
    paf_intern(p, index, b->h_names, b->h_names_off);
    rc = paf_upload_names(ctx, b, p, b->h_names.data(), b->h_names_off.data(), (uint32_t)(b->h_names_off.size() - 1), nullptr);
    if (rc != RB_OK) return rc;
    paf_fill_info(info, n, p.n_lines, p.n_rec, b->h_names, b->h_names_off, p.cg_bytes);
    return RB_OK;
}

rb_batch* rb_batch_upload_paf(rb_ctx* ctx, const uint8_t* data, uint64_t nbytes, rb_paf_info* info, int* status) {
    auto set = [&](int s) { if (status) *status = s; };
    if (!ctx) { set(RB_ERR_NO_DEVICE); return nullptr; }
    if (!data && nbytes) { set(fail(ctx, RB_ERR_BAD_ARG, "rb_batch_upload_paf: null data")); return nullptr; }
    if (info) memset(info, 0, sizeof *info);
    cudaSetDevice(ctx->device);
    rb_batch* b = new rb_batch();
    int rc = paf_upload_into(ctx, b, data, nbytes, info);
    if (rc == RB_OK && cudaStreamSynchronize(ctx->stream) != cudaSuccess) {
        (void)cudaGetLastError();
        rc = fail(ctx, RB_ERR_CUDA, "upload failed");
    }
    if (rc != RB_OK) cudaStreamSynchronize(ctx->stream);
    b->busy = false;
    set(rc);
    if (rc != RB_OK) {
        if (info) memset(info, 0, sizeof *info);
        rb_batch_free(ctx, b);
        return nullptr;
    }
    return b;
}

int rb_batch_set_windows(rb_ctx* ctx, rb_batch* b, const rb_windows* wins) {
    if (!ctx || !b) return RB_ERR_BAD_ARG;
    if (b->wsrc) return fail(ctx, RB_ERR_BAD_ARG, "rb_batch_set_windows: not on a slice");
    cudaSetDevice(ctx->device);
    rb_records R{};
    R.n_names = b->n_names;
    b->have_lift = false;
    int rc = upload_windows_begin(ctx, b, &R, wins);
    if (rc == RB_OK) rc = upload_windows_end(ctx, b, &R, wins);
    if (cudaStreamSynchronize(ctx->stream) != cudaSuccess && rc == RB_OK) {  // the caller may reuse its tables after this call
        (void)cudaGetLastError();
        rc = fail(ctx, RB_ERR_CUDA, "window upload failed");
    }
    b->busy = false;
    if (rc != RB_OK) b->n_win = 0;
    return rc;
}

// ---- BED text on the device (rb_batch_set_windows_bed; kernels in bed_parse_kernels.cu) -------------------------------------
// text -> HBM (or BGZF -> inflated in HBM) -> line starts -> per-line fields -> first non-comment line's field count -> contig
// lookup in a hash table of the batch's resident name table -> scans (bed_row, window index, comments) -> kept rows in file
// order -> (only if they are not in (t_id, st) order already) a stable radix sort -> the batch's w_* tables, contig ranges ->
// k_win_check -> the general layout ((t_id, bed_row) order) when its verdict asks for it -> ids.  Only the rb_bed_info scalars
// come back to the host; the text and every per-line table are freed before the call returns.
static int bed_upload_into(rb_ctx* ctx, rb_batch* b, const uint8_t* data, uint64_t nbytes, rb_bed_info* info) {
    cudaStream_t s = ctx->stream;
    uint32_t* sc = ctx->scalars.as<uint32_t>();
    volatile uint64_t* hs = reinterpret_cast<volatile uint64_t*>(ctx->h_scalars);
    DevBuf d_text, d_chunk, d_part, d_lines, d_cols, d_tbl, d_rows, d_sort, d_ids;
    DevScratch scratch{{&d_text, &d_chunk, &d_part, &d_lines, &d_cols, &d_tbl, &d_rows, &d_sort, &d_ids}};
    b->n_win = 0;
    b->wsrc = nullptr;
    b->general = false; b->default_ids = true; b->win_pending = false;
    b->have_lift = false;
    uint64_t n = 0;
    {
        const int rc = text_to_device(ctx, data, nbytes, d_text, n, "rb_batch_set_windows_bed");
        if (rc != RB_OK) return rc;
    }
    const uint8_t* text = d_text.as<uint8_t>();
    // 1. line starts
    uint64_t nl = 0;
    if (n) {
        const uint64_t nc = paf_chunks(n);
        CU(d_chunk.ensure((2 * nc + 2) * 8));
        CU(d_part.ensure(paf_scan_parts(nc) * 8));
        uint64_t* cnt = d_chunk.as<uint64_t>();
        uint64_t* off = cnt + nc;
        {
            KScope k(ctx, "k_paf_lines_count");
            launch_bed_lines_count(text, n, cnt, s);
        }
        {
            KScope k(ctx, "k_paf_scan");
            const uint64_t* in[1] = {cnt};
            uint64_t* out[1] = {off};
            launch_paf_scan(1, in, out, nc, d_part.as<uint64_t>(), s);
        }
        Publisher(ctx).u64(0, off + nc).go(s);
        CU(cudaStreamSynchronize(s));
        nl = hs[0];
        CU(d_lines.ensure((nl + 1) * 8));
        {
            KScope k(ctx, "k_paf_lines_fill");
            launch_bed_lines_fill(text, n, off, d_lines.as<uint64_t>(), s);
        }
    }
    // 2. per-line fields, the field count, contig lookup, scans, rows in file order
    size_t o = 0;
    auto carve = [&](size_t bytes) { const size_t at = o; o += align_up(bytes, 256); return at; };
    const size_t o_nf = carve(nl * 8), o_st = carve(nl * 8), o_en = carve(nl * 8), o_nm = carve(nl * 8), o_io = carve(nl * 8),
                 o_il = carve(nl * 8), o_ok = carve(nl + 8), o_cm = carve(nl * 8), o_pa = carve(nl * 8), o_ke = carve(nl * 8),
                 o_tid = carve(nl * 4), o_s0 = carve((nl + 1) * 8), o_s1 = carve((nl + 1) * 8), o_s2 = carve((nl + 1) * 8), o_sc = carve(64);
    CU(d_cols.ensure(o + 256));
    CU(d_part.ensure(3 * paf_scan_parts(nl) * 8));
    uint8_t* cb = d_cols.as<uint8_t>();
    auto u64at = [&](size_t at) { return reinterpret_cast<uint64_t*>(cb + at); };
    BedLineCols L{};
    L.line_start = d_lines.as<uint64_t>();
    L.n_fields = u64at(o_nf); L.st = u64at(o_st); L.en = u64at(o_en); L.name_len = u64at(o_nm); L.id_off = u64at(o_io); L.id_len = u64at(o_il);
    L.nums_ok = cb + o_ok; L.comment = u64at(o_cm); L.parses = u64at(o_pa); L.kept = u64at(o_ke);
    L.tid = reinterpret_cast<uint32_t*>(cb + o_tid);
    uint64_t* row_idx = u64at(o_s0);
    uint64_t* win_idx = u64at(o_s1);
    uint64_t* cmt_idx = u64at(o_s2);
    unsigned long long* dsc = reinterpret_cast<unsigned long long*>(cb + o_sc);  // first row, nf0, max st, unsorted flag
    CU(cudaMemsetAsync(dsc, 0, 32, s));
    CU(cudaMemsetAsync(dsc, 0xFF, 8, s));
    const uint64_t slots = bed_name_slots(b->n_names);
    CU(d_tbl.ensure(slots * 4));
    CU(cudaMemsetAsync(d_tbl.p, 0, slots * 4, s));
    {
        KScope k(ctx, "k_bed_names");
        launch_bed_names(b->names.as<uint8_t>(), b->names_off.as<uint64_t>(), b->n_names, d_tbl.as<uint32_t>(), slots, s);
    }
    {
        KScope k(ctx, "k_bed_fields");
        launch_bed_fields(text, n, nl, L, dsc, s);
    }
    {
        KScope k(ctx, "k_bed_judge");
        launch_bed_judge(text, nl, L, dsc, b->names.as<uint8_t>(), b->names_off.as<uint64_t>(), d_tbl.as<uint32_t>(), slots, dsc + 1, s);
    }
    {
        KScope k(ctx, "k_paf_scan");
        const uint64_t* in[3] = {L.parses, L.kept, L.comment};
        uint64_t* out[3] = {row_idx, win_idx, cmt_idx};
        launch_paf_scan(3, in, out, nl, d_part.as<uint64_t>(), s);
    }
    Publisher(ctx).u64(0, row_idx + nl).u64(1, win_idx + nl).u64(2, cmt_idx + nl).u64(3, dsc + 1).go(s);
    CU(cudaStreamSynchronize(s));
    CU(cudaGetLastError());
    const uint64_t n_parsed = hs[0], n_kept = hs[1], n_comments = hs[2], nf0 = hs[3];
    if (n_parsed > 0xFFFFFFFFull) { flush_times(ctx); return fail(ctx, RB_ERR_UNSUPPORTED, "rb_batch_set_windows_bed: more than 2^32 - 1 BED rows"); }
    const uint32_t nw = (uint32_t)n_kept;
    const bool default_ids = nf0 <= 3;
    CU(d_rows.ensure((size_t)nw * 32 + 5 * 256));
    BedRows R{};
    {
        size_t ro = 0;
        auto rcarve = [&](size_t bytes) { const size_t at = ro; ro += align_up(bytes, 256); return d_rows.as<uint8_t>() + at; };
        R.tid = reinterpret_cast<uint32_t*>(rcarve((size_t)nw * 4)); R.row = reinterpret_cast<uint32_t*>(rcarve((size_t)nw * 4));
        R.st = reinterpret_cast<uint64_t*>(rcarve((size_t)nw * 8)); R.en = reinterpret_cast<uint64_t*>(rcarve((size_t)nw * 8));
        R.line = reinterpret_cast<uint64_t*>(rcarve((size_t)nw * 8));
    }
    {
        KScope k(ctx, "k_bed_compact");
        launch_bed_compact(nl, L, row_idx, win_idx, R, dsc + 2, s);
    }
    {
        KScope k(ctx, "k_bed_order");
        launch_bed_order(R, nw, reinterpret_cast<uint32_t*>(dsc + 3), s);
    }
    Publisher(ctx).u64(0, dsc + 2).u32(1, dsc + 3).go(s);
    CU(cudaStreamSynchronize(s));
    const uint64_t max_st = hs[0];
    const bool unsorted = (hs[1] & 1u) != 0;
    // 3. the (t_id, st) layout, contig ranges, the layout check
    CU(b->w_st.ensure((size_t)nw * 8 + 8)); CU(b->w_en.ensure((size_t)nw * 8 + 8)); CU(b->w_bed_row.ensure((size_t)nw * 4 + 8));
    CU(b->w_tid.ensure((size_t)nw * 4 + 8));
    CU(b->cont_lo.ensure(((size_t)b->n_names + 1) * 4)); CU(b->cont_hi.ensure(((size_t)b->n_names + 1) * 4));
    auto bits = [](uint64_t v) { int k = 0; while (v) { k++; v >>= 1; } return k; };
    const int tb = bits(b->n_names ? b->n_names - 1 : 0), sb = bits(max_st);
    const size_t sort_bytes = bed_sort_scratch(nw);
    uint32_t* perm = nullptr;
    if (nw && unsorted) {
        CU(d_sort.ensure(sort_bytes + (size_t)nw * 4 + 256));
        perm = reinterpret_cast<uint32_t*>(d_sort.as<uint8_t>() + align_up(sort_bytes, 256));
        KScope k(ctx, "k_bed_sort");
        CU(launch_bed_sort(R, nw, tb, sb, false, d_sort.p, sort_bytes, perm, s));
    }
    uint64_t* id_span = nullptr;  // id offset / length per row in the final layout, then their scan input
    if (!default_ids) {
        CU(d_ids.ensure((size_t)nw * 16 + 512));
        id_span = d_ids.as<uint64_t>();
    }
    {
        KScope k(ctx, "k_bed_gather");
        launch_bed_gather(R, nw, perm, L.id_off, L.id_len, b->w_tid.as<uint32_t>(), b->w_st.as<uint64_t>(), b->w_en.as<uint64_t>(),
                          b->w_bed_row.as<uint32_t>(), id_span, id_span ? id_span + nw + 32 : nullptr, s);
    }
    CU(cudaMemsetAsync(b->cont_lo.p, 0, ((size_t)b->n_names + 1) * 4, s));
    CU(cudaMemsetAsync(b->cont_hi.p, 0, ((size_t)b->n_names + 1) * 4, s));
    {
        KScope k(ctx, "k_bed_cont");
        launch_bed_cont(b->w_tid.as<uint32_t>(), nw, b->cont_lo.as<uint32_t>(), b->cont_hi.as<uint32_t>(), s);
    }
    b->n_win = nw;
    b->default_ids = default_ids;
    rb_records Rn{};
    Rn.n_names = b->n_names;
    int rc = windows_check(ctx, b, &Rn, s);
    if (rc != RB_OK) return rc;
    b->win_pending = false;
    if (nw) {
        CU(cudaEventSynchronize(ctx->ev_win));
        b->general = (((uint32_t)hs[16]) & 2u) != 0;
    }
    if (b->general) {  // file order grouped by contig = (t_id, bed_row) order: R is in file order, so a stable sort by t_id
        CU(d_sort.ensure(sort_bytes + (size_t)nw * 4 + 256));
        perm = reinterpret_cast<uint32_t*>(d_sort.as<uint8_t>() + align_up(sort_bytes, 256));
        {
            KScope k(ctx, "k_bed_sort");
            CU(launch_bed_sort(R, nw, tb, sb, true, d_sort.p, sort_bytes, perm, s));
        }
        KScope k(ctx, "k_bed_gather");
        launch_bed_gather(R, nw, perm, L.id_off, L.id_len, b->w_tid.as<uint32_t>(), b->w_st.as<uint64_t>(), b->w_en.as<uint64_t>(),
                          b->w_bed_row.as<uint32_t>(), id_span, id_span ? id_span + nw + 32 : nullptr, s);
    }
    // 4. ids: offsets = scan of the lengths in the final layout, then the bytes
    uint64_t ids_bytes = 0;
    if (!default_ids) {
        CU(b->w_ids_off.ensure(((size_t)nw + 1) * 8));
        CU(d_part.ensure(paf_scan_parts(nw) * 8));
        {
            KScope k(ctx, "k_paf_scan");
            const uint64_t* in[1] = {id_span + nw + 32};
            uint64_t* out[1] = {b->w_ids_off.as<uint64_t>()};
            launch_paf_scan(1, in, out, nw, d_part.as<uint64_t>(), s);
        }
        Publisher(ctx).u64(0, b->w_ids_off.as<uint64_t>() + nw).go(s);
        CU(cudaStreamSynchronize(s));
        ids_bytes = hs[0];
        CU(b->w_ids.ensure(align_up(ids_bytes, 16) + 64));
        KScope k(ctx, "k_paf_copy_cg");
        launch_paf_copy_cg(text, nw, b->w_ids_off.as<uint64_t>(), nullptr, id_span, ids_bytes, b->w_ids.as<uint8_t>(), s);
    }
    CU(cudaStreamSynchronize(s));
    CU(cudaGetLastError());
    flush_times(ctx);
    if (info) {
        info->text_bytes = n; info->n_lines = nl; info->n_comments = n_comments; info->n_parsed = n_parsed;
        info->n_win = nw; info->n_fields = (uint32_t)std::min<uint64_t>(nf0, 0xFFFFFFFFull);
        info->default_ids = default_ids ? 1 : 0; info->general = b->general ? 1 : 0;
    }
    return RB_OK;
}

int rb_batch_set_windows_bed(rb_ctx* ctx, rb_batch* b, const uint8_t* data, uint64_t nbytes, rb_bed_info* info) {
    if (!ctx || !b) return RB_ERR_BAD_ARG;
    if (info) memset(info, 0, sizeof *info);
    if (!data && nbytes) return fail(ctx, RB_ERR_BAD_ARG, "rb_batch_set_windows_bed: null data");
    if (b->wsrc) return fail(ctx, RB_ERR_BAD_ARG, "rb_batch_set_windows_bed: not on a slice");
    cudaSetDevice(ctx->device);
    if (b->busy) { CU(cudaStreamSynchronize(ctx->stream)); b->busy = false; }
    int rc = bed_upload_into(ctx, b, data, nbytes, info);
    if (cudaStreamSynchronize(ctx->stream) != cudaSuccess && rc == RB_OK) {
        (void)cudaGetLastError();
        rc = fail(ctx, RB_ERR_CUDA, "BED parse failed");
    }
    if (rc != RB_OK) {
        flush_times(ctx);
        b->n_win = 0; b->general = false; b->win_pending = false;
        if (info) memset(info, 0, sizeof *info);
    }
    return rc;
}

int rb_batch_windows(rb_ctx* ctx, rb_batch* b, rb_windows* out) {
    if (!ctx || !b || !out) return RB_ERR_BAD_ARG;
    if (b->wsrc) return fail(ctx, RB_ERR_BAD_ARG, "rb_batch_windows: not on a slice");
    cudaSetDevice(ctx->device);
    cudaStream_t s = ctx->stream;
    memset(out, 0, sizeof *out);
    if (b->busy) { CU(cudaStreamSynchronize(s)); b->busy = false; }
    const size_t nw = b->n_win;
    uint64_t ids_bytes = 0;
    if (!b->default_ids && nw) {
        CU(cudaMemcpyAsync(&ids_bytes, b->w_ids_off.as<uint64_t>() + nw, 8, cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
    }
    // device copy at [0, o_end), the (t_id, st) layout of a general table after it
    const size_t o_tid = 0, o_st = align_up(nw * 4 + 1, 64), o_en = o_st + align_up(nw * 8 + 1, 64), o_row = o_en + align_up(nw * 8 + 1, 64),
                 o_off = o_row + align_up(nw * 4 + 1, 64), o_ids = o_off + align_up((nw + 1) * 8, 64), o_end = o_ids + align_up(ids_bytes + 1, 64);
    CU(b->win_out.ensure(b->general ? 2 * o_end : o_end));
    uint8_t* p = b->win_out.p;
    uint64_t* off = reinterpret_cast<uint64_t*>(p + o_off);
    off[0] = 0;
    if (nw) {
        CU(cudaMemcpyAsync(p + o_tid, b->w_tid.p, nw * 4, cudaMemcpyDeviceToHost, s));
        CU(cudaMemcpyAsync(p + o_st, b->w_st.p, nw * 8, cudaMemcpyDeviceToHost, s));
        CU(cudaMemcpyAsync(p + o_en, b->w_en.p, nw * 8, cudaMemcpyDeviceToHost, s));
        CU(cudaMemcpyAsync(p + o_row, b->w_bed_row.p, nw * 4, cudaMemcpyDeviceToHost, s));
        if (!b->default_ids) {
            CU(cudaMemcpyAsync(off, b->w_ids_off.p, (nw + 1) * 8, cudaMemcpyDeviceToHost, s));
            if (ids_bytes) CU(cudaMemcpyAsync(p + o_ids, b->w_ids.p, ids_bytes, cudaMemcpyDeviceToHost, s));
        }
        CU(cudaStreamSynchronize(s));
    }
    if (b->general && nw) {  // stored in (t_id, bed_row) order: a stable sort by (t_id, st) gives the rb_windows table back
        const uint32_t* tid = reinterpret_cast<const uint32_t*>(p + o_tid);
        const uint64_t* st = reinterpret_cast<const uint64_t*>(p + o_st);
        std::vector<uint32_t> perm(nw);
        for (size_t i = 0; i < nw; i++) perm[i] = (uint32_t)i;
        std::stable_sort(perm.begin(), perm.end(), [&](uint32_t a, uint32_t c) { return tid[a] != tid[c] ? tid[a] < tid[c] : st[a] < st[c]; });
        uint8_t* q = p + o_end;
        uint64_t* qoff = reinterpret_cast<uint64_t*>(q + o_off);
        qoff[0] = 0;
        for (size_t i = 0; i < nw; i++) {
            const uint32_t j = perm[i];
            reinterpret_cast<uint32_t*>(q + o_tid)[i] = tid[j];
            reinterpret_cast<uint64_t*>(q + o_st)[i] = st[j];
            reinterpret_cast<uint64_t*>(q + o_en)[i] = reinterpret_cast<const uint64_t*>(p + o_en)[j];
            reinterpret_cast<uint32_t*>(q + o_row)[i] = reinterpret_cast<const uint32_t*>(p + o_row)[j];
            if (!b->default_ids) {
                const uint64_t len = off[j + 1] - off[j];
                memcpy(q + o_ids + qoff[i], p + o_ids + off[j], len);
                qoff[i + 1] = qoff[i] + len;
            }
        }
        p = q;
    }
    out->n_win = (uint32_t)nw;
    out->t_id = reinterpret_cast<const uint32_t*>(p + o_tid);
    out->st = reinterpret_cast<const uint64_t*>(p + o_st);
    out->en = reinterpret_cast<const uint64_t*>(p + o_en);
    out->bed_row = reinterpret_cast<const uint32_t*>(p + o_row);
    out->ids = b->default_ids ? nullptr : p + o_ids;
    out->ids_off = b->default_ids ? nullptr : reinterpret_cast<const uint64_t*>(p + o_off);
    return RB_OK;
}

int rb_batch_records(rb_ctx* ctx, rb_batch* b, int with_cigar, rb_records* out) {
    if (!ctx || !b || !out) return RB_ERR_BAD_ARG;
    cudaSetDevice(ctx->device);
    cudaStream_t s = ctx->stream;
    memset(out, 0, sizeof *out);
    const size_t n = b->n_rec, nn = b->n_names;
    uint64_t names_bytes = 0;
    CU(cudaMemcpyAsync(&names_bytes, b->names_off.as<uint64_t>() + nn, 8, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    const uint64_t cg = with_cigar ? b->n_bytes : 0;
    const size_t o_off = 0, o_cols = align_up((n + 1) * 8, 64), o_ids = o_cols + align_up(n * 56, 64), o_strand = o_ids + align_up(n * 8, 64),
                 o_noff = o_strand + align_up(n + 1, 64), o_names = o_noff + align_up((nn + 1) * 8, 64),
                 o_cigar = o_names + align_up(names_bytes + 1, 64), o_end = o_cigar + align_up(cg + 1, 64);
    if (b->busy) { CU(cudaStreamSynchronize(s)); b->busy = false; }  // (the staging area may still feed an upload)
    CU(b->rec_out.ensure(o_end));
    uint8_t* p = b->rec_out.p;
    CU(cudaMemcpyAsync(p + o_off, b->cigar_off.p, (n + 1) * 8, cudaMemcpyDeviceToHost, s));
    if (n) {
        CU(cudaMemcpyAsync(p + o_cols, b->cols64.p, n * 56, cudaMemcpyDeviceToHost, s));
        CU(cudaMemcpyAsync(p + o_ids, b->ids32.p, n * 8, cudaMemcpyDeviceToHost, s));
        CU(cudaMemcpyAsync(p + o_strand, b->strand.p, n, cudaMemcpyDeviceToHost, s));
    }
    CU(cudaMemcpyAsync(p + o_noff, b->names_off.p, (nn + 1) * 8, cudaMemcpyDeviceToHost, s));
    if (names_bytes) CU(cudaMemcpyAsync(p + o_names, b->names.p, names_bytes, cudaMemcpyDeviceToHost, s));
    if (cg) CU(cudaMemcpyAsync(p + o_cigar, b->text_raw.as<uint8_t>() + TEXT_FRONT_PAD, cg, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    const uint64_t* cols = reinterpret_cast<const uint64_t*>(p + o_cols);
    out->n_rec = (uint32_t)n;
    out->cigar = with_cigar ? p + o_cigar : nullptr;
    out->cigar_nbytes = cg;
    out->cigar_off = reinterpret_cast<const uint64_t*>(p + o_off);
    out->q_len = cols; out->q_st = cols + n; out->q_en = cols + 2 * n; out->t_len = cols + 3 * n; out->t_st = cols + 4 * n;
    out->t_en = cols + 5 * n; out->mapq = cols + 6 * n;
    out->strand = p + o_strand;
    out->q_id = reinterpret_cast<const uint32_t*>(p + o_ids); out->t_id = out->q_id + n;
    out->names = p + o_names; out->names_off = reinterpret_cast<const uint64_t*>(p + o_noff); out->n_names = (uint32_t)nn;
    return RB_OK;
}

// ---- rb_liftover in slices -----------------------------------------------------------------------
// A call is cut into K runs of records that are consecutive in EMISSION order, of about equal CIGAR size (when the PAF
// is grouped by target these are plain runs of the caller's arrays; otherwise each slice is gathered run by run).  Each slice goes upload -> kernels -> download on its own
// ping-pong work area, and the download of slice k (copy stream, device->host DMA engine) runs under the upload and
// the kernels of slices k+1, k+2 (compute stream, host->device engine): PCIe is used in both directions at once and
// the call approaches the time of its largest transfer instead of the sum of all three stages.  It also bounds the
// HBM footprint of the intermediates by the slice size.  The rows land in one pinned block in emission order; the
// window tables are uploaded once and shared by all slices.
// Emission order of the records (liftover.rs:151-164): contigs by first appearance of t_name, file order inside.
// Returns false for name ids out of range (reported properly by the unsliced path); `identity` = file order already.
static bool emission_order(const rb_records* R, std::vector<uint32_t>& ord, bool& identity) {
    const uint32_t n = R->n_rec;
    for (uint32_t i = 0; i < n; i++)
        if (R->t_id[i] >= R->n_names) return false;
    std::vector<uint32_t> rank(n);
    ord.resize(n);
    emission_ranks(R->t_id, n, R->n_names, false, nullptr, ord.data(), rank.data());
    identity = true;
    for (uint32_t i = 0; i < n && identity; i++) identity = ord[i] == i;
    return true;
}

static int liftover_unsliced(rb_ctx* ctx, const rb_records* recs, const rb_windows* wins, int policy, uint32_t want, rb_lift_out* out,
                             rb_stats_out* stats) {
    rb_batch* b = ctx->scratch;
    int rc = upload_into(ctx, b, recs, wins);
    if (rc != RB_OK) return rc;
    rc = rb_batch_liftover(ctx, b, policy, want, stats != nullptr, nullptr);
    if (rc != RB_OK) return rc;
    return rb_batch_download_lift(ctx, b, want, out, stats);
}

// ---- rb_liftover / rb_stats on a multi-device context -----------------------------------------------
// The records are cut into one contiguous run of the EMISSION order per device (liftover.rs:151-164: contigs by first
// appearance, file order inside), balanced on CIGAR bytes; a cut snaps to the nearest contig boundary when that costs less
// than 5 % of a device's share.  Every device (one host thread each) uploads its records and the window rows of its
// contigs, runs the whole kernel sequence and reports its row / byte counts; the prefix over the devices says where each
// device's rows go in the ONE pinned output block, and every device copies its rows there itself (line offsets rebased
// on the device).  Nothing is exchanged between the GPUs: a (window, record) pair needs that record and that window only.
extern "C++" {
namespace {
struct Rendezvous {  // all device threads meet; the last one to arrive runs `fn` before anybody leaves
    std::mutex m;
    std::condition_variable cv;
    int n, count = 0, gen = 0;
    explicit Rendezvous(int n_) : n(n_) {}
    template <class F> void meet(F&& fn) {
        std::unique_lock<std::mutex> lk(m);
        const int g = gen;
        if (++count == n) { fn(); count = 0; gen++; cv.notify_all(); }
        else cv.wait(lk, [&] { return g != gen; });
    }
};

// cut[d] .. cut[d+1]: positions in `ord` of device d's records
bool partition_by_bytes(const rb_records* R, const std::vector<uint32_t>& ord, int D, std::vector<uint32_t>& cut) {
    const uint32_t n = (uint32_t)ord.size();
    std::vector<uint64_t> pre(n + 1, 0);
    for (uint32_t i = 0; i < n; i++) {
        const uint32_t r = ord[i];
        if (R->cigar_off[r + 1] < R->cigar_off[r]) return false;
        pre[i + 1] = pre[i] + (R->cigar_off[r + 1] - R->cigar_off[r]) + 64;  // (+64: records without a CIGAR still cost something)
    }
    const uint64_t total = pre[n], share = total / (uint64_t)D, slack = share / 20;
    cut.assign(1, 0);
    for (int d = 1; d < D; d++) {
        const uint64_t target = total * (uint64_t)d / (uint64_t)D;
        uint32_t i = (uint32_t)(std::lower_bound(pre.begin(), pre.end(), target) - pre.begin());
        if (i > n) i = n;
        // nearest contig boundary on either side, if it keeps the share within 5 %
        uint32_t lo = i, hi = i;
        while (lo > cut.back() && lo < n && R->t_id[ord[lo]] == R->t_id[ord[lo - 1]] && target - pre[lo] < slack) lo--;
        while (hi < n && hi > 0 && R->t_id[ord[hi]] == R->t_id[ord[hi - 1]] && pre[hi] - target < slack) hi++;
        const bool lo_ok = lo > cut.back() && lo < n && R->t_id[ord[lo]] != R->t_id[ord[lo - 1]] && target - pre[lo] <= slack;
        const bool hi_ok = hi < n && hi > 0 && R->t_id[ord[hi]] != R->t_id[ord[hi - 1]] && pre[hi] - target <= slack;
        if (lo_ok && (!hi_ok || target - pre[lo] <= pre[hi] - target)) i = lo;
        else if (hi_ok) i = hi;
        if (i <= cut.back() || i >= n) return false;  // a device would get nothing: not worth spreading
        cut.push_back(i);
    }
    cut.push_back(n);
    return true;
}

// The devices of a context (device 0: the context itself, then its peers) and the status of each in the call in progress.
struct Devices {
    rb_ctx* ctx;
    int n;
    std::vector<int> rc;
    explicit Devices(rb_ctx* c) : ctx(c), n(1 + (int)c->peers.size()), rc((size_t)n, RB_OK) {}
    rb_ctx* at(int d) const { return d ? ctx->peers[(size_t)d - 1] : ctx; }

    // fn(d, c) on every device, devices 1 .. n-1 on threads of their own and device 0 on the caller's.  Before it, each device
    // clears its error, gets its scratch batch and waits for a batch of an earlier call still in flight; rc[d] says whether that
    // worked (fn runs either way, so that it reaches every rendezvous of the call).
    template <class F> void run(F&& fn) {
        auto one = [&](int d) {
            rb_ctx* c = at(d);
            cudaSetDevice(c->device);
            c->err.clear(); c->err_rec = UINT64_MAX;
            if (!c->scratch) c->scratch = new rb_batch();
            rc[(size_t)d] = [c] {
                rb_ctx* ctx = c;  // (CU reports into this device's context)
                if (c->scratch->busy) { CU(cudaStreamSynchronize(c->stream)); c->scratch->busy = false; }
                return (int)RB_OK;
            }();
            fn(d, c);
        };
        std::vector<std::thread> pool;
        for (int d = 1; d < n; d++) pool.emplace_back(one, d);
        one(0);
        for (auto& th : pool) th.join();
        cudaSetDevice(ctx->device);
    }

    // the status that fails the call: the first failing device in device order, or (by_record: errors of the lift) the one that
    // reports the smallest record index.  ctx->err takes that device's message.
    int error(bool by_record) const {
        int k = -1;
        for (int d = 0; d < n; d++)
            if (rc[(size_t)d] != RB_OK && (k < 0 || (by_record && at(d)->err_rec < at(k)->err_rec))) k = d;
        if (k < 0) return RB_OK;
        if (k) ctx->err = at(k)->err;
        return rc[(size_t)k];
    }
};

// The window rows one device of a split rb_liftover uploads: those of the contigs of its records, which travel in front of their
// CIGAR text; on the first device also the rest of the table, for the check kernel looks at all of it.
struct WindowRows {
    std::vector<uint8_t> seen;                        // contigs whose rows are on their way
    std::vector<std::pair<uint32_t, uint32_t>> done;  // row ranges on their way

    // the rows of the contigs of records ord[lo .. hi)
    int contigs(rb_ctx* c, rb_batch* b, const rb_records* R, const rb_windows* W, const uint32_t* ord, uint32_t lo, uint32_t hi,
                cudaStream_t s) {
        seen.resize(R->n_names, 0);
        for (uint32_t i = lo; i < hi; i++) {
            const uint32_t t = R->t_id[ord[i]];
            if (seen[t]) continue;
            seen[t] = 1;
            const uint32_t r0 = b->h_clo[t], r1 = b->h_chi[t];
            if (r1 <= r0) continue;
            const int rc = windows_upload_rows(c, b, W, r0, r1, s);
            if (rc != RB_OK) return rc;
            done.emplace_back(r0, r1);
        }
        return RB_OK;
    }
    // every row not uploaded yet, then the table check (after `after`, if given) and its verdict
    int rest(rb_ctx* c, rb_batch* b, const rb_records* R, const rb_windows* W, cudaStream_t s, cudaEvent_t after = nullptr) {
        std::sort(done.begin(), done.end());
        uint32_t at = 0;
        int rc = RB_OK;
        for (auto& iv : done) {
            if (rc == RB_OK && iv.first > at) rc = windows_upload_rows(c, b, W, at, iv.first, s);
            at = std::max(at, iv.second);
        }
        if (rc == RB_OK && at < b->n_win) rc = windows_upload_rows(c, b, W, at, b->n_win, s);
        if (rc == RB_OK && after && cudaStreamWaitEvent(s, after, 0) != cudaSuccess) rc = fail(c, RB_ERR_CUDA, "cudaStreamWaitEvent");
        if (rc == RB_OK) rc = windows_check(c, b, R, s);
        if (rc == RB_OK) rc = upload_windows_end(c, b, R, W);  // waits for the verdict
        return rc;
    }
};

// for the length of a call: --qbed (the columns are swapped) and RB_WANT_STATS_TEXT, on the context and all its peers
struct CallFlags {
    rb_ctx* ctx;
    CallFlags(rb_ctx* c, bool invert, bool stats_text) : ctx(c) { set(invert, stats_text); }
    ~CallFlags() { set(false, false); }
    void set(bool invert, bool stats_text) {
        ctx->invert = invert; ctx->stats_text = stats_text;
        for (rb_ctx* p : ctx->peers) { p->invert = invert; p->stats_text = stats_text; }
    }
};
}  // namespace
}  // extern "C++"

// returns 1 when the call was not spread (the caller runs it on the first device), else an rb_status
static int liftover_multi(rb_ctx* ctx, const rb_records* recs, const rb_windows* wins, int policy, uint32_t want, rb_lift_out* out,
                          rb_stats_out* stats) {
    Devices dev(ctx);
    const int D = dev.n;
    if (!recs || !wins || !wins->n_win || recs->n_rec < 2u * (uint32_t)D || !recs->cigar_off || !recs->t_id ||
        recs->cigar_nbytes < ctx->multi_min_bytes || recs->cigar_off[recs->n_rec] != recs->cigar_nbytes || ctx->profiling)
        return 1;
    std::vector<uint32_t> ord, cut;
    bool identity = true;
    if (!emission_order(recs, ord, identity) || !partition_by_bytes(recs, ord, D, cut)) return 1;

    struct Dev { rb_summary sum{}; uint64_t row_base = 0, byte_base = 0; bool general = false; };
    std::vector<Dev> dv((size_t)D);
    Rendezvous rv(D);
    RowsOut rows;
    uint64_t tot_rows = 0, tot_bytes = 0, tot_pairs = 0;
    int call_rc = RB_OK;
    bool fall_back = false;

    dev.run([&](int d, rb_ctx* c) {
        Dev& me = dv[(size_t)d];
        rb_batch* b = c->scratch;
        cudaStream_t s = c->stream;
        int& status = dev.rc[(size_t)d];
        if (status == RB_OK) status = [&]() -> int {
            b->n_rec = 0; b->have_lift = b->have_stats = false;
            int rc = windows_prepare(c, b, recs, wins);
            WindowRows wr;
            if (rc == RB_OK) rc = wr.contigs(c, b, recs, wins, ord.data(), cut[(size_t)d], cut[(size_t)d + 1], s);
            if (rc == RB_OK) rc = windows_upload_aux(c, b, recs, wins, s);
            if (rc != RB_OK) return rc;
            const RecSel sel{identity ? nullptr : ord.data() + cut[(size_t)d], cut[(size_t)d], cut[(size_t)d + 1] - cut[(size_t)d]};
            rc = upload_cigar(c, b, recs, sel);
            if (rc == RB_OK) rc = upload_columns(c, b, recs, sel);
            if (rc == RB_OK) rc = rb_batch_liftover(c, b, policy, want, stats != nullptr, &me.sum);
            if (rc == RB_OK && d == 0) {
                rc = wr.rest(c, b, recs, wins, s);
                me.general = b->general;
            }
            return rc;
        }();
        if (status != RB_OK && b->busy) { cudaStreamSynchronize(s); b->busy = false; }
        rv.meet([&] {  // everybody's sizes are known: lay out the one output block
            call_rc = dev.error(true);
            for (const Dev& o : dv) fall_back |= o.general;  // nested rows / file order != sorted order: single-batch path
            if (call_rc != RB_OK || fall_back) return;
            for (Dev& o : dv) {
                o.row_base = tot_rows; o.byte_base = tot_bytes;
                tot_rows += o.sum.n_out; tot_bytes += o.sum.out_bytes; tot_pairs += o.sum.n_pairs;
            }
            cudaSetDevice(ctx->device);
            call_rc = rows.reserve(ctx, tot_rows, tot_bytes, want, stats != nullptr);
            cudaSetDevice(c->device);
        });
        if (call_rc != RB_OK || fall_back) return;
        // ---- this device's rows -> their place in the merged output ----
        status = [&]() -> int {
            rb_ctx* ctx = c;  // (CU reports into this device's context)
            if (want & RB_WANT_TEXT) launch_add_u64(b->out_line_off.as<uint64_t>(), me.sum.n_out, me.byte_base, s);
            const int rc = rows.copy_rows(c, b, 0, me.sum.n_out, 0, me.sum.out_bytes, me.row_base, me.byte_base, s);
            if (rc != RB_OK) return rc;
            CU(cudaStreamSynchronize(s));
            return RB_OK;
        }();
    });
    if (call_rc == RB_OK) call_rc = dev.error(false);
    if (call_rc != RB_OK || fall_back) { rows.release(); return call_rc != RB_OK ? call_rc : 1; }
    rows.finish(out, stats, tot_rows, tot_bytes, tot_pairs);
    return RB_OK;
}

// rb_stats on a multi-device context: runs of records in FILE order, balanced on CIGAR bytes; rows land at their record index
static int stats_multi(rb_ctx* ctx, const rb_records* recs, rb_stats_out* stats) {
    Devices dev(ctx);
    const int D = dev.n;
    if (!recs || recs->n_rec < 2u * (uint32_t)D || !recs->cigar_off || recs->cigar_nbytes < ctx->multi_min_bytes ||
        recs->cigar_off[recs->n_rec] != recs->cigar_nbytes || ctx->profiling)
        return 1;
    const uint32_t n = recs->n_rec;
    std::vector<uint32_t> cut(1, 0);
    for (int d = 1; d < D; d++) {
        const uint64_t target = recs->cigar_nbytes / (uint64_t)D * (uint64_t)d;
        uint32_t i = (uint32_t)(std::lower_bound(recs->cigar_off, recs->cigar_off + n + 1, target) - recs->cigar_off);
        if (i <= cut.back() || i >= n) return 1;
        cut.push_back(i);
    }
    cut.push_back(n);
    RowsOut rows;
    int rc = rows.reserve_stats(ctx, n);
    if (rc != RB_OK) return rc;
    dev.run([&](int d, rb_ctx* c) {
        rb_batch* b = c->scratch;
        int& status = dev.rc[(size_t)d];
        if (status == RB_OK) status = [&]() -> int {
            rb_ctx* ctx = c;  // (CU reports into this device's context)
            const RecSel sel{nullptr, cut[(size_t)d], cut[(size_t)d + 1] - cut[(size_t)d]};
            int rc = upload_cigar(c, b, recs, sel);
            if (rc == RB_OK) rc = windows_prepare(c, b, recs, nullptr);
            if (rc == RB_OK) rc = upload_columns(c, b, recs, sel);
            if (rc == RB_OK) rc = rb_batch_stats(c, b, nullptr);
            if (rc == RB_OK) rc = rows.copy_rows(c, b, 0, sel.n, 0, 0, sel.r0, 0, c->stream);
            if (rc != RB_OK) return rc;
            CU(cudaStreamSynchronize(c->stream));
            return RB_OK;
        }();
        if (status != RB_OK && b->busy) { cudaStreamSynchronize(c->stream); b->busy = false; }
    });
    rc = dev.error(false);  // devices hold runs of the file order: the first failing device holds the first failing record
    if (rc != RB_OK) { rows.release(); return rc; }
    rows.finish(nullptr, stats, n, 0, 0);
    return RB_OK;
}

// ---- rb_liftover_text: PAF and BED bytes in, the rows of `rb liftover` out -----------------------------------------------------
// One device (or a PAF below multi_min_bytes): rb_batch_upload_paf, rb_batch_set_windows_bed, rb_batch_liftover and the download on
// the context's scratch batch.  D devices, one host thread each:
//   split    plain text: D equal byte ranges, each uploaded by its own device; BGZF: runs of whole blocks balanced on ISIZE, each
//            inflated by its own device.  k_first_newline finds each range's first '\n'; text_split.hpp says which bytes each device
//            parses, and every device gathers them into a fresh buffer (its own bytes: a device copy; the others': peer copies).
//   parse    steps 1 - 3 of rb_batch_upload_paf on every device at once; then the host interns the names device by device (file
//            order: the ids of one device), ranks the contigs by first appearance in the whole file, and every device gets the
//            global name table, its ids, the emission order (contig rank, file index) and rec_base = records on devices before it.
//   windows  every device parses the whole BED against the same name table: identical tables and verdicts everywhere.
//   lift     rb_batch_liftover everywhere (rec_idx always materialised); a lift error reports the smallest global record index.
//   merge    global order = (contig rank, device): k_contig_runs finds each contig's rows on a device, the host lays out ONE pinned
//            block, k_rebase_runs moves the line offsets and every device copies its (contig, device) cells into place — one copy
//            per non-empty cell and output column.
static int liftover_text_one(rb_ctx* ctx, const uint8_t* paf, uint64_t paf_nbytes, const uint8_t* bed, uint64_t bed_nbytes, int policy,
                             uint32_t want, rb_lift_out* out, rb_stats_out* stats, rb_paf_info* paf_info, rb_bed_info* bed_info) {
    if (!ctx->scratch) ctx->scratch = new rb_batch();
    rb_batch* b = ctx->scratch;
    if (b->busy) { CU(cudaStreamSynchronize(ctx->stream)); b->busy = false; }
    int rc = paf_upload_into(ctx, b, paf, paf_nbytes, paf_info);
    if (rc == RB_OK && cudaStreamSynchronize(ctx->stream) != cudaSuccess) {
        (void)cudaGetLastError();
        rc = fail(ctx, RB_ERR_CUDA, "upload failed");
    }
    b->busy = false;
    if (rc == RB_OK) rc = bed_upload_into(ctx, b, bed, bed_nbytes, bed_info);
    if (rc == RB_OK) rc = rb_batch_liftover(ctx, b, policy, want, stats != nullptr, nullptr);
    if (rc == RB_OK) rc = rb_batch_download_lift(ctx, b, want, out, stats);
    if (rc != RB_OK) {
        cudaStreamSynchronize(ctx->stream);
        b->busy = false;
        b->n_win = 0; b->general = false; b->win_pending = false; b->have_lift = false;
        flush_times(ctx);
    }
    return rc;
}

static int liftover_text_multi(rb_ctx* ctx, const uint8_t* paf, uint64_t paf_nbytes, const uint8_t* bed, uint64_t bed_nbytes, int policy,
                               uint32_t want, rb_lift_out* out, rb_stats_out* stats, rb_paf_info* paf_info, rb_bed_info* bed_info) {
    Devices dev(ctx);
    const int D = dev.n;
    // 1. the input's byte ranges
    const bool bgzf = rb_is_bgzf(paf, paf_nbytes) != 0;
    if (!bgzf && paf_nbytes >= 2 && paf[0] == 0x1f && paf[1] == 0x8b)
        return fail(ctx, RB_ERR_BAD_ARG, "rb_batch_upload_paf: a plain gzip stream (not BGZF); inflate it first");
    std::vector<uint64_t> src((size_t)D + 1, paf_nbytes), blk_base((size_t)D, 0);
    src[0] = 0;
    if (bgzf) {
        std::vector<BgzfBlock> blocks;
        std::vector<uint64_t> starts;
        uint64_t total = 0;
        if (!bgzf_blocks(paf, paf_nbytes, blocks, total, &starts)) return fail(ctx, RB_ERR_BAD_ARG, "rb_inflate_bgzf: not a well-formed series of BGZF blocks");
        size_t k = 0;
        for (int d = 1; d < D; d++) {
            const uint64_t target = total / (uint64_t)D * (uint64_t)d + total % (uint64_t)D * (uint64_t)d / (uint64_t)D;
            while (k < blocks.size() && blocks[k].out_off < target) k++;
            src[(size_t)d] = k < blocks.size() ? starts[k] : paf_nbytes;
            blk_base[(size_t)d] = k;
        }
    } else {
        for (int d = 1; d < D; d++) src[(size_t)d] = paf_nbytes / (uint64_t)D * (uint64_t)d + paf_nbytes % (uint64_t)D * (uint64_t)d / (uint64_t)D;
    }
    const uint32_t want_lift = want | RB_WANT_NUMERIC;  // (rec_idx places the rows)
    const bool want_text = (want & (RB_WANT_TEXT | RB_WANT_STATS_TEXT)) != 0;

    struct Dev {
        DevBuf range, own, rank, runs_d, delta;
        uint64_t n = 0, first_nl = rbt::NO_NEWLINE, rec_base = 0;
        uint8_t last = 0;  // the range's last byte
        PafParsed p;
        rb_bed_info bi{};
        rb_summary sum{};
        std::vector<uint64_t> runs;            // row lo / row hi / byte lo / byte hi per contig rank
        std::vector<uint64_t> at_row, at_byte; // where each of its cells goes in the merged output
    };
    std::vector<Dev> dv((size_t)D);
    Rendezvous rv(D);
    std::vector<rbt::Owned> plan;
    std::vector<uint32_t> rank_of;  // name id -> contig rank (first appearance as t_name in the file)
    uint32_t n_ranks = 0, n_names = 0;
    rb_batch* b0 = ctx->scratch ? ctx->scratch : (ctx->scratch = new rb_batch());
    RowsOut rows;
    uint64_t tot_rows = 0, tot_bytes = 0, tot_pairs = 0;
    int call_rc = RB_OK;

    dev.run([&](int d, rb_ctx* c) {
        Dev& me = dv[(size_t)d];
        int& status = dev.rc[(size_t)d];
        rb_batch* b = c->scratch;
        cudaStream_t s = c->stream;
        uint32_t* sc = c->scalars.as<uint32_t>();
        volatile uint64_t* hs = reinterpret_cast<volatile uint64_t*>(c->h_scalars);
        auto cleanup = [&] {
            if (b->busy) { cudaStreamSynchronize(s); b->busy = false; }
            me.range.release(); me.own.release(); me.rank.release(); me.runs_d.release(); me.delta.release();
        };
        // 1. this device's range -> HBM, its first '\n'
        if (status == RB_OK) status = [&]() -> int {
            rb_ctx* ctx = c;  // (CU reports into this device's context)
            const uint64_t len = src[(size_t)d + 1] - src[(size_t)d];
            if (bgzf) {
                const int rc = inflate_to_device(c, paf + src[(size_t)d], len, me.range, me.n, TEXT_PAD, blk_base[(size_t)d]);
                if (rc != RB_OK) return rc;
            } else {
                me.n = len;
                CU(me.range.ensure(len + TEXT_PAD));
                if (len) CU(h2d_copy(me.range.p, paf + src[(size_t)d], len, s));
            }
            if (me.n) {
                CU(cudaMemsetAsync(sc + SC_ERR_TOK, 0xFF, 8, s));
                {
                    KScope k(c, "k_first_newline");
                    launch_first_newline(me.range.as<uint8_t>(), me.n, reinterpret_cast<unsigned long long*>(sc + SC_ERR_TOK), s);
                }
                Publisher(c).u64(0, sc + SC_ERR_TOK).go(s);
            }
            CU(cudaStreamSynchronize(s));
            if (me.n) {
                me.first_nl = hs[0];
                CU(cudaMemcpy(&me.last, me.range.as<uint8_t>() + me.n - 1, 1, cudaMemcpyDeviceToHost));
            }
            return RB_OK;
        }();
        rv.meet([&] {
            call_rc = dev.error(false);
            if (call_rc != RB_OK) return;
            std::vector<uint64_t> size((size_t)D), nl((size_t)D);
            std::vector<uint8_t> ends_nl((size_t)D);
            for (int k = 0; k < D; k++) {
                size[(size_t)k] = dv[(size_t)k].n; nl[(size_t)k] = dv[(size_t)k].first_nl;
                ends_nl[(size_t)k] = dv[(size_t)k].n && dv[(size_t)k].last == '\n';
            }
            plan = rbt::plan_line_split(size, nl, ends_nl);
        });
        if (call_rc != RB_OK) { cleanup(); return; }
        // 2. the lines this device owns -> one fresh buffer
        status = [&]() -> int {
            rb_ctx* ctx = c;  // (CU reports into this device's context)
            const rbt::Owned& o = plan[(size_t)d];
            CU(me.own.ensure(o.bytes + TEXT_PAD));
            uint64_t at = 0;
            for (const rbt::Piece& pc : o.pieces) {
                const Dev& from = dv[(size_t)pc.src];
                if (pc.src == d) CU(cudaMemcpyAsync(me.own.as<uint8_t>() + at, from.range.as<uint8_t>() + pc.off, pc.len, cudaMemcpyDeviceToDevice, s));
                else CU(cudaMemcpyPeerAsync(me.own.as<uint8_t>() + at, c->device, from.range.as<uint8_t>() + pc.off, dev.at(pc.src)->device, pc.len, s));
                at += pc.len;
            }
            CU(cudaStreamSynchronize(s));
            return RB_OK;
        }();
        rv.meet([&] { call_rc = dev.error(false); });  // (every copy out of the ranges has finished)
        me.range.release();
        if (call_rc != RB_OK) { cleanup(); return; }
        // 3. parse
        status = paf_parse_text(c, b, me.own.as<uint8_t>(), plan[(size_t)d].bytes, me.p);
        me.own.release();
        rv.meet([&] {
            uint64_t lines = 0, recs = 0, text = 0, cg = 0;
            for (int k = 0; k < D; k++) {  // the first error or panic in file order
                Dev& o = dv[(size_t)k];
                if (dev.rc[(size_t)k] != RB_OK) { call_rc = dev.error(false); return; }  // (k is the first failing device)
                if (o.p.panic != ~0ull) { call_rc = paf_panic(ctx, o.p.panic, lines); return; }
                o.rec_base = recs;
                lines += o.p.n_lines; recs += o.p.n_rec; text += o.p.text_bytes; cg += o.p.cg_bytes;
            }
            if (lines > 0xFFFFFFFFull) { call_rc = fail(ctx, RB_ERR_REF_PAF_PARSE, "more than 2^32 lines"); return; }
            std::unordered_map<std::string, uint32_t> index;
            b0->h_names.clear();
            b0->h_names_off.assign(1, 0);
            for (int k = 0; k < D; k++) paf_intern(dv[(size_t)k].p, index, b0->h_names, b0->h_names_off);
            n_names = (uint32_t)(b0->h_names_off.size() - 1);
            rank_of.assign(n_names, UINT32_MAX);
            for (int k = 0; k < D; k++) {
                const PafParsed& q = dv[(size_t)k].p;
                for (uint32_t r = 0; r < q.n_rec; r++) {
                    const uint32_t t = q.ids[(size_t)q.n_rec + r];
                    if (rank_of[t] == UINT32_MAX) rank_of[t] = n_ranks++;
                }
            }
            for (uint32_t& r : rank_of) if (r == UINT32_MAX) r = 0;  // (query-only names: never looked up)
            paf_fill_info(paf_info, text, lines, recs, b0->h_names, b0->h_names_off, cg);
        });
        if (call_rc != RB_OK) { cleanup(); return; }
        // 4. names, windows, lift, the contig runs of the rows
        status = [&]() -> int {
            rb_ctx* ctx = c;  // (CU reports into this device's context)
            int rc = paf_upload_names(c, b, me.p, b0->h_names.data(), b0->h_names_off.data(), n_names, rank_of.data());
            if (rc != RB_OK) return rc;
            b->rec_base = (uint32_t)me.rec_base;
            CU(cudaStreamSynchronize(s));
            b->busy = false;
            rc = bed_upload_into(c, b, bed, bed_nbytes, &me.bi);
            if (rc != RB_OK || b->n_rec == 0) return rc;
            rc = rb_batch_liftover(c, b, policy, want_lift, stats != nullptr, &me.sum);
            if (rc != RB_OK) return rc;
            const uint64_t nk = me.sum.n_out, sk = b->row_stride ? b->row_stride : nk;
            CU(me.rank.ensure((size_t)n_names * 4 + 8));
            CU(me.runs_d.ensure((size_t)n_ranks * 32 + 64));
            if (n_names) CU(cudaMemcpyAsync(me.rank.p, rank_of.data(), (size_t)n_names * 4, cudaMemcpyHostToDevice, s));
            CU(cudaMemsetAsync(me.runs_d.p, 0, (size_t)n_ranks * 32, s));
            {
                KScope k(c, "k_contig_runs");
                launch_contig_runs(nk, reinterpret_cast<const uint32_t*>(b->out_num.as<uint64_t>() + 6 * sk), b->rec_base,
                                   b->ids32.as<uint32_t>() + b->n_rec, me.rank.as<uint32_t>(), want_text ? b->out_line_off.as<uint64_t>() : nullptr,
                                   me.sum.out_bytes, me.runs_d.as<uint64_t>(), n_ranks, s);
            }
            me.runs.resize((size_t)n_ranks * 4);
            if (n_ranks) CU(cudaMemcpyAsync(me.runs.data(), me.runs_d.p, (size_t)n_ranks * 32, cudaMemcpyDeviceToHost, s));
            CU(cudaStreamSynchronize(s));
            flush_times(c);
            return RB_OK;
        }();
        auto layout = [&] {  // everybody's runs are known: lay out the one output block, cells in (contig rank, device) order
            call_rc = dev.error(true);
            if (call_rc != RB_OK) return;
            for (int k = 0; k < D; k++) {
                dv[(size_t)k].at_row.assign(n_ranks, 0); dv[(size_t)k].at_byte.assign(n_ranks, 0);
                tot_pairs += dv[(size_t)k].sum.n_pairs;
            }
            for (uint32_t r = 0; r < n_ranks; r++)
                for (int k = 0; k < D; k++) {
                    Dev& o = dv[(size_t)k];
                    if (o.runs.empty()) continue;
                    o.at_row[r] = tot_rows; o.at_byte[r] = tot_bytes;
                    tot_rows += o.runs[n_ranks + r] - o.runs[r];
                    tot_bytes += o.runs[3 * (size_t)n_ranks + r] - o.runs[2 * (size_t)n_ranks + r];
                }
            uint64_t rows_in = 0;
            for (int k = 0; k < D; k++) rows_in += dv[(size_t)k].sum.n_out;
            if (!want_text)  // (no line offsets: the byte count is the devices' sum, as out->paf_nbytes of rb_liftover reports it)
                for (int k = 0; k < D; k++) tot_bytes += dv[(size_t)k].sum.out_bytes;
            if (rows_in != tot_rows) { call_rc = fail(ctx, RB_ERR_CUDA, "rb_liftover_text: the rows of a device are not grouped by contig"); return; }
            call_rc = rows.reserve(ctx, tot_rows, tot_bytes, want, stats != nullptr);
        };
        rv.meet([&] {
            cudaSetDevice(ctx->device);  // (the pinned pool belongs to the first device's context)
            layout();
            cudaSetDevice(c->device);
        });
        if (call_rc != RB_OK) { cleanup(); return; }
        // 5. this device's cells -> their places in the merged output
        status = [&]() -> int {
            rb_ctx* ctx = c;  // (CU reports into this device's context)
            const uint64_t nk = me.sum.n_out, sk = b->row_stride ? b->row_stride : nk;
            if (me.runs.empty() || nk == 0) return RB_OK;
            const uint32_t* rec_idx = reinterpret_cast<const uint32_t*>(b->out_num.as<uint64_t>() + 6 * sk);
            const uint64_t* runs = me.runs.data();
            if (want_text) {
                std::vector<uint64_t> delta(n_ranks, 0);
                for (uint32_t r = 0; r < n_ranks; r++) delta[r] = me.at_byte[r] - runs[2 * (size_t)n_ranks + r];
                CU(me.delta.ensure((size_t)n_ranks * 8 + 8));
                CU(cudaMemcpyAsync(me.delta.p, delta.data(), (size_t)n_ranks * 8, cudaMemcpyHostToDevice, s));  // (pageable: staged before the call returns)
                KScope k(c, "k_rebase_runs");
                launch_rebase_runs(nk, rec_idx, b->rec_base, b->ids32.as<uint32_t>() + b->n_rec, me.rank.as<uint32_t>(), me.delta.as<uint64_t>(),
                                   b->out_line_off.as<uint64_t>(), s);
            }
            for (uint32_t r = 0; r < n_ranks; r++) {
                const uint64_t lo = runs[r], hi = runs[n_ranks + r], blo = runs[2 * (size_t)n_ranks + r], bhi = runs[3 * (size_t)n_ranks + r];
                if (hi <= lo) continue;
                const int rc = rows.copy_rows(c, b, lo, hi - lo, blo, bhi - blo, me.at_row[r], me.at_byte[r], s);
                if (rc != RB_OK) return rc;
            }
            CU(cudaStreamSynchronize(s));
            flush_times(c);
            return RB_OK;
        }();
        cleanup();
    });
    if (call_rc == RB_OK) call_rc = dev.error(false);
    if (call_rc != RB_OK) { rows.release(); return call_rc; }
    if (bed_info) *bed_info = dv[0].bi;
    rows.finish(out, stats, tot_rows, tot_bytes, tot_pairs);
    return RB_OK;
}

int rb_liftover_text(rb_ctx* ctx, const uint8_t* paf, uint64_t paf_nbytes, const uint8_t* bed, uint64_t bed_nbytes, int policy,
                     uint32_t want, rb_lift_out* out, rb_stats_out* stats, rb_paf_info* paf_info, rb_bed_info* bed_info) {
    if (!ctx) return RB_ERR_NO_DEVICE;
    if (paf_info) memset(paf_info, 0, sizeof *paf_info);
    if (bed_info) memset(bed_info, 0, sizeof *bed_info);
    if (!out) return fail(ctx, RB_ERR_BAD_ARG, "out is null");
    memset(out, 0, sizeof *out);
    if (stats) memset(stats, 0, sizeof *stats);
    if ((!paf && paf_nbytes) || (!bed && bed_nbytes)) return fail(ctx, RB_ERR_BAD_ARG, "rb_liftover_text: null data");
    if (want & RB_WANT_QBED) return fail(ctx, RB_ERR_BAD_ARG, "rb_liftover_text: RB_WANT_QBED is not supported");
    if (policy != RB_POLICY_RIGHTMOST && policy != RB_POLICY_EARLY_EXIT) return fail(ctx, RB_ERR_BAD_ARG, "unknown policy %d", policy);
    if ((want & RB_WANT_STATS_TEXT) && (want & RB_WANT_TEXT)) return fail(ctx, RB_ERR_BAD_ARG, "RB_WANT_STATS_TEXT and RB_WANT_TEXT exclude each other");
    cudaSetDevice(ctx->device);
    if (ctx->peers.empty() || paf_nbytes < ctx->multi_min_bytes)
        return liftover_text_one(ctx, paf, paf_nbytes, bed, bed_nbytes, policy, want, out, stats, paf_info, bed_info);
    const int rc = liftover_text_multi(ctx, paf, paf_nbytes, bed, bed_nbytes, policy, want, out, stats, paf_info, bed_info);
    if (rc != RB_OK) {
        if (paf_info && !paf_info->names_off) memset(paf_info, 0, sizeof *paf_info);
        memset(out, 0, sizeof *out);
        if (stats) memset(stats, 0, sizeof *stats);
    }
    return rc;
}

// ---- rb_liftover in slices, on one device or several ------------------------------------------------
// A large call is cut into K runs of records that are consecutive in EMISSION order (liftover.rs:151-164), of about equal
// CIGAR size; slice k belongs to device k mod D (D = 1: the whole pipeline on one GPU).  Every device (one host thread each)
// works through its slices in order on a ping-pong pair of work areas and three streams: the UPLOAD stream copies the next
// slice (its CIGAR text, gathered run by run when the file order is not the emission order, and the window rows of its
// contigs), the COMPUTE stream runs the kernels, the COPY stream sends the rows of the slice before to the host — so both
// PCIe directions and the SMs of every GPU are busy at once, and the HBM footprint of the intermediates is bounded by two
// slices per device.  The rows of all devices land in ONE pinned block in emission order: where slice k's rows go is the sum
// of the sizes of the slices before it — a host-side wait on the other device threads, which run the slices just before
// this one at the same time (nothing else is exchanged between the GPUs).  Row tables are laid out with the exact upper bound
// on rows (host-side binary searches over the sorted windows); the text size is extrapolated from the first slice, and an
// underestimate — or a window table that turns out to be nested / not in file order — makes the function return 1: the
// caller then takes the path that sizes everything exactly.
static int ensure_slice_streams(rb_ctx* ctx) {
    if (ctx->copy_stream) return RB_OK;
    CU(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&ctx->up_stream, cudaStreamNonBlocking));
    for (int k = 0; k < 2; k++) {
        CU(cudaEventCreateWithFlags(&ctx->ev_up[k], cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&ctx->ev_done[k], cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&ctx->ev_d2h[k], cudaEventDisableTiming));
    }
    return RB_OK;
}

static int liftover_sliced(rb_ctx* ctx, const rb_records* recs, const rb_windows* wins, int policy, uint32_t want, rb_lift_out* out,
                           rb_stats_out* stats) {
    const uint64_t SLICE_MIN_BYTES = ctx->slice_min_bytes;
    Devices dev(ctx);
    const int D = dev.n;
    std::vector<uint32_t> ord;  // records in emission order
    bool identity = true;
    const bool try_slices = SLICE_MIN_BYTES && !ctx->profiling && recs && wins && wins->n_win && recs->n_rec >= 2 && recs->cigar_off &&
                            recs->t_id && recs->t_st && recs->t_en && recs->cigar_nbytes >= 2 * SLICE_MIN_BYTES &&
                            (policy == RB_POLICY_RIGHTMOST || policy == RB_POLICY_EARLY_EXIT) &&
                            recs->cigar_off[recs->n_rec] == recs->cigar_nbytes && emission_order(recs, ord, identity);
    if (!try_slices) return 1;
    const bool trace = getenv("RB_TRACE") != nullptr;
    const auto t_begin = std::chrono::steady_clock::now();
    auto T = [&](const char* what, uint32_t k) {
        if (trace) fprintf(stderr, "[rb_liftover] %8.3f ms  %s %u\n",
                           std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count(), what, k);
    };

    // ---- slice boundaries (record granularity, balanced on CIGAR bytes) and an upper bound on the rows ----
    const uint32_t n = recs->n_rec;
    const uint64_t total_bytes = recs->cigar_nbytes;
    // at most 8 slices per device (RB_MAX_SLICES overrides).  Measured at C5 on one B200 (12.6 GB up, 17.6 GB down): 8 / 16 / 32 / 64
    // slices -> 447 / 431 / 433 / 436 ms per call, 30 / 15 / 8 / 4 GB of HBM in use, 1.6 / 2.6 / 2.7 / 3.5 s for the first call:
    // the fill and drain of the pipeline are not what keeps the call at 70 of the link's 95 GB/s (both directions)
    uint64_t k_cap = 8ull * (uint64_t)D;
    if (const char* e = getenv("RB_MAX_SLICES")) k_cap = std::max<uint64_t>(2, strtoull(e, nullptr, 10));
    const uint32_t K = (uint32_t)std::min<uint64_t>(k_cap, std::max<uint64_t>(2, total_bytes / SLICE_MIN_BYTES));
    std::vector<uint32_t> cut(1, 0);  // slice k = records ord[cut[k] .. cut[k+1]) : consecutive in EMISSION order
    {
        // the very first slice is half the size of the others: its rows reach the copy engine sooner, yet their download still
        // covers the production of the next slice; from then on the downloads are the bottleneck
        const uint64_t unit = total_bytes / (2 * (uint64_t)K - 1);  // sizes 1 : 2 : 2 : ... in units
        uint64_t acc = 0, target = unit;
        uint32_t k = 1;
        for (uint32_t i = 0; i < n && k < K; i++) {
            const uint32_t r = ord[i];
            if (recs->cigar_off[r + 1] < recs->cigar_off[r]) break;  // malformed offsets: reported by the upload
            acc += recs->cigar_off[r + 1] - recs->cigar_off[r];
            if (acc >= target && i + 1 < n) { cut.push_back(i + 1); k++; target = unit + 2 * unit * (uint64_t)(k - 1); }
        }
    }
    cut.push_back(n);
    const uint32_t n_slices = (uint32_t)cut.size() - 1;
    if (n_slices < (uint32_t)D) return 1;  // fewer slices than devices (a few huge records): the exact multi-device path
    dev.run([&](int d, rb_ctx* c) {  // streams, work areas, host-side window bookkeeping (contig ranges); the rows travel with the slices
        int& status = dev.rc[(size_t)d];
        if (status == RB_OK) status = ensure_slice_streams(c);
        if (status != RB_OK) return;
        c->scratch->n_rec = 0; c->scratch->have_lift = c->scratch->have_stats = false;
        for (int k = 0; k < 2; k++) {
            if (!c->slice[k]) c->slice[k] = new rb_batch();
            c->slice[k]->wsrc = c->scratch;
        }
        status = windows_prepare(c, c->scratch, recs, wins);
    });
    if (const int rc = dev.error(false)) return rc;
    rb_batch* wb0 = ctx->scratch;
    uint64_t cap_rows = 0;  // pairs of the unstripped records >= pairs examined >= rows
    for (uint32_t i = 0; i < n; i++) {
        const uint32_t lo = wb0->h_clo[recs->t_id[i]], hi = wb0->h_chi[recs->t_id[i]];
        const uint64_t* a0 = std::upper_bound(wins->en + lo, wins->en + hi, recs->t_st[i]);   // first en > t_st (en is monotone here)
        const uint64_t* a1 = std::lower_bound(wins->st + lo, wins->st + hi, recs->t_en[i]);   // first st >= t_en
        const uint32_t i0 = (uint32_t)(a0 - wins->en), i1 = (uint32_t)(a1 - wins->st);
        if (i1 > i0) cap_rows += i1 - i0;
    }

    // ---- state shared by the device threads ----
    struct Shared {
        std::mutex m;
        std::condition_variable cv;
        std::vector<rb_summary> sum;       // per slice, valid once known[k]
        std::vector<uint8_t> known;
        bool abort = false;                // an error, or the estimates do not hold: everybody stops
        bool fall_back = false;            // ... and the caller takes the exact path
    } sh;
    sh.sum.assign(n_slices, rb_summary{});
    sh.known.assign(n_slices, 0);
    RowsOut rows;
    memset(out, 0, sizeof *out);
    if (stats) memset(stats, 0, sizeof *stats);

    auto stop = [&](bool fall_back) {
        std::lock_guard<std::mutex> lk(sh.m);
        sh.fall_back = sh.fall_back || fall_back;
        sh.abort = true;
        sh.cv.notify_all();
    };

    dev.run([&](int d, rb_ctx* c) {
        rb_batch* wb = c->scratch;
        cudaStream_t A = c->stream, B = c->copy_stream, U = c->up_stream;
        std::vector<uint32_t> mine;  // this device's slices
        for (uint32_t k = (uint32_t)d; k < n_slices; k += (uint32_t)D) mine.push_back(k);
        WindowRows wr;  // a slice only needs the window rows of its own contigs
        auto upload_slice = [&](size_t j) {  // j = position in `mine`
            const uint32_t k = mine[j];
            rb_batch* sb = c->slice[j & 1];
            const RecSel sel{identity ? nullptr : ord.data() + cut[k], cut[k], cut[k + 1] - cut[k]};
            // on the upload stream, beside the kernels of the slice before; the work area's own previous kernels (two slices
            // back) must have finished reading its inputs
            if (j >= 2 && cudaStreamWaitEvent(U, c->ev_done[j & 1], 0) != cudaSuccess) return fail(c, RB_ERR_CUDA, "cudaStreamWaitEvent");
            int r2 = j ? wr.contigs(c, wb, recs, wins, ord.data(), cut[k], cut[k + 1], U) : (int)RB_OK;
            if (r2 != RB_OK) return r2;
            c->upload_on = U;
            r2 = upload_cigar(c, sb, recs, sel);
            if (r2 == RB_OK) r2 = upload_columns(c, sb, recs, sel);
            c->upload_on = nullptr;
            sb->wsrc = wb;
            if (r2 == RB_OK && cudaEventRecord(c->ev_up[j & 1], U) != cudaSuccess) r2 = fail(c, RB_ERR_CUDA, "cudaEventRecord");
            return r2;
        };
        auto run = [&]() -> int {
            rb_ctx* ctx = c;  // (CU reports into this device's context)
            if (mine.empty()) return RB_OK;
            int rc = wr.contigs(c, wb, recs, wins, ord.data(), cut[mine[0]], cut[mine[0] + 1], A);
            if (rc == RB_OK) rc = windows_upload_aux(c, wb, recs, wins, A);
            if (rc != RB_OK) return rc;
            CU(cudaEventRecord(c->ev_wfirst, A));
            rc = upload_slice(0);
            if (rc != RB_OK) return rc;
            for (size_t j = 0; j < mine.size(); j++) {
                const uint32_t k = mine[j];
                rb_batch* sb = c->slice[j & 1];
                if (j + 1 < mine.size()) {  // the next slice's host->device copies go in front of this slice's kernels
                    rc = upload_slice(j + 1);
                    if (rc != RB_OK) return rc;
                }
                CU(cudaStreamWaitEvent(A, c->ev_up[j & 1], 0));                // this slice's inputs have arrived
                if (j >= 2) CU(cudaStreamWaitEvent(A, c->ev_d2h[j & 1], 0));  // this work area's previous rows have left the device
                sb->byte_base = 0;
                rb_summary sm{};
                rc = rb_batch_liftover(c, sb, policy, want, stats != nullptr, &sm);
                if (rc != RB_OK) return rc;
                if (d == 0) T("kernels enqueued (sizes known)", k);
                CU(cudaEventRecord(c->ev_done[j & 1], A));
                uint64_t byte_base = 0, row_base = 0;
                {   // publish this slice's sizes; wait for the slices in front of it (they run on the other devices right now)
                    std::unique_lock<std::mutex> lk(sh.m);
                    sh.sum[k] = sm;
                    sh.known[k] = 1;
                    sh.cv.notify_all();
                    sh.cv.wait(lk, [&] {
                        if (sh.abort) return true;
                        for (uint32_t q = 0; q < k; q++)
                            if (!sh.known[q]) return false;
                        return k == 0 || rows.blk != nullptr;
                    });
                    if (sh.abort) return RB_OK;
                    for (uint32_t q = 0; q < k; q++) { byte_base += sh.sum[q].out_bytes; row_base += sh.sum[q].n_out; }
                    if (k == 0) {  // sizes of the first slice are known: reserve the pinned output (text size extrapolated, rows bounded)
                        const uint64_t slice_bytes = sb->n_bytes;
                        const double scale = slice_bytes ? (double)total_bytes / (double)slice_bytes : 1.0;
                        size_t text_est = 0;
                        if (want & RB_WANT_TEXT) {
                            text_est = (size_t)((double)sm.out_bytes * scale * 1.25) + (size_t)std::min<uint64_t>(4u << 20, total_bytes / 4 + 4096);  // slices differ in their rows-per-byte mix
                            if (sm.n_out == 0) text_est = (size_t)total_bytes + (size_t)cap_rows * 200 + 4096;  // nothing to extrapolate from
                        }
                        rc = rows.reserve(c, cap_rows, text_est, want, stats != nullptr);  // (slice 0 is the first device's: c is ctx)
                        if (rc != RB_OK) return rc;
                        sh.cv.notify_all();
                    }
                }
                if (((want & RB_WANT_TEXT) && byte_base + sm.out_bytes > rows.cap_text) || row_base + sm.n_out > cap_rows) {
                    // the text extrapolation was too small (or the table is not the sorted, non-nested layout the row bound assumes)
                    if (d == 0) T("text estimate too small: falling back", k);
                    stop(true);
                    return RB_OK;
                }
                // ---- device -> host of this slice on the copy stream ----
                CU(cudaStreamWaitEvent(B, c->ev_done[j & 1], 0));
                if (want & RB_WANT_TEXT) launch_add_u64(sb->out_line_off.as<uint64_t>(), sm.n_out, byte_base, B);  // offsets in the caller's concatenated text
                rc = rows.copy_rows(c, sb, 0, sm.n_out, 0, sm.out_bytes, row_base, byte_base, B);
                if (rc != RB_OK) return rc;
                CU(cudaEventRecord(c->ev_d2h[j & 1], B));
            }
            if (d == 0) {  // rows no slice of this device needed, then the table check (its verdict is read before the call returns)
                rc = wr.rest(c, wb, recs, wins, U, c->ev_wfirst);
                if (rc != RB_OK) return rc;
                if (wb->general) {  // nested rows / file order != sorted order: the single-batch path handles those (rare)
                    T("general window layout: falling back", 0);
                    stop(true);
                    return RB_OK;
                }
            }
            CU(cudaStreamSynchronize(B));
            return RB_OK;
        };
        int& status = dev.rc[(size_t)d];
        if (status == RB_OK) status = run();
        if (status != RB_OK) stop(false);
        // whatever happened: nothing of this call may still be in flight on this device when the function returns
        c->upload_on = nullptr;
        cudaStreamSynchronize(U);
        cudaStreamSynchronize(A);
        cudaStreamSynchronize(B);
        for (int k = 0; k < 2; k++)
            if (c->slice[k]) c->slice[k]->busy = false;
        wb->busy = false;
    });
    T("all devices drained", n_slices);
    const int rc = dev.error(true);  // the first error in record order wins
    if (rc != RB_OK || sh.fall_back) { rows.release(); return rc != RB_OK ? rc : 1; }  // (1: the exact path)
    uint64_t row_base = 0, byte_base = 0, pairs = 0;
    for (uint32_t k = 0; k < n_slices; k++) { row_base += sh.sum[k].n_out; byte_base += sh.sum[k].out_bytes; pairs += sh.sum[k].n_pairs; }
    rows.finish(out, stats, row_base, byte_base, pairs);
    return RB_OK;
}

// query and target change places: the column pointers are swapped (the ops get inverted on the device right after tokenising)
static rb_records swap_query_target(const rb_records& r) {
    rb_records s = r;
    std::swap(s.q_len, s.t_len); std::swap(s.q_st, s.t_st); std::swap(s.q_en, s.t_en);
    std::swap(s.q_id, s.t_id);
    return s;
}

int rb_liftover(rb_ctx* ctx, const rb_records* recs, const rb_windows* wins, int policy, uint32_t want, rb_lift_out* out,
                rb_stats_out* stats) {
    if (!ctx) return RB_ERR_NO_DEVICE;
    if (!out) return fail(ctx, RB_ERR_BAD_ARG, "out is null");
    // liftover --qbed (liftover.rs:139-148): every record swaps query and target first
    const bool invert = (want & RB_WANT_QBED) && recs;
    rb_records swapped;
    if (invert) {
        swapped = swap_query_target(*recs);
        recs = &swapped;
    }
    want &= ~RB_WANT_QBED;
    const bool stats_text = (want & RB_WANT_STATS_TEXT) != 0;
    if (stats_text) {
        if (want & RB_WANT_TEXT) return fail(ctx, RB_ERR_BAD_ARG, "RB_WANT_STATS_TEXT and RB_WANT_TEXT exclude each other");
        want = (want & ~RB_WANT_STATS_TEXT) | RB_WANT_TEXT;  // from here on the stats rows are "the text"
    }
    CallFlags flags(ctx, invert, stats_text);
    cudaSetDevice(ctx->device);
    {   // large calls: slices dealt round-robin to the context's devices, both PCIe directions and the SMs busy at once
        const int src = liftover_sliced(ctx, recs, wins, policy, want, out, stats);
        if (src != 1) return src;  // (1: not sliced — small call, slicing off, or an estimate / window layout that needs the exact path)
    }
    if (!ctx->peers.empty() && (policy == RB_POLICY_RIGHTMOST || policy == RB_POLICY_EARLY_EXIT)) {
        const int mrc = liftover_multi(ctx, recs, wins, policy, want, out, stats);
        if (mrc != 1) return mrc;  // (1: not spread — too small, or a window layout the single-batch path handles)
    }
    if (!ctx->scratch) ctx->scratch = new rb_batch();
    return liftover_unsliced(ctx, recs, wins, policy, want, out, stats);
}

// replaces the `for paf in records { aligned_pairs(); break_paf_on_indels(); println! }` loop of `rb break-paf`
// (main.rs:271-281)
int rb_break_paf(rb_ctx* ctx, const rb_records* recs, uint32_t max_size, int policy, uint32_t want, rb_lift_out* out,
                 rb_stats_out* stats) {
    if (!ctx) return RB_ERR_NO_DEVICE;
    if (!out) return fail(ctx, RB_ERR_BAD_ARG, "out is null");
    cudaSetDevice(ctx->device);
    if (!ctx->scratch) ctx->scratch = new rb_batch();
    rb_batch* b = ctx->scratch;
    b->file_order = true;  // rows follow the records in file order, not contig by contig
    int rc = upload_into(ctx, b, recs, nullptr);
    b->file_order = false;
    if (rc != RB_OK) return rc;
    rc = rb_batch_break(ctx, b, max_size, policy, want, stats != nullptr, nullptr);
    if (rc != RB_OK) return rc;
    return rb_batch_download_lift(ctx, b, want, out, stats);
}

// replaces the `for rec in &paf.records { println!("{}", paf_swap_query_and_target(rec)); }` loop of `rb invert`
// (main.rs:176-182, paf.rs:1050-1094)
int rb_invert(rb_ctx* ctx, const rb_records* recs, uint32_t want, rb_lift_out* out) {
    if (!ctx) return RB_ERR_NO_DEVICE;
    if (!out || !recs) return fail(ctx, RB_ERR_BAD_ARG, "recs / out is null");
    cudaSetDevice(ctx->device);
    if (!ctx->scratch) ctx->scratch = new rb_batch();
    rb_batch* b = ctx->scratch;
    const rb_records swapped = swap_query_target(*recs);
    CallFlags flags(ctx, true, false);
    b->file_order = true;
    int rc = upload_into(ctx, b, &swapped, nullptr);
    b->file_order = false;
    if (rc != RB_OK) return rc;
    rc = batch_invert(ctx, b, want & ~RB_WANT_QBED, nullptr);
    if (rc != RB_OK) return rc;
    return rb_batch_download_lift(ctx, b, want & ~RB_WANT_QBED, out, nullptr);
}

// `rb trim-paf` = Paf::overlapping_paf_recs + the print loop (main.rs:218-230, paf.rs:210-305, trim_overlap.rs:36-86) in three
// steps: begin (upload in query-name order, tokenise, strip, scans, untruncated views), rounds (on the device: per query name
// the pair to trim, its split point, the two truncations), end (one row per record).  rb_trim_paf() runs them back to back;
// the stepping calls exist for the multi-GPU form, where the decision to run another round is global (see rbcuda.h).
int rb_trim_paf_begin(rb_ctx* ctx, const rb_records* recs, int match_score, int diff_score, int indel_score, int policy) {
    if (!ctx) return RB_ERR_NO_DEVICE;
    if (!recs) return fail(ctx, RB_ERR_BAD_ARG, "recs is null");
    if (ctx->scratch) ctx->scratch->trim_ready = false;
    if (policy != RB_POLICY_RIGHTMOST && policy != RB_POLICY_EARLY_EXIT) return fail(ctx, RB_ERR_BAD_ARG, "unknown search policy %d", policy);
    if (recs->n_rec && (!recs->q_id || !recs->names_off || (!recs->names && recs->n_names && recs->names_off[recs->n_names])))
        return fail(ctx, RB_ERR_BAD_ARG, "rb_records: null column");
    cudaSetDevice(ctx->device);
    if (!ctx->scratch) ctx->scratch = new rb_batch();
    rb_batch* b = ctx->scratch;
    cudaStream_t s = ctx->stream;
    const uint32_t n = recs->n_rec;

    // records.sort_by_key(|rec| rec.q_name.clone()) — stable, byte-wise (paf.rs:224)
    for (uint32_t i = 0; i < n; i++)
        if (recs->q_id[i] >= recs->n_names) return fail(ctx, RB_ERR_BAD_ARG, "name id out of range at record %u", i);
    auto name_of = [&](uint32_t r, const uint8_t*& p, size_t& len) {
        const uint32_t q = recs->q_id[r];
        p = recs->names + recs->names_off[q];
        len = (size_t)(recs->names_off[q + 1] - recs->names_off[q]);
    };
    auto name_cmp = [&](uint32_t x, uint32_t y) {
        const uint8_t *px, *py;
        size_t lx, ly;
        name_of(x, px, lx); name_of(y, py, ly);
        const int c = memcmp(px, py, lx < ly ? lx : ly);
        return c ? c : (lx < ly ? -1 : (lx > ly ? 1 : 0));
    };
    std::vector<uint32_t>& perm = b->trim_perm;
    perm.resize(n);
    for (uint32_t i = 0; i < n; i++) perm[i] = i;
    std::stable_sort(perm.begin(), perm.end(), [&](uint32_t x, uint32_t y) { return name_cmp(x, y) < 0; });

    const RecSel sel_all{perm.data(), 0, n};
    b->file_order = true;
    int rc = upload_cigar(ctx, b, recs, sel_all);
    if (rc == RB_OK) rc = windows_prepare(ctx, b, recs, nullptr);
    if (rc == RB_OK) rc = upload_columns(ctx, b, recs, sel_all);
    b->file_order = false;
    if (rc != RB_OK) {
        if (b->busy) { cudaStreamSynchronize(s); b->busy = false; }
        return rc;
    }
    b->have_lift = false;
    rc = run_tok(ctx, b);
    if (rc != RB_OK) return rc;
    uint32_t* sc = ctx->scalars.as<uint32_t>();
    ErrSlots err{reinterpret_cast<unsigned long long*>(sc + SC_ERR_TOK), reinterpret_cast<unsigned long long*>(sc + SC_ERR_REC)};
    {   // remove_trailing_indels on every record (paf.rs:218-221)
        KScope k(ctx, "k_rec_prep");
        launch_rec_prep(1, rec_input(b), b->op_off.as<uint64_t>(), b->ops.as<uint32_t>(), nullptr, WinView{}, b->recs.as<RecInfo>(),
                        b->pair_cnt.as<uint32_t>(), StatsDev{}, err, s);
    }
    rc = run_scan(ctx, b, nullptr);
    if (rc != RB_OK) return rc;
    {
        KScope k(ctx, "k_rec_prep");
        launch_rec_prep(2, rec_input(b), b->op_off.as<uint64_t>(), b->ops.as<uint32_t>(), b->samples.as<Ctr>(), WinView{},
                        b->recs.as<RecInfo>(), b->pair_cnt.as<uint32_t>(), StatsDev{}, err, s);
    }
    volatile uint64_t* hs = reinterpret_cast<volatile uint64_t*>(ctx->h_scalars);
    Publisher(ctx).u64(0, sc + SC_ERR_TOK).u64(1, sc + SC_ERR_REC).u64(2, b->op_off.as<uint64_t>() + n).u32(3, sc + SC_MISC).go(s);
    CU(cudaStreamSynchronize(s));
    b->busy = false;
    if ((uint32_t)hs[3] & 1u) {
        launch_check_clips(b->ops.as<uint32_t>(), b->op_off.as<uint64_t>(), n, err, s);
        Publisher(ctx).u64(0, sc + SC_ERR_TOK).u64(1, sc + SC_ERR_REC).go(s);
        CU(cudaStreamSynchronize(s));
    }
    rc = map_err(ctx, b, hs[0], hs[1]);
    if (rc != RB_OK) { flush_times(ctx); return rc; }
    const uint64_t n_ops = hs[2];

    // per-op query / score prefixes and the untruncated views
    const TrimScores scores{match_score, diff_score, indel_score};
    CU(b->trim_qp.ensure(n_ops * 4 + 64));  // (the op count is known by now: 12 B per op, not per byte of text / 2)
    CU(b->trim_wp.ensure(n_ops * 8 + 64));
    CU(b->trim_ap.ensure(n_ops * 4 + 64));  // alignment columns before each op (the early-exit policy's probe arithmetic)
    b->trim_policy = policy;
    CU(b->trim_views.ensure((size_t)n * sizeof(TrimView) + 64));
    {
        KScope k(ctx, "k_trim_scan");
        launch_trim_scan(b->ops.as<uint32_t>(), b->recs.as<RecInfo>(), n, scores, b->trim_qp.as<uint32_t>(), b->trim_ap.as<uint32_t>(),
                         b->trim_wp.as<long long>(), b->trim_views.as<TrimView>(), policy, s);
    }
    std::vector<TrimView> h_views(n);
    if (n) CU(cudaMemcpyAsync(h_views.data(), b->trim_views.p, (size_t)n * sizeof(TrimView), cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    std::vector<TrimSpan> spans(n);
    for (uint32_t i = 0; i < n; i++) {
        if (h_views[i].bad)
            return fail(ctx, RB_ERR_UNSUPPORTED, "record %u: rb_trim_paf wants records that start and end on an M/=/X op after the indel strip", perm[i]);
        spans[i].q_st = h_views[i].q_st; spans[i].q_en = h_views[i].q_en;
        spans[i].name = i ? spans[i - 1].name + (name_cmp(perm[i - 1], perm[i]) != 0 ? 1u : 0u) : 0u;
    }
    const uint64_t max_score = (uint64_t)std::max({std::llabs((long long)match_score), std::llabs((long long)diff_score),
                                                   std::llabs((long long)indel_score)});
    // query-name groups of the sorted set; the rounds themselves run on the device (k_trim_select picks each name's pair from
    // the current spans), enqueued in batches — the host only looks at the 32-byte round state after every batch
    std::vector<uint32_t> grp_off;
    for (uint32_t i = 0; i < n; i++)
        if (i == 0 || spans[i].name != spans[i - 1].name) grp_off.push_back(i);
    const uint32_t n_groups = (uint32_t)grp_off.size();
    grp_off.push_back(n);
    for (uint32_t g = 0; g < n_groups; g++)
        if (grp_off[g + 1] - grp_off[g] > 65535u)
            return fail(ctx, RB_ERR_UNSUPPORTED, "more than 65535 records on one query name (record %u)", perm[grp_off[g]]);
    b->trim_scores[0] = match_score; b->trim_scores[1] = diff_score; b->trim_scores[2] = indel_score;
    b->trim_max_score = max_score; b->trim_groups = n_groups; b->trim_n_ops = n_ops;
    const size_t o_sel = 0, o_keys = o_sel + ((size_t)n_groups + 1) * sizeof(TrimPairSel), o_info = o_keys + ((size_t)n_groups + 1) * 8,
                 o_grp = o_info + 32, o_end = o_grp + ((size_t)n_groups + 2) * 4;
    CU(b->trim_sel.ensure(o_end + 64));
    uint8_t* tb = b->trim_sel.as<uint8_t>();
    CU(b->trim_drop.ensure((size_t)n + 64));
    CU(cudaMemsetAsync(b->trim_drop.p, 0, (size_t)n + 1, s));
    CU(cudaMemsetAsync(tb + o_info, 0, 32, s));
    CU(cudaMemcpyAsync(tb + o_grp, grp_off.data(), ((size_t)n_groups + 1) * 4, cudaMemcpyHostToDevice, s));
    CU(cudaStreamSynchronize(s));  // grp_off is a pageable local
    b->trim_o[0] = o_sel; b->trim_o[1] = o_keys; b->trim_o[2] = o_info; b->trim_o[3] = o_grp;
    b->trim_ready = true;
    return RB_OK;
}

// `batch` rounds enqueued back to back, then one look at the 32-byte round state.  auto_done: a round that leaves nothing
// waiting ends the call (single-GPU form); otherwise the caller decides (multi-GPU form: OR over the ranks).
static int trim_rounds(rb_ctx* ctx, rb_batch* b, int batch, bool auto_done, uint32_t* waiting, uint32_t* done) {
    cudaStream_t s = ctx->stream;
    uint8_t* tb = b->trim_sel.as<uint8_t>();
    const size_t o_sel = b->trim_o[0], o_keys = b->trim_o[1], o_info = b->trim_o[2], o_grp = b->trim_o[3];
    const TrimScores scores{b->trim_scores[0], b->trim_scores[1], b->trim_scores[2]};
    const std::vector<uint32_t>& perm = b->trim_perm;
    struct { uint32_t waiting, done, rounds, status, err_l, err_r, last_waiting, pad; } info{};
    {
        KScope k(ctx, "k_trim_rounds");
        launch_trim_rounds(batch, auto_done, reinterpret_cast<const uint32_t*>(tb + o_grp), b->trim_groups, b->ops.as<uint32_t>(),
                           b->recs.as<RecInfo>(), b->trim_qp.as<uint32_t>(), b->trim_wp.as<long long>(), b->trim_ap.as<uint32_t>(),
                           b->trim_policy, scores, b->trim_max_score,
                           b->trim_views.as<TrimView>(), b->trim_drop.as<uint8_t>(), tb + o_sel,
                           reinterpret_cast<unsigned long long*>(tb + o_keys), tb + o_info, s);
    }
    CU(cudaMemcpyAsync(&info, tb + o_info, 32, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    if (info.status == 1) {
        flush_times(ctx);
        b->trim_ready = false;
        return fail(ctx, RB_ERR_REF_INTEGRITY, "records %u / %u: truncate_record_by_query leaves spans that disagree with the CIGAR "
                    "(check_integrity().unwrap() panics, paf.rs:819-822)", perm[info.err_l], perm[info.err_r]);
    }
    if (info.status) {
        flush_times(ctx);
        b->trim_ready = false;
        return fail(ctx, RB_ERR_UNSUPPORTED, "records %u / %u: overlap x score exceeds the reference's i32 sums", perm[info.err_l], perm[info.err_r]);
    }
    if (waiting) *waiting = info.last_waiting;
    if (done) *done = info.done;
    return RB_OK;
}

int rb_trim_paf_round(rb_ctx* ctx, int* waiting) {
    if (!ctx) return RB_ERR_NO_DEVICE;
    rb_batch* b = ctx->scratch;
    if (!b || !b->trim_ready) return fail(ctx, RB_ERR_BAD_ARG, "rb_trim_paf_round without rb_trim_paf_begin");
    cudaSetDevice(ctx->device);
    uint32_t w = 0;
    const int rc = trim_rounds(ctx, b, 1, false, &w, nullptr);
    if (waiting) *waiting = w ? 1 : 0;
    return rc;
}

int rb_trim_paf_end(rb_ctx* ctx, int remove_contained, uint32_t want, rb_lift_out* out, rb_stats_out* stats) {
    if (!ctx) return RB_ERR_NO_DEVICE;
    if (!out) return fail(ctx, RB_ERR_BAD_ARG, "out is null");
    rb_batch* b = ctx->scratch;
    if (!b || !b->trim_ready) return fail(ctx, RB_ERR_BAD_ARG, "rb_trim_paf_end without rb_trim_paf_begin");
    cudaSetDevice(ctx->device);
    cudaStream_t s = ctx->stream;
    b->trim_ready = false;
    if (want & RB_WANT_STATS_TEXT) return fail(ctx, RB_ERR_BAD_ARG, "RB_WANT_STATS_TEXT is an rb_liftover mode");
    b->stats_text = false;
    const uint32_t n = b->n_rec;
    const uint64_t n_ops = b->trim_n_ops;
    want &= ~RB_WANT_QBED;
    int rc = RB_OK;
    b->trim_has_drop = remove_contained != 0 && n > 0;
    const uint64_t P = n;
    CU(b->pair_res.ensure(P * sizeof(PairRes) + 64));
    CU(b->line_len.ensure(P * 4 + 64));
    CU(b->line_off.ensure((P + 1) * 8 + 64));
    CU(b->out_idx.ensure((P + 1) * 8 + 64));
    CU(b->plans.ensure((P / LIFT_THREADS + 2) * sizeof(LiftPlan)));
    const size_t ln_blocks = P / (size_t)SER_LINES + 4;  // k_emit looks back over blocks of SER_LINES pairs (k_scan_lines needs fewer)
    CU(b->ln_state.ensure(ln_blocks * 4)); CU(b->ln_agg.ensure(ln_blocks * 16)); CU(b->ln_pre.ensure(ln_blocks * 16));
    CU(cudaMemsetAsync(b->ln_state.p, 0, ln_blocks * 4, s));
    WinView win{};
    win.from_record = 1u;  // a row's id is its record's: empty, or the "_TO.." suffix of the indel strip
    rc = lift_tail(ctx, b, win, RB_POLICY_RIGHTMOST, TAIL_TRIM, want, stats != nullptr, P, n_ops, nullptr);
    if (rc != RB_OK) return rc;
    return rb_batch_download_lift(ctx, b, want, out, stats);
}


int rb_trim_paf(rb_ctx* ctx, const rb_records* recs, int match_score, int diff_score, int indel_score, int remove_contained, int policy,
                uint32_t want, rb_lift_out* out, rb_stats_out* stats) {
    if (!ctx) return RB_ERR_NO_DEVICE;
    if (!out || !recs) return fail(ctx, RB_ERR_BAD_ARG, "recs / out is null");
    int rc = rb_trim_paf_begin(ctx, recs, match_score, diff_score, indel_score, policy);
    if (rc != RB_OK) return rc;
    rb_batch* b = ctx->scratch;
    const uint64_t n = b->n_rec;
    for (uint64_t it = 0;; it++) {  // batches of 8 rounds; rounds after convergence are no-ops on the device
        uint32_t done = 0;
        rc = trim_rounds(ctx, b, 8, true, nullptr, &done);
        if (rc != RB_OK) return rc;
        if (done) break;
        if (it > n * n / 8 + 8) { b->trim_ready = false; return fail(ctx, RB_ERR_UNSUPPORTED, "trim rounds do not converge"); }
    }
    return rb_trim_paf_end(ctx, remove_contained, want, out, stats);
}

int rb_stats(rb_ctx* ctx, const rb_records* recs, rb_stats_out* stats) {
    if (!ctx) return RB_ERR_NO_DEVICE;
    if (!stats) return fail(ctx, RB_ERR_BAD_ARG, "stats is null");
    cudaSetDevice(ctx->device);
    if (!ctx->peers.empty()) {
        const int mrc = stats_multi(ctx, recs, stats);
        if (mrc != 1) return mrc;
    }
    if (!ctx->scratch) ctx->scratch = new rb_batch();
    int rc = upload_into(ctx, ctx->scratch, recs, nullptr);
    if (rc != RB_OK) return rc;
    rc = rb_batch_stats(ctx, ctx->scratch, nullptr);
    if (rc != RB_OK) return rc;
    return rb_batch_download_stats(ctx, ctx->scratch, stats);
}

}  // extern "C"
