// rb_kernels.cuh — launchers of the sm_100a kernels (definitions in rb_kernels.cu).
#pragma once
#include <cuda_runtime.h>

#include "lift_core.cuh"
#include "rb_common.cuh"
#include "trim_core.cuh"

namespace rb {

#ifndef RB_TOK_THREADS
#define RB_TOK_THREADS 256
#endif
constexpr int TOK_THREADS = RB_TOK_THREADS;
#ifndef RB_TOK_EARLY_PUBLISH
#define RB_TOK_EARLY_PUBLISH 1  // k_tokenise: op count published before the decode, look-back walked after it (0: the round-1 order)
#endif
constexpr int TOK_TILE = TOK_THREADS * 16;  // text bytes per tokeniser tile
constexpr int TEXT_FRONT_PAD = 16;          // bytes of 0xFF in front of the text (look-behind halo of tile 0)
#ifndef RB_SMP_THREADS
#define RB_SMP_THREADS 256
#endif
constexpr int SMP_THREADS = RB_SMP_THREADS;
constexpr int SMP_OPS = SMP_THREADS * (int)SAMPLE;  // ops per sample-scan block
constexpr int SL_WCAP = 2048;                // window boundaries of one block staged in shared memory (each of starts / ends)
// tuning knobs (overridable with -D for sweeps on the GPU box, see tools/sweep.sh)
#ifndef RB_LIFT_THREADS
#define RB_LIFT_THREADS 128
#endif
#ifndef RB_LIFT_CCAP
#define RB_LIFT_CCAP 96
#endif
#ifndef RB_LIFT_MINB
#define RB_LIFT_MINB 6
#endif
#ifndef RB_LIFT_STAGE_SMP
#define RB_LIFT_STAGE_SMP 1  // 0: the samples of a k_lift block stay in global memory (L1/L2), only its ops are staged
#endif
#ifndef RB_LIFT_CHAIN
#define RB_LIFT_CHAIN 1  // 1: on tiling windows a pair's start boundary is derived from its left neighbour's end boundary
#endif
#ifndef RB_SMP2_LB2
#define RB_SMP2_LB2 0  // k_samples2: 1 = look-back over self-validating 128-bit slots, one L2 trip per round and no fences, instead of
                       // flag -> fence -> payload.  Parity-clean, measured: 0.309 against 0.319 ms at C4, 1.97 against 1.86 ms at
                       // 8 haplotypes x 10 kb — the round is dominated by the 13-word ordered reduction, not by the two trips
#endif
#ifndef RB_SMP_MINB
#define RB_SMP_MINB 3
#endif
#ifndef RB_EMIT_MINB
#define RB_EMIT_MINB 6
#endif
#ifndef RB_EMIT_STAGE_TEXT
#define RB_EMIT_STAGE_TEXT 0  // 1: k_emit FAST blocks of canonical records stage the text span of their rows in place of the op words and
                              // copy the untouched ops shared -> shared instead of formatting them.  Parity-clean, measured at C4:
                              // 0.938 / 0.961 against 0.955 ms — the ragged byte heads and tails of ~40-byte runs cost what the
                              // formatter's divisions did
#endif
#ifndef RB_EMIT_DIRECT
#define RB_EMIT_DIRECT 1  // k_emit: blocks whose rows are mostly long verbatim runs copy those text -> output directly (0: through the line buffer)
#endif
#ifndef RB_EMIT_MID_TEXT
#define RB_EMIT_MID_TEXT 0  // k_emit FAST blocks: short runs of untouched ops are copied from the input text (0: formatted from the op words)
#endif
constexpr int LIFT_THREADS = RB_LIFT_THREADS;  // pairs per k_lift block
constexpr int LIFT_CCAP = RB_LIFT_CCAP;        // 32-op chunks of one record a k_lift block stages in shared memory
constexpr int LNS_THREADS = 256;
constexpr int SER_LINES = 128;              // lines per serialiser block
#ifndef RB_SER_CAP_KB
#define RB_SER_CAP_KB 26
#endif
constexpr int SER_CAP = RB_SER_CAP_KB * 1024;  // smem bytes for composing a line group

struct ScanPayload {  // look-back payload of the segmented sample scan: 64 B, 16-byte aligned
    Ctr c;
    uint32_t flag;    // a record head lies inside the span this aggregate covers
    uint32_t pad[3];
};

struct WinView {
    const uint64_t* st;
    const uint64_t* en;
    const uint64_t* en_pm;     // prefix max of en within the contig (== en when en is monotone)
    const uint64_t* ids_off;
    const uint8_t* ids;
    const uint32_t* bed_row;
    const uint32_t* cont_lo;   // per name id: window range of that contig
    const uint32_t* cont_hi;
    const uint32_t* pair_win;  // general path: explicit window per pair (nullptr on the fast path)
    uint32_t general;          // 1: arrays are in BED file order (grouped by contig), pairs come from the brute-force join
    uint32_t from_record;      // 1: `rb break-paf` — the windows were generated from each record's own large indels
                               //    (liftover.rs:182-226): a row's id is its record's id, empty windows are skipped
};

struct RecInput {  // device copies of rb_records columns
    const uint64_t* cigar_off;
    const uint64_t *q_len, *q_st, *q_en, *t_len, *t_st, *t_en, *mapq;
    const uint8_t* strand;
    const uint32_t *q_id, *t_id;
    const uint64_t* names_off;
    const uint8_t* names;
    uint32_t n_rec;
    uint32_t no_text;  // 1: the op words no longer spell the input text (query/target swapped): never copy ops from it
};

struct StatsDev {  // device SoA of rb_stats_out
    uint32_t *equal, *diff, *ins, *del, *ins_ev, *del_ev, *matches;
    float *id_m, *id_e, *id_a;
};
struct NumDev {  // device SoA of the numeric mirror
    uint64_t *q_st, *q_en, *t_st, *t_en, *nmatch, *aln_len;
    uint32_t *rec_idx, *win_idx;
};

// error slots (device, u64 each, initialised to ~0): min over (key << 8 | code)
struct ErrSlots {
    unsigned long long* tok;  // key = byte position in the text
    unsigned long long* rec;  // key = record index
};

int init_kernel_attrs();  // once per device: dynamic shared-memory limits of the kernels that need more than the default
void launch_add_u64(uint64_t* p, uint64_t n, uint64_t delta, cudaStream_t s);
void launch_tokenise(const uint8_t* text, uint64_t n_tiles, uint32_t* ops, unsigned long long* tile_state,
                     unsigned int* ticket, ErrSlots err, uint32_t* misc_flags, cudaStream_t s);
// tokeniser + sampled segmented scan in one pass (k_rec_heads + k_tok_scan): what launch_tokenise + launch_scan_lift(false) produce,
// without reading the op words back.  tile_first (u32 per tile) must be filled with 0xFF, seg_state (u32 per tile) zeroed.
void launch_tok_scan(const uint8_t* text, uint64_t n_tiles, const uint64_t* cigar_off, uint32_t n_rec, uint32_t* ops,
                     unsigned long long* tile_state, unsigned int* ticket, ErrSlots err, uint32_t* misc_flags, uint32_t* tile_first,
                     uint64_t* head_pos, Ctr* samples, uint32_t* seg_state, ScanPayload* seg_agg, ScanPayload* seg_pre, cudaStream_t s);
void launch_rec_ops(const uint8_t* text, const uint64_t* cigar_off, uint32_t n_rec, const unsigned long long* tile_state,
                    uint64_t* op_off, uint32_t* heads, ErrSlots err, cudaStream_t s);
// fast-path (sorted BED, right-most policy) arguments of k_scan_lift: where the half results go
struct LiftArgs {
    const RecInfo* recs;       // after k_rec_prep mode 1
    const uint64_t* op_off;
    uint32_t n_rec;
    const uint32_t* rec_rank;  // record -> position in emission order
    const uint64_t* pair_off;  // emission-ordered pair offsets
    const uint64_t* w_st;
    const uint64_t* w_en;
    HalfS* hs;
    HalfE* he;
};
// sampled segmented scan; lift == true additionally resolves the window boundaries of every record (fast path)
void launch_scan_lift(bool lift, const uint32_t* ops, const uint64_t* n_ops_dev, uint64_t n_ops_bound, const uint32_t* heads,
                      Ctr* samples, uint32_t* blk_state, ScanPayload* blk_agg, ScanPayload* blk_pre, unsigned int* ticket,
                      LiftArgs la, cudaStream_t s, bool no_subs = false);  // no_subs: absolute samples only (wide windows)
void launch_combine(uint64_t n_pairs, const uint64_t* pair_off, const uint32_t* rec_order, uint32_t n_rec, const RecInfo* recs,
                    const uint32_t* ops, WinView win, const uint64_t* names_off, const HalfS* hs, const HalfE* he, PairRes* res,
                    uint32_t* line_len, ErrSlots err, cudaStream_t s);
// liftover --qbed (paf.rs:1050-1094 paf_swap_query_and_target): I <-> D in every op, op order reversed on '-' records
void launch_invert_ops(uint32_t* ops, const uint64_t* op_off, uint32_t n_rec, const uint8_t* strand, uint64_t n_ops_bound,
                       cudaStream_t s);
void launch_check_clips(const uint32_t* ops, const uint64_t* op_off, uint32_t n_rec, ErrSlots err, cudaStream_t s);
// mode 0: rb stats (after the scan) ; mode 1: liftover phase A (strip + join, before the scan) ; mode 2: phase B (after the scan)
void launch_rec_prep(int mode, RecInput in, const uint64_t* op_off, const uint32_t* ops, const Ctr* samples, WinView win,
                     RecInfo* recs, uint32_t* pair_cnt, StatsDev st, ErrSlots err, cudaStream_t s);
void launch_pair_scan(const uint32_t* pair_cnt, const uint32_t* rec_order, uint32_t n_rec, uint64_t* pair_off, cudaStream_t s);
// per block of LIFT_THREADS consecutive pairs (emission order): its record, if it has only one, and the run of chunks it touches
enum : uint32_t { PLAN_UNIFORM = 1u,  // every pair of the block belongs to one record
                  PLAN_FAST = 2u };   // ... and k_emit lifts the block itself, out of shared memory (k_lift skips it)
struct LiftPlan {
    uint32_t k0;        // emission rank of the record of the block's first pair
    uint32_t uniform;   // PLAN_* flags
    uint64_t c_lo, c_hi;  // chunks of the first start boundary / last end boundary (~0: not applicable)
};
// rb invert: the CIGAR bytes of the whole-record rows (after launch_serialise)
void launch_whole_text(const uint32_t* ops, const uint64_t* op_off, uint32_t n_rec, const RecInfo* recs, const Ctr* samples,
                       const uint64_t* line_off, uint8_t* out_text, uint64_t n_ops_bound, cudaStream_t s);
// rb invert: one whole-record row per record (fills PairRes, line lengths, pair list, plans)
void launch_whole_rows(uint32_t n_rec, const RecInfo* recs, PairRes* res, uint32_t* line_len, uint64_t* pair_off, LiftPlan* plans,
                       cudaStream_t s);
// mark_fast: blocks k_emit can lift itself get PLAN_FAST (the caller then runs k_lift with skip_fast and k_emit)
void launch_lift_plan(uint64_t n_pairs, const uint64_t* pair_off, const uint32_t* rec_order, uint32_t n_rec, const RecInfo* recs,
                      const Ctr* samples, WinView win, LiftPlan* plans, cudaStream_t s, bool mark_fast = false);
void launch_lift(uint64_t n_pairs, const uint64_t* pair_off, const uint32_t* rec_order, uint32_t n_rec, const RecInfo* recs,
                 const uint32_t* ops, const Ctr* samples, WinView win, const uint64_t* names_off, int policy, const LiftPlan* plans,
                 PairRes* res, uint32_t* line_len, ErrSlots err, cudaStream_t s, bool skip_fast = false, bool wide = false);
                 // wide: the call's windows are wide (no block fits the staging area): the variant without staging arrays, 8 blocks / SM
void launch_scan_lines(const uint32_t* line_len, uint64_t n, uint64_t* line_off, uint64_t* out_idx, uint32_t* blk_state,
                       ulonglong2* blk_agg, ulonglong2* blk_pre, unsigned int* ticket, cudaStream_t s);
void launch_serialise(uint64_t n_pairs, const uint64_t* pair_off, const uint32_t* rec_order, uint32_t n_rec, const RecInfo* recs,
                      const uint32_t* ops, const uint8_t* text, WinView win, const uint64_t* names_off, const uint8_t* names,
                      const LiftPlan* plans, const PairRes* res, const uint64_t* line_off, const uint64_t* out_idx, uint8_t* out_text,
                      uint64_t* out_line_off, NumDev num, StatsDev st, uint64_t byte_base, uint32_t rec_base, const uint32_t* orig_idx,
                      uint32_t group, uint32_t defer_big, cudaStream_t s, const uint32_t* only_flagged = nullptr);
// lift (FAST blocks) + line scan + serialiser in one pass (k_emit): totals[0..3] = bytes, rows, overflow flag, blocks left to
// k_serialise; lb_bytes / lb_rows = one zeroed 64-bit look-back word per block of SER_LINES pairs
void launch_emit(uint64_t n_pairs, const uint64_t* pair_off, const uint32_t* rec_order, uint32_t n_rec, const RecInfo* recs,
                 const uint32_t* ops, const Ctr* samples, const uint8_t* text, WinView win, const uint64_t* names_off, const uint8_t* names,
                 const LiftPlan* plans, PairRes* res, const uint32_t* line_len, uint64_t* line_off, uint64_t* out_idx,
                 uint32_t* blk_flags, uint8_t* out_text, uint64_t cap_text, uint64_t* out_line_off, NumDev num, StatsDev st,
                 uint64_t byte_base, uint32_t rec_base, const uint32_t* orig_idx, unsigned long long* lb_bytes,
                 unsigned long long* lb_rows, unsigned int* ticket, unsigned long long* totals, ErrSlots err, cudaStream_t s,
                 bool stats_text = false, bool wide = false);  // wide: no block is PLAN_FAST (the plan was made without mark_fast): less smem, more L1
// few, long rows: the long verbatim runs of input text that k_serialise (defer_big = 1) left out, spread over the grid
void launch_copy_mid(uint64_t n_pairs, const uint64_t* pair_off, const uint32_t* rec_order, uint32_t n_rec, const RecInfo* recs,
                     const PairRes* res, const uint64_t* line_off, const uint8_t* text, uint8_t* out_text, uint32_t seg_y, cudaStream_t s);
struct PublishArgs {  // up to 8 device scalars (u32 or u64) -> slots of a mapped pinned u64 array
    const void* src[8];
    uint8_t slot[8];
    uint8_t wide[8];
    int n;
    unsigned long long* dst;
};
void launch_publish(const PublishArgs& a, cudaStream_t s);
// `rb break-paf` (liftover.rs:182-226, main.rs:271-281): the windows of a record are the target intervals between its
// insertions / deletions longer than max_size.  count pass (per 32-op chunk) -> exclusive scan -> fill pass -> per-record
// window ranges and the window table itself; everything downstream is the liftover path.
void launch_break_scan(bool fill, const uint32_t* ops, const uint64_t* n_ops_dev, uint64_t n_ops_bound, const uint32_t* heads,
                       const Ctr* samples, const uint64_t* op_off, uint32_t n_rec, const RecInfo* recs, uint32_t max_size,
                       uint32_t* cnt, const uint64_t* bp_off, uint64_t* bp_end, uint64_t* bp_next, uint64_t* rec_bp0, uint64_t* rec_bp1,
                       cudaStream_t s);
void launch_break_recs(uint32_t n_rec, RecInfo* recs, const uint64_t* rec_bp0, const uint64_t* rec_bp1, const uint64_t* bp_end,
                       const uint64_t* bp_next, uint64_t* w_st, uint64_t* w_en, uint32_t* pair_cnt, cudaStream_t s);
// `rb trim-paf` (trim_overlap.rs:36-86, paf.rs:210-305; kernels in trim_kernels.cu).
void launch_trim_scan(const uint32_t* ops, const RecInfo* recs, uint32_t n_rec, TrimScores sc, uint32_t* qp, uint32_t* ap, long long* wp,
                      TrimView* views, int policy, cudaStream_t s);
// n_rounds rounds of select -> pairs -> cut -> round_end, enqueued back to back (rounds after convergence are no-ops).
// grp_off = n_groups + 1 record offsets of the query names in the name-sorted set; sel = 24 B, keys = 8 B per group;
// info = 32 B {waiting, done, rounds, status, err_l, err_r, last_waiting, -}, zeroed by the caller before the first round;
// auto_done: a round that leaves nothing waiting sets `done` (otherwise the caller decides when to stop).
// policy == POLICY_EARLY_EXIT: the score prefixes (wp) of the records cut in a round are re-scanned for their new views (k_trim_rescan)
void launch_trim_rounds(int n_rounds, bool auto_done, const uint32_t* grp_off, uint32_t n_groups, const uint32_t* ops, const RecInfo* recs, const uint32_t* qp,
                        long long* wp, const uint32_t* ap, int policy, TrimScores sc, unsigned long long max_score, TrimView* views,
                        uint8_t* contained, void* sel, unsigned long long* keys, void* info, cudaStream_t s);
void launch_trim_rows(uint32_t n_rec, const RecInfo* recs, const TrimView* views, const uint32_t* ops, const Ctr* samples,
                      const uint8_t* dropped, PairRes* res, uint32_t* line_len, uint64_t* pair_off, LiftPlan* plans, cudaStream_t s);
// BGZF inflate on the device (inflate_kernels.cu): one table row per block, one thread per block
struct BgzfBlock {
    uint64_t cdata;    // offset of the block's raw DEFLATE payload in the compressed buffer
    uint64_t out_off;  // where its bytes go in the inflated text
    uint32_t clen, out_len, crc, pad;  // payload bytes, ISIZE and CRC-32 of the trailer
};
void launch_inflate_bgzf(const uint8_t* comp, const BgzfBlock* blk, uint32_t n_blk, uint8_t* out, unsigned long long* err, cudaStream_t s);
// PAF text -> a resident batch (paf_parse_kernels.cu; the rules are paf_parse_core.cuh's).  Per-line columns of k_paf_fields:
struct PafLineCols {
    uint8_t* state;      // paf_parse_core.cuh LS_*
    uint64_t* keep;      // 1 for a kept line (scan input: record index)
    uint64_t* cg_len;    // cg payload bytes of a kept line (scan input: cigar_off)
    uint64_t* name_len;  // q + t name bytes of a kept line (scan input: name bytes)
    uint64_t* v;         // 7 x n_lines: q_len q_st q_en t_len t_st t_en mapq
    uint8_t* strand;
    uint64_t *qn_off, *tn_off, *cg_off;
    uint32_t* qn_len;
};
uint64_t paf_chunks(uint64_t n);      // k_paf_lines_* blocks (64 KiB of text each): entries of chunk_cnt
uint64_t paf_tiles(uint64_t n);       // 4 KiB whitespace tiles: entries of tile_ws
uint64_t paf_scan_parts(uint64_t n);  // u64 per scanned column of the scan's block sums
void launch_paf_lines_count(const uint8_t* text, uint64_t n, uint64_t* chunk_cnt, uint8_t* tile_ws, uint32_t* last_byte, cudaStream_t s);
void launch_paf_lines_fill(const uint8_t* text, uint64_t n, const uint64_t* chunk_off, uint64_t* line_start, cudaStream_t s);
// exclusive scans of nv <= 3 columns: out[v][0 .. n) and the total at out[v][n]; part = nv * paf_scan_parts(n) u64
void launch_paf_scan(int nv, const uint64_t* const* in, uint64_t* const* out, uint64_t n, uint64_t* part, cudaStream_t s);
void launch_paf_fields(const uint8_t* text, const uint64_t* line_start, uint64_t n_lines, const uint8_t* tile_ws, PafLineCols L,
                       unsigned long long* first_panic, cudaStream_t s);
void launch_paf_pack(const uint8_t* text, uint64_t n_lines, PafLineCols L, const uint64_t* rec_idx, const uint64_t* cg_pos,
                     const uint64_t* name_pos, uint32_t n_rec, uint64_t* cols64, uint8_t* strand, uint64_t* cigar_off, uint32_t* rec_line,
                     uint8_t* names, uint64_t* rec_name_off, uint32_t* rec_qlen, cudaStream_t s);
void launch_paf_copy_cg(const uint8_t* text, uint32_t n_rec, const uint64_t* cigar_off, const uint32_t* rec_line, const uint64_t* cg_off,
                        uint64_t cg_bytes, uint8_t* dst, cudaStream_t s);
// rb_liftover_text on several devices (text_multi_kernels.cu).  *first = min(*first, offset of the first '\n' in text[0, n));
// runs = 4 u64 tables of n_ranks entries (row start, row end, byte start, byte end of each contig's rows), zeroed by the caller;
// a row's contig rank is rank_of[t_id[rec_idx - rec_base]]; rebase: line_off[row] += delta[its rank]
void launch_first_newline(const uint8_t* text, uint64_t n, unsigned long long* first, cudaStream_t s);
void launch_contig_runs(uint64_t n, const uint32_t* rec_idx, uint32_t rec_base, const uint32_t* t_id, const uint32_t* rank_of,
                        const uint64_t* line_off, uint64_t out_bytes, uint64_t* runs, uint32_t n_ranks, cudaStream_t s);
void launch_rebase_runs(uint64_t n, const uint32_t* rec_idx, uint32_t rec_base, const uint32_t* t_id, const uint32_t* rank_of,
                        const uint64_t* delta, uint64_t* line_off, cudaStream_t s);
// BED text -> the window tables of a batch (bed_parse_kernels.cu; the rules are bed_parse_core.cuh's).  Per-line columns:
struct BedLineCols {
    const uint64_t* line_start;
    uint64_t *n_fields, *st, *en, *name_len, *id_off, *id_len;
    uint8_t* nums_ok;
    uint64_t *comment, *parses, *kept;  // 0 / 1 (scan inputs: comment count, bed_row, window index)
    uint32_t* tid;                      // name id of a kept line, ~0 otherwise
};
struct BedRows {  // kept rows in file order
    uint32_t *tid, *row;
    uint64_t *st, *en, *line;
};
void launch_bed_lines_count(const uint8_t* text, uint64_t n, uint64_t* chunk_cnt, cudaStream_t s);
void launch_bed_lines_fill(const uint8_t* text, uint64_t n, const uint64_t* chunk_off, uint64_t* line_start, cudaStream_t s);
uint64_t bed_name_slots(uint32_t n_names);  // u32 slots of the device name table (a power of two)
void launch_bed_names(const uint8_t* names, const uint64_t* names_off, uint32_t n_names, uint32_t* table, uint64_t slots, cudaStream_t s);
void launch_bed_fields(const uint8_t* text, uint64_t n, uint64_t n_lines, BedLineCols L, unsigned long long* first_row, cudaStream_t s);
void launch_bed_judge(const uint8_t* text, uint64_t n_lines, BedLineCols L, const unsigned long long* first_row, const uint8_t* names,
                      const uint64_t* names_off, const uint32_t* table, uint64_t slots, unsigned long long* nf0_out, cudaStream_t s);
void launch_bed_compact(uint64_t n_lines, BedLineCols L, const uint64_t* row_idx, const uint64_t* win_idx, BedRows R, unsigned long long* max_st,
                        cudaStream_t s);
void launch_bed_order(BedRows R, uint32_t n, uint32_t* unsorted, cudaStream_t s);  // *unsorted |= 1 if R is not in (t_id, st) order
size_t bed_sort_scratch(uint32_t n);
cudaError_t launch_bed_sort(BedRows R, uint32_t n, int tb, int sb, bool by_tid_only, void* scratch, size_t scratch_bytes, uint32_t* perm,
                            cudaStream_t s);
// rows perm[k] (perm nullptr: k) of R -> row k of the w_* tables; id_off / id_len (nullable) = the field-4 span of that row's line
void launch_bed_gather(BedRows R, uint32_t n, const uint32_t* perm, const uint64_t* line_id_off, const uint64_t* line_id_len, uint32_t* w_tid,
                       uint64_t* w_st, uint64_t* w_en, uint32_t* w_row, uint64_t* id_off, uint64_t* id_len, cudaStream_t s);
void launch_bed_cont(const uint32_t* w_tid, uint32_t n, uint32_t* cont_lo, uint32_t* cont_hi, cudaStream_t s);
void launch_win_check(const uint32_t* t_id, const uint64_t* st, const uint64_t* en, const uint32_t* row, uint32_t n_win,
                      uint32_t n_names, uint32_t* flags, cudaStream_t s);
// general path (unsorted / nested BED rows): the reference's cartesian product + overlap filter (liftover.rs:123-127)
void launch_pair_count_bf(const RecInfo* recs, uint32_t n_rec, WinView win, uint32_t* pair_cnt, cudaStream_t s);
void launch_pair_fill_bf(const RecInfo* recs, const uint32_t* rec_rank, uint32_t n_rec, WinView win,
                         const uint64_t* pair_off, uint32_t* pair_win, cudaStream_t s);

}  // namespace rb
