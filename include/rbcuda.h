/* rbcuda.h — C ABI of the B200 (sm_100a) PAF liftover + stats path.
 *
 * The reference (rustybam v0.1.33) has no plugin/FFI interface; the seams this library plugs
 * into are two library calls made by its driver (file:line into the reference tree):
 *
 *   src/main.rs:197    liftover::trim_paf_by_rgns(&[bed::Region], &[paf::PafRecord], invert) -> Vec<PafRecord>
 *                      (src/liftover.rs:134-167; printed with Display, src/paf.rs:923-943, at main.rs:210-212)
 *                      ==> rb_liftover()
 *   src/main.rs:53-56  bamstats::stats_from_paf(PafRecord) -> Stats  (src/bamstats.rs:91-154)
 *                      ==> rb_stats()          (and, fused per lifted row, the rb_stats_out of rb_liftover)
 *
 * A Rust host (INTEGRATION.md shows the `ffi.rs` binding) keeps text / bgzip I/O and the
 * src/paf.rs record API, packs the cg:Z: payloads and the numeric columns into the SoA buffers
 * below (pinned host memory recommended, any host memory accepted) and gets back the bytes
 * `rb liftover` would print plus the counters `rb stats --paf` would print for those rows.
 *
 * Conventions
 *   - plain pointers and sizes only; no C++/torch types; no exceptions cross the boundary
 *   - inputs are caller-owned and only read; outputs are library-owned pinned host memory that
 *     stays valid until the matching rb_free_* call (or rb_ctx_destroy)
 *   - one calling thread per rb_ctx; contexts are independent (no global state)
 *   - return value: RB_OK (0) or a negative rb_status; rb_last_error() gives the text
 *   - NO CPU FALLBACK: without a usable sm_100 device every entry point fails with
 *     RB_ERR_NO_DEVICE
 *   - where the reference would panic (process exit status 101) the call fails with one of the
 *     RB_ERR_REF_* codes and produces no output
 */
#ifndef RBCUDA_H
#define RBCUDA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct rb_ctx rb_ctx;
typedef struct rb_batch rb_batch;

typedef enum rb_status {
    RB_OK = 0,
    RB_ERR_NO_DEVICE = -1,       /* no CUDA device with compute capability 10.x */
    RB_ERR_CUDA = -2,            /* CUDA runtime error (text in rb_last_error) */
    RB_ERR_BAD_ARG = -3,         /* null pointer, unsorted windows, id out of range, ... */
    RB_ERR_REF_CIGAR_PARSE = -4, /* rust-htslib CigarString::try_from fails -> `expect` panic, paf.rs:399 */
    RB_ERR_REF_INTEGRITY = -5,   /* check_integrity().unwrap() panics, paf.rs:70 */
    RB_ERR_REF_STRIP = -6,       /* remove_trailing_indels panics: empty CIGAR, leading deletion, all-indel; paf.rs:663,782 */
    RB_ERR_REF_INDEX = -7,       /* "Problem getting index in cigar", liftover.rs:31-49 */
    RB_ERR_UNSUPPORTED = -8,     /* outside this path's documented domain: op length >= 2^28, per-record sums >= 2^32 */
    RB_ERR_OOM = -9,
    RB_ERR_REF_PAF_PARSE = -10   /* PafRecord::new asserts: a line of < 12 columns, or an extra token that is not a tag (paf.rs:381,387-389) */
} rb_status;

/* binary_search duplicate policy of the reference's toolchain (SURVEY.md Q2): which of several
 * equal target positions `core::slice::binary_search` returns at paf.rs:542. */
#define RB_POLICY_RIGHTMOST 0  /* Rust < 1.52 and >= 1.82 (default) */
#define RB_POLICY_EARLY_EXIT 1 /* Rust 1.52 ..= 1.81 */

/* what rb_liftover / rb_batch_download_lift materialise on the host */
#define RB_WANT_TEXT 1u    /* paf_text + line_off */
#define RB_WANT_NUMERIC 2u /* q_st .. aln_len, rec_idx, win_idx */
/* rb_liftover only: `liftover --qbed` — the windows are in QUERY coordinates; every record swaps query and target
 * (I <-> D, op order reversed on '-' strands; paf.rs:1050-1094) before it is lifted, and is printed swapped */
#define RB_WANT_QBED 4u
/* rb_liftover / rb_batch_liftover only: paf_text + line_off hold, instead of the PAF rows, the rows `rb stats --paf` prints for
 * them (bamstats.rs:239-270; the header line, main.rs:51, is the host's) — i.e. the final output of
 * `rb liftover --bed .. | rb stats --paf`, formatted on the device (shortest-round-trip f32 digits included): a third of the
 * bytes of the PAF rows cross PCIe.  Not together with RB_WANT_TEXT. */
#define RB_WANT_STATS_TEXT 8u

/* PAF records, SoA, n_rec rows in FILE order (src/paf.rs:346-368 PafRecord, columns 1-12 + cg:Z:). */
typedef struct rb_records {
    uint32_t n_rec;
    const uint8_t* cigar;      /* concatenated cg:Z: payload bytes, no separators */
    uint64_t cigar_nbytes;
    const uint64_t* cigar_off; /* n_rec + 1 offsets into cigar */
    const uint64_t* q_len;
    const uint64_t* q_st;
    const uint64_t* q_en;
    const uint64_t* t_len;
    const uint64_t* t_st;
    const uint64_t* t_en;
    const uint64_t* mapq;
    const uint8_t* strand;     /* '+' or '-' */
    const uint32_t* q_id;      /* index into the name table */
    const uint32_t* t_id;      /* index into the name table; equal t_id <=> equal t_name */
    const uint8_t* names;      /* concatenated name bytes */
    const uint64_t* names_off; /* n_names + 1 */
    uint32_t n_names;
} rb_records;

/* BED windows (src/bed.rs:14-21 Region), SoA, sorted by (t_id, st) — stable, so equal keys keep
 * BED file order.  bed_row = row index in the BED file: it defines the emission order within a
 * record (liftover.rs:123-126) and is echoed in rb_lift_out.win_idx.  ids = Region.id per window
 * (BED column 4, else "{chrom}:{st+1}-{en}", bed.rs:150-153), parallel to st/en.  For a BED file
 * without a 4th column pass ids = ids_off = NULL: the library formats the default id on the device
 * (no per-window string ever exists on the host or crosses PCIe). */
typedef struct rb_windows {
    uint32_t n_win;
    const uint32_t* t_id;
    const uint64_t* st;
    const uint64_t* en;
    const uint32_t* bed_row;
    const uint8_t* ids;      /* nullable together with ids_off */
    const uint64_t* ids_off; /* n_win + 1 */
} rb_windows;

/* Lifted rows in the reference's emission order (`rb -t 1 liftover`): contigs by first appearance
 * of t_name among the records, record-major, BED-row-minor (liftover.rs:151-164). */
typedef struct rb_lift_out {
    uint64_t n_out;
    uint8_t* paf_text;    /* exactly the bytes `rb liftover` prints on stdout ('\n' after every row) */
    uint64_t paf_nbytes;
    uint64_t* line_off;   /* n_out + 1 */
    uint64_t* q_st;       /* numeric mirror of the rows (RB_WANT_NUMERIC) */
    uint64_t* q_en;
    uint64_t* t_st;
    uint64_t* t_en;
    uint64_t* nmatch;
    uint64_t* aln_len;
    uint32_t* rec_idx;    /* input record of each row */
    uint32_t* win_idx;    /* bed_row of each row */
    uint64_t n_pairs;     /* overlapping (window, record) pairs examined (>= n_out; Q7 drops) */
    void* _owner;
} rb_lift_out;

/* bamstats.rs:15-36 Stats counters (u32, like the reference) and the three f32 identities. */
typedef struct rb_stats_out {
    uint64_t n;
    uint32_t* equal;
    uint32_t* diff;
    uint32_t* ins;
    uint32_t* del;
    uint32_t* ins_events;
    uint32_t* del_events;
    uint32_t* matches;
    float* id_by_matches;
    float* id_by_events;
    float* id_by_all;
    void* _owner;
} rb_stats_out;

typedef struct rb_summary {
    uint64_t n_ops;       /* CIGAR ops tokenised */
    uint64_t n_pairs;
    uint64_t n_out;
    uint64_t out_bytes;   /* bytes of PAF text produced */
    uint64_t cigar_bytes; /* bytes of CIGAR text consumed */
} rb_summary;

typedef struct rb_kernel_time {
    char name[32];
    uint64_t launches;
    double ms; /* CUDA-event time summed over launches since the last reset */
} rb_kernel_time;

/* ---- context ---- */
rb_ctx* rb_ctx_create(const int* device_ids, int n_devices, int* status);
void rb_ctx_destroy(rb_ctx* ctx);
const char* rb_last_error(const rb_ctx* ctx);
/* launch everything on the caller's stream (a cudaStream_t, e.g. torch's current stream); NULL = own stream */
int rb_ctx_set_stream(rb_ctx* ctx, void* cuda_stream);
/* how rb_liftover resolves the window boundaries (results are identical; see DESIGN.md §4):
 *   RB_LIFT_SEARCH  one search per (window, record) pair over the sampled prefix sums (default)
 *   RB_LIFT_STREAM  sorted BED rows + right-most policy: boundaries are resolved while the prefix scan streams
 *                   over the ops; other inputs silently use RB_LIFT_SEARCH */
#define RB_LIFT_SEARCH 0
#define RB_LIFT_STREAM 1
int rb_ctx_set_lift_mode(rb_ctx* ctx, int mode);
/* rb_liftover cuts a call whose records are in emission order (PAF grouped by target) into up to 8 slices of
 * consecutive records, each of at least `min_slice_bytes` of CIGAR text; the device->host copies of a slice overlap the
 * upload and the kernels of the following ones.  Default 16 MiB; 0 = never slice.  Results do not depend on it. */
int rb_ctx_set_slicing(rb_ctx* ctx, uint64_t min_slice_bytes);
/* per-kernel CUDA-event timing (off by default; adds an event pair around every launch) */
int rb_ctx_set_profiling(rb_ctx* ctx, int on);
int rb_ctx_kernel_times(rb_ctx* ctx, rb_kernel_time* out, int cap, int reset); /* returns count */

/* ---- the drop-in calls: host buffers in, pinned host buffers out ---- */
/* replaces liftover::trim_paf_by_rgns + Display (+ stats_from_paf per emitted row when stats != NULL) */
int rb_liftover(rb_ctx* ctx, const rb_records* recs, const rb_windows* wins, int policy, uint32_t want,
                rb_lift_out* out, rb_stats_out* stats /* nullable */);
/* replaces the `for paf in records { stats_from_paf(paf) }` loop of `rb stats --paf` (main.rs:53-56) */
int rb_stats(rb_ctx* ctx, const rb_records* recs, rb_stats_out* stats);
/* replaces the loop of `rb break-paf --max-size N` (main.rs:271-281, liftover::break_paf_on_indels liftover.rs:182-226):
 * every record is cut at its insertions / deletions longer than max_size; rows in FILE order; win_idx = piece number
 * within the call; the id of a row is its record's id (empty, or the "_TO.." suffix of the indel strip) */
int rb_break_paf(rb_ctx* ctx, const rb_records* recs, uint32_t max_size, int policy, uint32_t want, rb_lift_out* out,
                 rb_stats_out* stats /* nullable */);
/* replaces the loop of `rb invert` (main.rs:176-182, paf::paf_swap_query_and_target paf.rs:1050-1094): one row per record in
 * FILE order — query and target columns swapped, I and D exchanged, the ops reversed on the '-' strand; nothing is stripped or
 * merged; nmatch / aln_len are the ones check_integrity infers from the CIGAR (paf.rs:825-857); id empty; win_idx = 0 */
int rb_invert(rb_ctx* ctx, const rb_records* recs, uint32_t want, rb_lift_out* out);
/* replaces `paf.overlapping_paf_recs(match, diff, indel, remove_contained)` + the print loop of `rb trim-paf` (main.rs:218-230;
 * paf.rs:210-305, trim_overlap.rs:36-86): records that overlap on the same query are cut at the split point that maximises
 * (score of the left record before it) + (score of the right record after it), largest overlap first, one pair per query name
 * and round until no pair is left.  One row per record, ordered by query name (stable, byte-wise — the reference's
 * sort_by_key); rec_idx = the caller's record index, win_idx = 0; untouched records are printed as they are (after the indel
 * strip), truncated ones re-collapsed.  Both search policies (paf.rs:564-574 is a binary_search over per-column query positions
 * that repeat on every deletion column): under RB_POLICY_EARLY_EXIT the score of a position in front of a deletion depends on the
 * record's current truncation, and the records cut in a round are scanned again on the device;
 * records must start and end on an M/=/X op after the strip.  Where a truncation leaves spans that disagree with the CIGAR the
 * reference panics (paf.rs:819-822) -> RB_ERR_REF_INTEGRITY. */
int rb_trim_paf(rb_ctx* ctx, const rb_records* recs, int match_score, int diff_score, int indel_score, int remove_contained, int policy,
                uint32_t want, rb_lift_out* out, rb_stats_out* stats /* nullable */);
/* The same in steps, for a record set that is spread over several GPUs BY QUERY NAME (records only ever interact with records
 * of their own query name, paf.rs:229-239).  The reference's decision to run another round is global — `if unseen > 0` counts
 * the waiting pairs of ALL names (paf.rs:283-285) — and a name's result depends on it: a record that was contained when its
 * name's last pair was cut can overlap the cut records partially afterwards, and is only trimmed if some OTHER name forces
 * one more round.  So every rank runs rb_trim_paf_round() in lockstep, the ranks OR their `waiting` flags (the one collective
 * of this sub-command: one integer per round) and stop together when nobody waits; rb_trim_paf_end() then returns the rank's
 * rows, and the name groups of all ranks concatenate in query-name order.  One rb_ctx per rank; begin .. end must not be
 * interleaved with other calls on the same context. */
int rb_trim_paf_begin(rb_ctx* ctx, const rb_records* recs, int match_score, int diff_score, int indel_score, int policy);
int rb_trim_paf_round(rb_ctx* ctx, int* waiting /* out: 1 if a pair of this rank had to wait for the next round */);
int rb_trim_paf_end(rb_ctx* ctx, int remove_contained, uint32_t want, rb_lift_out* out, rb_stats_out* stats /* nullable */);
void rb_free_lift_out(rb_ctx* ctx, rb_lift_out* out);
void rb_free_stats_out(rb_ctx* ctx, rb_stats_out* stats);

/* ---- resident batches: upload once, run the kernels with inputs already in HBM ---- */
rb_batch* rb_batch_upload(rb_ctx* ctx, const rb_records* recs, const rb_windows* wins /* nullable */, int* status);
/* `want`: which outputs the kernels materialise in HBM (RB_WANT_* bits); rb_batch_download_lift may ask for a subset */
int rb_batch_liftover(rb_ctx* ctx, rb_batch* b, int policy, uint32_t want, int with_stats, rb_summary* summary);
int rb_batch_stats(rb_ctx* ctx, rb_batch* b, rb_summary* summary);
/* break-paf on a batch uploaded without windows (rows in the batch's emission order) */
int rb_batch_break(rb_ctx* ctx, rb_batch* b, uint32_t max_size, int policy, uint32_t want, int with_stats, rb_summary* summary);
int rb_batch_download_lift(rb_ctx* ctx, rb_batch* b, uint32_t want, rb_lift_out* out, rb_stats_out* stats);
int rb_batch_download_stats(rb_ctx* ctx, rb_batch* b, rb_stats_out* stats);
void rb_batch_free(rb_ctx* ctx, rb_batch* b);

/* ---- PAF text parsed on the device (Paf::from_file, paf.rs:62-78,379-430, quirk for quirk as the host reader restates it) ---- */
typedef struct rb_paf_info {
    uint64_t text_bytes;  /* PAF text parsed (the inflated size for BGZF input) */
    uint64_t n_lines, skipped;
    uint32_t n_rec, n_names;
    const uint8_t* names; const uint64_t* names_off;  /* the batch's name table: ids by first appearance in file order, query name
                                                          before target name per record; library-owned, valid until rb_batch_free */
    uint64_t cigar_bytes;
} rb_paf_info;
/* PAF text, or BGZF bytes (recognised with rb_is_bgzf), -> a resident batch without windows; lines are split, tokenised and packed on
 * the device (the context's first device), only the name bytes of the records come back for interning.  Where the reference panics
 * the call fails: RB_ERR_REF_PAF_PARSE (< 12 columns, a bad tag), RB_ERR_REF_CIGAR_PARSE (a skipped line with a malformed cg tag);
 * rb_last_error names the 1-based line.  A plain (single-member) gzip file is refused with RB_ERR_BAD_ARG: inflate it first.
 * info is nullable. */
rb_batch* rb_batch_upload_paf(rb_ctx* ctx, const uint8_t* data, uint64_t nbytes, rb_paf_info* info, int* status);
/* windows for a batch that was uploaded without them (t_id = ids of that batch's name table); replaces any it had */
int rb_batch_set_windows(rb_ctx* ctx, rb_batch* b, const rb_windows* wins);
/* the batch's records as rb_records in library-owned pinned memory (CIGAR bytes only if with_cigar), valid until rb_batch_free or the
 * next rb_batch_records on the batch */
int rb_batch_records(rb_ctx* ctx, rb_batch* b, int with_cigar, rb_records* out);

/* ---- BED text parsed on the device (bed::parse_bed, bed.rs:140-194, quirk for quirk as rbh::Windows::pack_text restates it) ---- */
typedef struct rb_bed_info {
    uint64_t text_bytes;   /* BED text parsed (the inflated size for BGZF input) */
    uint64_t n_lines;      /* non-empty lines: runs of '\n' / '\r' separate lines */
    uint64_t n_comments;   /* lines whose first byte is '#' */
    uint64_t n_parsed;     /* rows that parse: these number the BED rows (bed_row), whether or not their contig is in the batch */
    uint32_t n_win;        /* rows kept: contig name present in the batch's name table */
    uint32_t n_fields;     /* field count of the first non-comment line: every row must have it */
    int default_ids;       /* 1: n_fields <= 3, ids are "{chrom}:{st+1}-{en}" formatted on the device */
    int general;           /* 1: rows nested / file order != sorted order -> the brute-force join layout (Q5) */
} rb_bed_info;
/* BED text, or BGZF bytes (rb_is_bgzf), -> the windows of batch b, replacing any it had; contig names resolve against b's name
 * table (query and target names, like Paf::find_name).  Parsed, sorted and packed on the device. info is nullable.
 * RB_ERR_BAD_ARG: a slice, null data, a plain (single-member) gzip stream, corrupt BGZF; RB_ERR_UNSUPPORTED: more than 2^32 - 1
 * parsed rows.  On failure the batch is left without windows. */
int rb_batch_set_windows_bed(rb_ctx* ctx, rb_batch* b, const uint8_t* data, uint64_t nbytes, rb_bed_info* info);
/* the batch's windows in the rb_windows layout (sorted by (t_id, st), stable; ids NULL when default), library-owned pinned,
 * valid until rb_batch_free or the next rb_batch_windows on the batch */
int rb_batch_windows(rb_ctx* ctx, rb_batch* b, rb_windows* out);

/* `rb liftover --bed` from the files' bytes: paf / bed = plain text or BGZF (rb_is_bgzf), as rb_batch_upload_paf /
 * rb_batch_set_windows_bed take them.  On an N-device context the PAF is split into N byte ranges cut at line starts, and every
 * device parses, tokenises and lifts its own lines (a PAF below multi_min_bytes, RB_MULTI_MIN_BYTES, stays on the first device). The
 * rows are returned in the reference's emission order in one pinned block, laid out exactly as rb_liftover lays them out.  want:
 * RB_WANT_TEXT / RB_WANT_NUMERIC / RB_WANT_STATS_TEXT as in rb_liftover; RB_WANT_QBED -> RB_ERR_BAD_ARG.  Errors, statuses and
 * messages are those of the one-device batch path. Line numbers and record indices count over the whole file. infos are nullable;
 * paf_info is filled once the PAF has parsed (also when a later step fails), bed_info on success; paf_info->names stays valid until
 * the next call on ctx. */
int rb_liftover_text(rb_ctx* ctx, const uint8_t* paf, uint64_t paf_nbytes, const uint8_t* bed, uint64_t bed_nbytes, int policy,
                     uint32_t want, rb_lift_out* out, rb_stats_out* stats /* nullable */, rb_paf_info* paf_info, rb_bed_info* bed_info);

/* ---- host helper: stable sort of BED rows by (t_id, st) into the rb_windows layout ----
 * perm_out[n_win] receives, for each sorted position, the BED row it came from. */
int rb_sort_windows(uint32_t n_win, const uint32_t* t_id, const uint64_t* st, uint32_t* perm_out);

/* replaces the inflate step of `myio::reader` for BGZF input (myio.rs:41-64: `.bgz` goes through gzp::BgzfSyncReader before
 * Paf::from_file reads lines, paf.rs:62-78): `bgzf` = the file's bytes (a series of BGZF blocks, what bgzip writes); the blocks are
 * inflated on the device, one thread per block, CRC-32 and ISIZE of every trailer verified; *text = the inflated bytes in
 * library-owned pinned host memory (rb_free_text), *text_nbytes their count.  RB_ERR_BAD_ARG: not BGZF / corrupt data.  A plain
 * single-member .gz is one dependent stream and is not handled here (rb_is_bgzf tells them apart). */
int rb_is_bgzf(const uint8_t* data, uint64_t nbytes);
int rb_inflate_bgzf(rb_ctx* ctx, const uint8_t* bgzf, uint64_t nbytes, uint8_t** text, uint64_t* text_nbytes);
void rb_free_text(rb_ctx* ctx, uint8_t* text);

/* ---- host helper: page-lock caller-owned buffers (cudaHostRegister) so that the H2D copies of
 * rb_liftover / rb_batch_upload are asynchronous DMA; for hosts without their own CUDA binding.  Allocate such buffers
 * page-aligned and padded to whole pages (a page shared with another object would end up half page-locked), and call
 * rb_host_unregister BEFORE freeing them.  Large ranges are registered in GiB-aligned pieces. */
int rb_host_register(void* ptr, uint64_t nbytes);
int rb_host_unregister(void* ptr);

const char* rb_version(void);

#ifdef __cplusplus
}
#endif
#endif /* RBCUDA_H */
