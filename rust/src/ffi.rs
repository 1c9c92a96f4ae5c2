//! src/ffi.rs of the drop-in: the binding of include/rbcuda.h (librbcuda, CUDA for sm_100a).
//! Replaces, at their call sites, liftover::trim_paf_by_rgns (src/main.rs:197), bamstats::stats_from_paf (src/main.rs:53-56),
//! liftover::break_paf_on_indels (main.rs:271-281), paf_swap_query_and_target (main.rs:176-182) and
//! Paf::overlapping_paf_recs (main.rs:218-230).  NOT compiled in this repository's image (no cargo / rustc here); the ctypes
//! binding rustybam_b200/capi.py declares the same symbols and tests/test_host_cpu.py checks them against the built library.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)] pub struct rb_ctx { _p: [u8; 0] }
#[repr(C)] pub struct rb_batch { _p: [u8; 0] }

#[repr(C)]
pub struct rb_records {
    pub n_rec: u32,
    pub cigar: *const u8, pub cigar_nbytes: u64, pub cigar_off: *const u64,
    pub q_len: *const u64, pub q_st: *const u64, pub q_en: *const u64,
    pub t_len: *const u64, pub t_st: *const u64, pub t_en: *const u64, pub mapq: *const u64,
    pub strand: *const u8, pub q_id: *const u32, pub t_id: *const u32,
    pub names: *const u8, pub names_off: *const u64, pub n_names: u32,
}
#[repr(C)]
pub struct rb_windows {
    pub n_win: u32, pub t_id: *const u32, pub st: *const u64, pub en: *const u64,
    pub bed_row: *const u32, pub ids: *const u8, pub ids_off: *const u64,
}
#[repr(C)]
pub struct rb_lift_out {
    pub n_out: u64, pub paf_text: *mut u8, pub paf_nbytes: u64, pub line_off: *mut u64,
    pub q_st: *mut u64, pub q_en: *mut u64, pub t_st: *mut u64, pub t_en: *mut u64,
    pub nmatch: *mut u64, pub aln_len: *mut u64, pub rec_idx: *mut u32, pub win_idx: *mut u32,
    pub n_pairs: u64, pub _owner: *mut c_void,
}
#[repr(C)]
pub struct rb_stats_out {
    pub n: u64,
    pub equal: *mut u32, pub diff: *mut u32, pub ins: *mut u32, pub del: *mut u32,
    pub ins_events: *mut u32, pub del_events: *mut u32, pub matches: *mut u32,
    pub id_by_matches: *mut f32, pub id_by_events: *mut f32, pub id_by_all: *mut f32,
    pub _owner: *mut c_void,
}
#[repr(C)]
pub struct rb_paf_info {
    pub text_bytes: u64, pub n_lines: u64, pub skipped: u64,
    pub n_rec: u32, pub n_names: u32,
    pub names: *const u8, pub names_off: *const u64,
    pub cigar_bytes: u64,
}
#[repr(C)]
pub struct rb_bed_info {
    pub text_bytes: u64, pub n_lines: u64, pub n_comments: u64, pub n_parsed: u64,
    pub n_win: u32, pub n_fields: u32,
    pub default_ids: c_int, pub general: c_int,
}
#[repr(C)]
pub struct rb_summary { pub n_ops: u64, pub n_pairs: u64, pub n_out: u64, pub out_bytes: u64, pub cigar_bytes: u64 }
extern "C" {
    pub fn rb_ctx_create(device_ids: *const c_int, n: c_int, status: *mut c_int) -> *mut rb_ctx;
    pub fn rb_ctx_destroy(ctx: *mut rb_ctx);
    pub fn rb_last_error(ctx: *const rb_ctx) -> *const c_char;
    pub fn rb_liftover(ctx: *mut rb_ctx, recs: *const rb_records, wins: *const rb_windows, policy: c_int,
                       want: u32, out: *mut rb_lift_out, stats: *mut rb_stats_out) -> c_int;
    pub fn rb_stats(ctx: *mut rb_ctx, recs: *const rb_records, stats: *mut rb_stats_out) -> c_int;
    pub fn rb_break_paf(ctx: *mut rb_ctx, recs: *const rb_records, max_size: u32, policy: c_int, want: u32,
                        out: *mut rb_lift_out, stats: *mut rb_stats_out) -> c_int;
    pub fn rb_invert(ctx: *mut rb_ctx, recs: *const rb_records, want: u32, out: *mut rb_lift_out) -> c_int;
    pub fn rb_trim_paf(ctx: *mut rb_ctx, recs: *const rb_records, match_score: c_int, diff_score: c_int, indel_score: c_int,
                       remove_contained: c_int, policy: c_int, want: u32, out: *mut rb_lift_out, stats: *mut rb_stats_out) -> c_int;
    pub fn rb_free_lift_out(ctx: *mut rb_ctx, out: *mut rb_lift_out);
    pub fn rb_free_stats_out(ctx: *mut rb_ctx, stats: *mut rb_stats_out);
    pub fn rb_sort_windows(n: u32, t_id: *const u32, st: *const u64, perm_out: *mut u32) -> c_int;
    /// myio.rs:41-64 — the inflate step of `reader()` for BGZF input, on the device; `text` is pinned, library-owned (rb_free_text)
    pub fn rb_is_bgzf(data: *const u8, nbytes: u64) -> c_int;
    pub fn rb_inflate_bgzf(ctx: *mut rb_ctx, bgzf: *const u8, nbytes: u64, text: *mut *mut u8, text_nbytes: *mut u64) -> c_int;
    pub fn rb_free_text(ctx: *mut rb_ctx, text: *mut u8);
    pub fn rb_host_register(ptr: *mut c_void, nbytes: u64) -> c_int;
    pub fn rb_host_unregister(ptr: *mut c_void) -> c_int;
    pub fn rb_trim_paf_begin(ctx: *mut rb_ctx, recs: *const rb_records, match_score: c_int, diff_score: c_int, indel_score: c_int, policy: c_int) -> c_int;
    pub fn rb_trim_paf_round(ctx: *mut rb_ctx, waiting: *mut c_int) -> c_int;
    pub fn rb_trim_paf_end(ctx: *mut rb_ctx, remove_contained: c_int, want: u32, out: *mut rb_lift_out, stats: *mut rb_stats_out) -> c_int;
    /// paf.rs:62-78 Paf::from_file on the device: PAF text or BGZF bytes -> a resident batch (name table in `info`, library-owned)
    pub fn rb_batch_upload_paf(ctx: *mut rb_ctx, data: *const u8, nbytes: u64, info: *mut rb_paf_info, status: *mut c_int) -> *mut rb_batch;
    pub fn rb_batch_set_windows(ctx: *mut rb_ctx, b: *mut rb_batch, wins: *const rb_windows) -> c_int;
    pub fn rb_batch_records(ctx: *mut rb_ctx, b: *mut rb_batch, with_cigar: c_int, out: *mut rb_records) -> c_int;
    /// bed.rs:140-194 bed::parse_bed on the device: BED text or BGZF bytes -> the batch's windows (names resolve against its name table)
    pub fn rb_batch_set_windows_bed(ctx: *mut rb_ctx, b: *mut rb_batch, data: *const u8, nbytes: u64, info: *mut rb_bed_info) -> c_int;
    pub fn rb_batch_windows(ctx: *mut rb_ctx, b: *mut rb_batch, out: *mut rb_windows) -> c_int;
    /// `rb liftover --bed` from the files' bytes (PAF and BED text or BGZF), the PAF parsed across every device of the context
    pub fn rb_liftover_text(ctx: *mut rb_ctx, paf: *const u8, paf_nbytes: u64, bed: *const u8, bed_nbytes: u64, policy: c_int, want: u32,
                            out: *mut rb_lift_out, stats: *mut rb_stats_out, paf_info: *mut rb_paf_info, bed_info: *mut rb_bed_info) -> c_int;
    pub fn rb_batch_liftover(ctx: *mut rb_ctx, b: *mut rb_batch, policy: c_int, want: u32, with_stats: c_int, summary: *mut rb_summary) -> c_int;
    pub fn rb_batch_download_lift(ctx: *mut rb_ctx, b: *mut rb_batch, want: u32, out: *mut rb_lift_out, stats: *mut rb_stats_out) -> c_int;
    pub fn rb_batch_free(ctx: *mut rb_ctx, b: *mut rb_batch);
    // tuning (optional): slice threshold of rb_liftover, boundary driver
    pub fn rb_ctx_set_slicing(ctx: *mut rb_ctx, min_slice_bytes: u64) -> c_int;
    pub fn rb_ctx_set_lift_mode(ctx: *mut rb_ctx, mode: c_int) -> c_int;
}

pub const RB_POLICY_RIGHTMOST: c_int = 0;
pub const RB_POLICY_EARLY_EXIT: c_int = 1;
pub const RB_WANT_TEXT: u32 = 1;
pub const RB_WANT_NUMERIC: u32 = 2;
pub const RB_WANT_QBED: u32 = 4;
/// rb_liftover: paf_text holds the rows `rb stats --paf` prints for the lifted rows (formatted on the GPU) instead of PAF rows
pub const RB_WANT_STATS_TEXT: u32 = 8;

/// One context for `n` GPUs: rb_liftover / rb_stats spread the records over them and merge the rows into ONE output in the
/// reference's emission order (liftover.rs:151-164); nothing else changes at the call sites.
pub fn context(devices: &[c_int]) -> *mut rb_ctx {
    let mut status: c_int = 0;
    let ctx = unsafe { rb_ctx_create(devices.as_ptr(), devices.len() as c_int, &mut status) };
    assert!(!ctx.is_null(), "no usable sm_100 CUDA device (status {}): this build has no CPU path", status);
    ctx
}
