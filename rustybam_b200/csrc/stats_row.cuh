// stats_row.cuh — one row of `rb stats --paf` (bamstats.rs:239-270) from a record's columns and its Stats, __host__ __device__:
// k_stats_rows composes the rows of rb_stats_text with it, and tests/native/stats_row_check.cpp holds it against rbh::append_row.
//   reference block, strand, query block (qbed: query block first), the three identities with Rust's `{}` for f32 (f32_fmt.cuh),
//   matches, mismatches, deletion events, insertion events, deletions, insertions; tab-separated, '\n' at the end.
#pragma once
#include <stdint.h>

#include "f32_fmt.cuh"
#include "put_digits.cuh"

namespace rb {

struct StatsRow {
    const uint8_t* q_name;
    const uint8_t* t_name;
    uint32_t q_name_len, t_name_len;
    uint64_t q_st, q_en, q_len, t_st, t_en, t_len;  // the record's columns as read: stats_from_paf strips nothing
    uint8_t strand;
    uint32_t equal, diff, ins, del, ins_events, del_events, matches;
    uint32_t id_bits[3];  // id_by_matches, id_by_events, id_by_all as f32 bit patterns
    F32Dec id_dec[3];     // their shortest digits: stats_row_digits fills them, stats_row_len and stats_row_put read them
};

// (apart from the rest: the digit search may call the big-integer core, and a caller that runs it before loading the other fields
// keeps little alive across that call)
RB_HD void stats_row_digits(StatsRow& r) {
    for (int k = 0; k < 3; k++) r.id_dec[k] = f32_shortest_fast(r.id_bits[k]);
}

// Stats keeps the coordinates as i64 (bamstats.rs:91-154 casts the u64 columns with `as i64`): a column >= 2^63 prints negative
RB_HD uint32_t i64_len(uint64_t v) { return (int64_t)v < 0 ? 1u + ndigits64(0ull - v) : ndigits64(v); }
RB_HD uint8_t* put_i64(uint8_t* p, uint64_t v) {
    if ((int64_t)v < 0) { *p++ = '-'; v = 0ull - v; }
    return put_u64(p, v);
}

RB_HD uint32_t stats_row_len(const StatsRow& r) {
    uint32_t n = r.q_name_len + r.t_name_len + 1u + 18u;  // names, strand, 17 tabs and the newline
    n += i64_len(r.q_st) + i64_len(r.q_en) + i64_len(r.q_len) + i64_len(r.t_st) + i64_len(r.t_en) + i64_len(r.t_len);
    for (int k = 0; k < 3; k++) n += f32_display_len(r.id_bits[k], r.id_dec[k]);
    return n + ndigits32(r.equal) + ndigits32(r.diff) + ndigits32(r.del_events) + ndigits32(r.ins_events) + ndigits32(r.del) + ndigits32(r.ins);
}

RB_HD uint8_t* stats_row_block(uint8_t* p, const uint8_t* name, uint32_t name_len, uint64_t st, uint64_t en, uint64_t len) {
    p = put_bytes(p, name, name_len);
    *p++ = '\t'; p = put_i64(p, st); *p++ = '\t'; p = put_i64(p, en); *p++ = '\t'; p = put_i64(p, len); *p++ = '\t';
    return p;
}

// writes the stats_row_len(r) bytes of the row at p; returns p + that
RB_HD uint8_t* stats_row_put(uint8_t* p, const StatsRow& r, bool qbed) {
    if (qbed) p = stats_row_block(p, r.q_name, r.q_name_len, r.q_st, r.q_en, r.q_len);
    else p = stats_row_block(p, r.t_name, r.t_name_len, r.t_st, r.t_en, r.t_len);
    *p++ = r.strand; *p++ = '\t';
    if (qbed) p = stats_row_block(p, r.t_name, r.t_name_len, r.t_st, r.t_en, r.t_len);
    else p = stats_row_block(p, r.q_name, r.q_name_len, r.q_st, r.q_en, r.q_len);
    for (int k = 0; k < 3; k++) { p = f32_display_put(p, r.id_bits[k], r.id_dec[k]); *p++ = '\t'; }
    p = put_u32(p, r.equal); *p++ = '\t'; p = put_u32(p, r.diff); *p++ = '\t'; p = put_u32(p, r.del_events); *p++ = '\t';
    p = put_u32(p, r.ins_events); *p++ = '\t'; p = put_u32(p, r.del); *p++ = '\t'; p = put_u32(p, r.ins); *p++ = '\n';
    return p;
}

}  // namespace rb
