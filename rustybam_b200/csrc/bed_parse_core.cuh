// bed_parse_core.cuh — the per-line rules of rbh::Windows::pack_text (host/rbhost.cpp; bio 1.6.0 bed::Reader over csv as bed.rs:140-194
// uses it), __host__ __device__: k_bed_fields / k_bed_judge (bed_parse_kernels.cu) apply them on the GPU and
// tests/native/bed_parse_check.cpp runs them against the host packer on the CPU.
//
//   lines    end at '\n' or '\r'; a run of them is one separator, so no line is empty; a line starting with '#' is a comment
//   fields   split on '\t' only (spaces belong to the field); the field count of the FIRST non-comment line is every row's
//            (even when that line itself does not parse); a row with another count, or fewer than 3, is skipped
//   numbers  st / en: at least one byte, ASCII digits only, no u64 overflow, else the row is skipped (st > en is not checked)
//   bed_row  index among the rows that parse, in file order, whatever their contig
//   kept     field 1 byte-equal to a name of the batch's name table; t_id = that name's id
//   ids      field 4 verbatim (may be empty) when the field count is > 3, else the default id (formatted on the device)
#pragma once
#include <cstdint>

#ifdef __CUDACC__
#define RB_BP_HD __host__ __device__ __forceinline__
#else
#define RB_BP_HD inline
#endif

namespace rbbp {

RB_BP_HD bool is_eol(uint8_t c) { return c == '\n' || c == '\r'; }

// the strict number of bio's BED reader: non-empty, digits only, fits u64
RB_BP_HD bool parse_num(const uint8_t* s, uint64_t n, uint64_t& out) {
    if (n == 0) return false;
    uint64_t v = 0;
    for (uint64_t i = 0; i < n; i++) {
        if (s[i] < '0' || s[i] > '9') return false;
        const uint64_t d = (uint64_t)(s[i] - '0');
        if (v > (UINT64_MAX - d) / 10) return false;
        v = v * 10 + d;
    }
    out = v;
    return true;
}

// What one line [a, b) (no EOL byte inside, b > a) yields; spans are offsets into the text
struct BedLine {
    uint64_t n_fields;
    uint64_t st, en;
    uint64_t name_len;        // field 1 starts at the line's first byte
    uint64_t id_off, id_len;  // field 4 (0, 0 when there are fewer than 4 fields)
    bool comment;
    bool nums_ok;             // fields 2 and 3 exist and parse
};

RB_BP_HD void bed_line(const uint8_t* text, uint64_t a, uint64_t b, BedLine& L) {
    L.n_fields = 0; L.st = L.en = 0; L.name_len = 0; L.id_off = L.id_len = 0;
    L.comment = text[a] == '#';
    L.nums_ok = false;
    if (L.comment) return;
    uint64_t o1 = 0, l1 = 0, o2 = 0, l2 = 0;  // fields 2 and 3 (scalars, not an array: no local memory on the device)
    uint64_t nf = 0, p = a;
    for (uint64_t q = a;; q++) {
        if (q == b || text[q] == '\t') {
            if (nf == 0) L.name_len = q - p;
            else if (nf == 1) { o1 = p; l1 = q - p; }
            else if (nf == 2) { o2 = p; l2 = q - p; }
            else if (nf == 3) { L.id_off = p; L.id_len = q - p; }
            nf++;
            p = q + 1;
            if (q == b) break;
        }
    }
    L.n_fields = nf;
    L.nums_ok = nf >= 3 && parse_num(text + o1, l1, L.st) && parse_num(text + o2, l2, L.en);
}

// the row parses (it gets a bed_row) against nf0, the field count of the first non-comment line
RB_BP_HD bool row_parses(const BedLine& L, uint64_t nf0) { return !L.comment && L.n_fields == nf0 && nf0 >= 3 && L.nums_ok; }

// FNV-1a over a name's bytes: the device name table (k_bed_names / k_bed_judge) hashes with it
RB_BP_HD uint64_t name_hash(const uint8_t* s, uint64_t n) {
    uint64_t h = 1469598103934665603ull;
    for (uint64_t i = 0; i < n; i++) h = (h ^ s[i]) * 1099511628211ull;
    return h ^ (h >> 29);
}

}  // namespace rbbp
