// paf_parse_core.cuh — the per-token rules of PafRecord::new (paf.rs:379-430, restated by rbh::Paf::from_text in
// host/rbhost.cpp), __host__ __device__: k_paf_fields (paf_parse_kernels.cu) applies them on the GPU and
// tests/native/paf_parse_check.cpp runs the serial line parser below against the host reader on the CPU.
//
//   lines   split at '\n', one trailing '\r' dropped, a last line without a terminator counts, an empty line is a line
//   tokens  split on ' ', '\t', '\n', '\x0C', '\r' (split_ascii_whitespace)
//   < 12 tokens                                   -> panic  "assertion failed: t.len() >= 12"
//   an extra token without (..):(.): somewhere    -> panic  "assertion failed: PAF_TAG.is_match(token)"; the first cg tag wins
//   columns 1,2,3,6,7,8,9,10,11 not parse::<u64>, or a strand of more than one byte -> the line is skipped, unless its cg payload
//   fails the CIGAR syntax check                  -> panic  "Unable to parse cigar string."
#pragma once
#include <cstdint>

#ifdef __CUDACC__
#define RB_PP_HD __host__ __device__ __forceinline__
#else
#define RB_PP_HD inline
#endif

namespace rbpp {

// per-line state, in the order the kinds are decided
enum : uint8_t { LS_OK = 0, LS_SKIPPED = 1, LS_FEW_COLUMNS = 2, LS_BAD_TAG = 3, LS_BAD_CIGAR = 4 };

RB_PP_HD bool is_ws(uint8_t c) { return c <= ' ' && (c == ' ' || c == '\t' || c == '\n' || c == '\x0C' || c == '\r'); }

// Rust str::parse::<u64>: optional '+', at least one digit, overflow = does not parse.  At most 21 bytes are read before
// it decides, whatever the token's length.
RB_PP_HD bool parse_u64(const uint8_t* s, uint64_t n, uint64_t& out) {
    uint64_t i = 0;
    if (n && s[0] == '+') i = 1;
    if (i >= n) return false;
    uint64_t v = 0;
    for (; i < n; i++) {
        if (s[i] < '0' || s[i] > '9') return false;
        const uint64_t d = (uint64_t)(s[i] - '0');
        if (v > (UINT64_MAX - d) / 10) return false;
        v = v * 10 + d;
    }
    out = v;
    return true;
}

// PAF_TAG (paf.rs:21) matches at offset a of a token of tn bytes
RB_PP_HD bool tag_at(const uint8_t* tok, uint64_t a, uint64_t tn) { return a + 5 <= tn && tok[a + 2] == ':' && tok[a + 4] == ':'; }

// CigarString::try_from as paf.rs:398-399 calls it, syntax only (what rbhost.cpp's cigar_syntax_ok checks): <digits fitting u32>
// <one of MIDNSHP=X> repeated; H only as the first or last op, S only at the ends or separated from them by H only
RB_PP_HD bool cigar_syntax_ok(const uint8_t* s, uint64_t n) {
    uint64_t i = 0;
    while (i < n) {
        uint64_t j = i;
        unsigned long long v = 0;
        while (j < n && s[j] >= '0' && s[j] <= '9') {
            v = v * 10 + (unsigned long long)(s[j] - '0');
            if (v > 0xFFFFFFFFull) return false;
            j++;
        }
        if (j == i || j >= n) return false;
        const uint8_t op = s[j];
        if (!(op == 'M' || op == 'I' || op == 'D' || op == 'N' || op == 'S' || op == 'H' || op == 'P' || op == '=' || op == 'X')) return false;
        if (op == 'H' && i != 0 && j + 1 != n) return false;
        if (op == 'S' && i != 0 && j + 1 != n && s[i - 1] != 'H') {
            for (uint64_t k = j + 1; k < n; k++)
                if (!((s[k] >= '0' && s[k] <= '9') || s[k] == 'H')) return false;
        }
        i = j + 1;
    }
    return true;
}

// What one line yields (spans are offsets into the text)
struct LineOut {
    uint64_t v[7];  // q_len q_st q_en t_len t_st t_en mapq
    uint64_t qn_off, tn_off, cg_off, cg_len;
    uint32_t qn_len, tn_len;
    uint8_t state, strand;
};

// The decision once the tokens are known: tok_off / tok_len = the first 12 tokens (n_tok = how many there are, capped at 12),
// bad_tag = some extra token failed tag_at everywhere, has_cg / cg_* = the cg payload: the first one, except that an empty
// payload does not hold the place (the host reader tests `cg_n == 0`, so a later cg tag replaces an empty one).
RB_PP_HD void line_finish(const uint8_t* text, const uint64_t* tok_off, const uint64_t* tok_len, uint32_t n_tok, bool bad_tag,
                          bool has_cg, uint64_t cg_off, uint64_t cg_len, LineOut& L) {
    L.qn_off = L.tn_off = L.cg_off = L.cg_len = 0;
    L.qn_len = L.tn_len = 0;
    L.strand = '+';
    for (int k = 0; k < 7; k++) L.v[k] = 0;
    if (n_tok < 12) { L.state = LS_FEW_COLUMNS; return; }
    if (bad_tag) { L.state = LS_BAD_TAG; return; }
    const int colidx[9] = {1, 2, 3, 6, 7, 8, 9, 10, 11};
    uint64_t v[9];
    bool ok = true;
    for (int c = 0; c < 9 && ok; c++) ok = parse_u64(text + tok_off[colidx[c]], tok_len[colidx[c]], v[c]);
    if (!ok || tok_len[4] != 1) {
        L.state = (has_cg && !cigar_syntax_ok(text + cg_off, cg_len)) ? LS_BAD_CIGAR : LS_SKIPPED;
        return;
    }
    L.state = LS_OK;
    L.v[0] = v[0]; L.v[1] = v[1]; L.v[2] = v[2]; L.v[3] = v[3]; L.v[4] = v[4]; L.v[5] = v[5]; L.v[6] = v[8];
    L.strand = text[tok_off[4]];
    L.qn_off = tok_off[0]; L.qn_len = (uint32_t)tok_len[0];
    L.tn_off = tok_off[5]; L.tn_len = (uint32_t)tok_len[5];
    if (has_cg) { L.cg_off = cg_off; L.cg_len = cg_len; }
}

// Serial form over one line [b, e) (line terminator and '\r' already removed): the statement the GPU kernel is checked against.
RB_PP_HD void parse_line_serial(const uint8_t* text, uint64_t b, uint64_t e, LineOut& L) {
    uint64_t tok_off[12], tok_len[12];
    uint32_t n_tok = 0;
    bool bad_tag = false, has_cg = false;
    uint64_t cg_off = 0, cg_len = 0;
    uint64_t p = b;
    for (;;) {
        while (p < e && is_ws(text[p])) p++;
        if (p >= e) break;
        uint64_t q = p;
        while (q < e && !is_ws(text[q])) q++;
        if (n_tok < 12) {
            tok_off[n_tok] = p; tok_len[n_tok] = q - p; n_tok++;
        } else if (!bad_tag) {
            const uint64_t tn = q - p;
            uint64_t m = tn;
            for (uint64_t a = 0; a + 5 <= tn; a++)
                if (tag_at(text + p, a, tn)) { m = a; break; }
            if (m == tn) bad_tag = true;
            else if (cg_len == 0 && text[p + m] == 'c' && text[p + m + 1] == 'g') { has_cg = true; cg_off = p + m + 5; cg_len = tn - (m + 5); }
        }
        p = q;
    }
    line_finish(text, tok_off, tok_len, n_tok, bad_tag, has_cg, cg_off, cg_len, L);
}

}  // namespace rbpp
