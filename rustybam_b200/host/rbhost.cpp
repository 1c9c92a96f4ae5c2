// rbhost.cpp — host-side text I/O, packing and printing (see rbhost.hpp for the reference lines).
#include "rbhost.hpp"
#include "f32_fast.hpp"
#include "../csrc/name_intern.hpp"

#include <cerrno>
#include <unistd.h>
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <zlib.h>

#include <algorithm>
#include <memory>
#include <charconv>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <thread>
#include <atomic>
#include <iostream>
#include <sstream>

namespace rbh {

// ---------------------------------------------------------------------------------------------
// myio.rs:41-64 — extension decides: .gz / .bgz -> inflate (zlib reads concatenated BGZF members), else plain
// ---------------------------------------------------------------------------------------------
static std::string read_plain(const std::string& path) {
    std::string out;
    FILE* f = fopen(path.c_str(), "rb");
    if (!f) throw Panic("Error: cannot read input file " + path);
    fseek(f, 0, SEEK_END);
    const long sz = ftell(f);
    fseek(f, 0, SEEK_SET);
    if (sz > 0) {
        out.resize((size_t)sz);
        if (fread(&out[0], 1, (size_t)sz, f) != (size_t)sz) { fclose(f); throw Panic("short read on " + path); }
    }
    fclose(f);
    return out;
}

// BGZF: a series of gzip members, each with a 'BC' extra subfield holding (block size - 1) and at most 64 KiB of
// payload, ISIZE in the trailer.  Blocks are located serially (header hops), inflated in parallel (raw deflate).
// Returns false if `raw` is not a well-formed BGZF file.
static bool inflate_bgzf(const std::string& raw, std::string& text) {
    struct Block { size_t cdata, clen, out_off, out_len; };
    std::vector<Block> blocks;
    const unsigned char* p = reinterpret_cast<const unsigned char*>(raw.data());
    const size_t n = raw.size();
    size_t pos = 0, total = 0;
    while (pos < n) {
        if (n - pos < 18 || p[pos] != 0x1f || p[pos + 1] != 0x8b || p[pos + 2] != 8 || !(p[pos + 3] & 4)) return false;
        const size_t xlen = p[pos + 10] | (p[pos + 11] << 8);
        size_t x = pos + 12, xend = x + xlen, bsize = 0;
        if (xend > n) return false;
        while (x + 4 <= xend) {
            const size_t slen = p[x + 2] | (p[x + 3] << 8);
            if (p[x] == 'B' && p[x + 1] == 'C' && slen == 2 && x + 6 <= xend) bsize = (size_t)(p[x + 4] | (p[x + 5] << 8)) + 1;
            x += 4 + slen;
        }
        if (bsize == 0 || pos + bsize > n || bsize < xlen + 20) return false;
        const size_t isize = (size_t)p[pos + bsize - 4] | ((size_t)p[pos + bsize - 3] << 8) | ((size_t)p[pos + bsize - 2] << 16) |
                             ((size_t)p[pos + bsize - 1] << 24);
        blocks.push_back(Block{xend, bsize - xlen - 20, total, isize});
        total += isize;
        pos += bsize;
    }
    text.resize(total);
    std::atomic<size_t> next{0};
    std::atomic<bool> ok{true};
    auto work = [&] {
        for (;;) {
            const size_t k = next.fetch_add(1);
            if (k >= blocks.size() || !ok.load()) break;
            const Block& b = blocks[k];
            if (b.out_len == 0) continue;
            z_stream zs;
            memset(&zs, 0, sizeof zs);
            if (inflateInit2(&zs, -15) != Z_OK) { ok = false; break; }
            zs.next_in = const_cast<Bytef*>(p + b.cdata);
            zs.avail_in = (uInt)b.clen;
            zs.next_out = reinterpret_cast<Bytef*>(&text[b.out_off]);
            zs.avail_out = (uInt)b.out_len;
            const int rc = inflate(&zs, Z_FINISH);
            inflateEnd(&zs);
            if (rc != Z_STREAM_END || zs.avail_out != 0) { ok = false; break; }
        }
    };
    const unsigned nt = (unsigned)std::min<size_t>(std::max(1u, std::thread::hardware_concurrency()), std::max<size_t>(1, blocks.size() / 16));
    if (nt <= 1) work();
    else {
        std::vector<std::thread> pool;
        for (unsigned t = 0; t < nt; t++) pool.emplace_back(work);
        for (auto& th : pool) th.join();
    }
    return ok.load();
}

std::string read_raw(const std::string& path) { return read_plain(path); }

std::string read_all(const std::string& path) {
    auto ends_with = [&](const char* suf) {
        const size_t n = strlen(suf);
        return path.size() >= n && path.compare(path.size() - n, n, suf) == 0;
    };
    std::string out;
    if (path == "-") {  // read(2) in 8 MiB pieces (std::cin's stream buffer, synchronised with stdio, moves a byte at a time: 25 s for
                        // the 510 MB `rb liftover` pipes into `rb stats --paf`)
        std::vector<char> buf(8u << 20);
        for (;;) {
            const ssize_t n = ::read(0, buf.data(), buf.size());
            if (n < 0) { if (errno == EINTR) continue; throw Panic("error reading stdin"); }
            if (n == 0) break;
            out.append(buf.data(), (size_t)n);
        }
        return out;
    }
    if (ends_with(".bgz")) {  // BGZF (myio.rs:56-60): independent blocks -> inflated on all host threads
        std::string raw = read_plain(path);
        std::string text;
        if (inflate_bgzf(raw, text)) return text;
        // not BGZF after all: fall through to the serial gzip reader
    }
    if (ends_with(".gz") || ends_with(".bgz")) {
        gzFile f = gzopen(path.c_str(), "rb");
        if (!f) throw Panic("couldn't open " + path);
        gzbuffer(f, 1 << 20);
        std::vector<char> buf(1 << 22);
        for (;;) {
            const int n = gzread(f, buf.data(), (unsigned)buf.size());
            if (n < 0) { gzclose(f); throw Panic("error inflating " + path); }
            if (n == 0) break;
            out.append(buf.data(), (size_t)n);
        }
        gzclose(f);
        return out;
    }
    return read_plain(path);
}


// ---------------------------------------------------------------------------------------------
// PAF
// ---------------------------------------------------------------------------------------------
static inline bool is_ws(char c) {  // (one compare for the bytes of a token: every ASCII whitespace byte is <= ' ')
    return (unsigned char)c <= ' ' && (c == ' ' || c == '\t' || c == '\n' || c == '\x0C' || c == '\r');
}

static bool parse_u64(const char* s, size_t n, uint64_t& out) {  // Rust str::parse::<u64>
    size_t i = 0;
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

uint32_t Paf::name_id(const std::string& s) {
    const auto ins = index_.emplace(s, (uint32_t)names.size());  // O(1) amortised per name
    if (ins.second) names.push_back(s);
    return ins.first->second;
}
int64_t Paf::find_name(const std::string& s) const {
    const auto it = index_.find(s);
    return it == index_.end() ? -1 : (int64_t)it->second;
}

// paf.rs:62-78 + 379-430: lines() split at '\n' (one trailing '\r' dropped), split_ascii_whitespace,
// >= 12 columns or panic, every extra token must look like a tag or panic, first cg:Z: wins,
// unparsable numeric column -> the line is skipped.  The CIGAR payload is copied verbatim.
// first ASCII-whitespace byte in [p, e) ('\n' cannot occur inside a line): libc's vectorised memchr instead of a
// byte loop — the cg:Z: token of a whole-genome record is hundreds of kilobytes long
static inline const char* next_ws(const char* p0, const char* e) {
    // short tokens (names, numbers, most tags): a byte loop beats four library calls; only what is still going after 48 bytes
    // (the cg:Z: payload) is handed to memchr
    const char* lim = (e - p0 > 48) ? p0 + 48 : e;
    const char* p = p0;
    for (; p < lim; p++)
        if (is_ws(*p)) return p;
    if (p == e) return e;
    const char* q = (const char*)memchr(p, '\t', (size_t)(e - p));
    if (!q) q = e;
    static const char others[3] = {' ', '\x0C', '\r'};
    for (char c : others) {
        const char* r = (const char*)memchr(p, c, (size_t)(q - p));
        if (r) q = r;
    }
    return q;
}

namespace {
// CigarString::try_from(&[u8]) of rust-htslib as paf.rs:398-399 calls it (.expect -> panic), syntax only: <digits fitting
// u32><one of MIDNSHP=X> repeated; H only as the first or last op, S only at the ends or separated from them by H only.
// Kept records get this check on the GPU (k_tokenise, k_rec_ops, k_check_clips); the host runs it only for lines it is
// about to SKIP because a numeric column does not parse — the reference parses the cg tag first (paf.rs:386-399) and
// panics on a malformed one before it ever looks at the numbers (paf.rs:401-417).
bool cigar_syntax_ok(const char* s, size_t n) {
    size_t i = 0;
    while (i < n) {
        size_t j = i;
        unsigned long long v = 0;
        while (j < n && s[j] >= '0' && s[j] <= '9') {
            v = v * 10 + (unsigned long long)(s[j] - '0');
            if (v > 0xFFFFFFFFull) return false;
            j++;
        }
        if (j == i || j >= n) return false;  // no length, or the text ends in a number
        const char op = s[j];
        if (!memchr("MIDNSHP=X", op, 9)) return false;
        if (op == 'H' && i != 0 && j + 1 != n) return false;
        if (op == 'S' && i != 0 && j + 1 != n && s[i - 1] != 'H') {
            for (size_t k = j + 1; k < n; k++)
                if (!((s[k] >= '0' && s[k] <= '9') || s[k] == 'H')) return false;
        }
        i = j + 1;
    }
    return true;
}

struct ParsedLine {     // what PafRecord::new extracts from one line (paf.rs:379-430), before name interning (no initialisers: see from_text)
    const char *q_name, *t_name, *cg;
    size_t q_name_n, t_name_n, cg_n;
    uint64_t v[9];
    uint8_t strand;
    uint8_t state;  // 0 ok, 1 skipped (unparsable numeric column), 2 panic: < 12 columns, 3 panic: bad tag, 4 panic: bad cg on a skipped line
};

void parse_line(const char* text, size_t i, size_t e, ParsedLine& L) {
    L.q_name = L.t_name = L.cg = nullptr;
    L.q_name_n = L.t_name_n = L.cg_n = 0;
    L.strand = '+';
    L.state = 0;
    std::pair<const char*, size_t> t[12];
    size_t nt = 0, p = i;
    const char* end = text + e;
    auto next_token = [&](const char*& tok, size_t& tn) {
        const char* a = text + p;
        while (a < end && is_ws(*a)) a++;
        if (a >= end) { p = e; return false; }
        const char* b = next_ws(a, end);
        tok = a; tn = (size_t)(b - a);
        p = (size_t)(b - text);
        return true;
    };
    const char* tok; size_t tn;
    while (nt < 12 && next_token(tok, tn)) t[nt++] = {tok, tn};
    if (nt < 12) { L.state = 2; return; }
    while (next_token(tok, tn)) {  // tags: (..):(.):(.*) somewhere in the token (paf.rs:21,387-389); first cg wins
        size_t m = SIZE_MAX;
        for (size_t a = 0; a + 5 <= tn; a++)
            if (tok[a + 2] == ':' && tok[a + 4] == ':') { m = a; break; }
        if (m == SIZE_MAX) { L.state = 3; return; }
        if (tok[m] == 'c' && tok[m + 1] == 'g' && L.cg_n == 0) { L.cg = tok + m + 5; L.cg_n = tn - (m + 5); }
    }
    static const int colidx[9] = {1, 2, 3, 6, 7, 8, 9, 10, 11};
    bool ok = true;
    for (int c = 0; c < 9 && ok; c++) ok = parse_u64(t[colidx[c]].first, t[colidx[c]].second, L.v[c]);
    if (!ok || t[4].second != 1) {  // skipped — unless its cg tag is malformed: the reference panics on that first
        L.state = (L.cg && !cigar_syntax_ok(L.cg, L.cg_n)) ? 4 : 1;
        return;
    }
    L.strand = (uint8_t)t[4].first[0];
    L.q_name = t[0].first; L.q_name_n = t[0].second;
    L.t_name = t[5].first; L.t_name_n = t[5].second;
}
}  // namespace

// Lines are parsed in parallel (host threads), records are assembled in file order: name ids, skipped-line count
// and the first panic are exactly those of the serial loop of Paf::from_file (paf.rs:62-78).
Paf Paf::from_text(const char* text, size_t n) {
    Paf paf;
    std::vector<std::pair<size_t, size_t>> lines;  // [begin, end) without the line terminator
    const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
    {   // line terminators: every thread scans one piece of the text (one memchr pass over many GB is seconds on one core)
        const unsigned ns = n < (64u << 20) ? 1u : hw;
        std::vector<std::vector<size_t>> nls(ns);
        auto scan = [&](unsigned t) {
            const size_t a = n / ns * t, b = (t + 1 == ns) ? n : n / ns * (t + 1);
            for (size_t i = a; i < b;) {
                const char* nl = (const char*)memchr(text + i, '\n', b - i);
                if (!nl) break;
                nls[t].push_back((size_t)(nl - text));
                i = (size_t)(nl - text) + 1;
            }
        };
        if (ns == 1) scan(0);
        else {
            std::vector<std::thread> pool;
            for (unsigned t = 0; t < ns; t++) pool.emplace_back(scan, t);
            for (auto& th : pool) th.join();
        }
        size_t i = 0;
        for (unsigned t = 0; t < ns; t++)
            for (const size_t j : nls[t]) {
                size_t e = j;
                if (e > i && text[e - 1] == '\r') e--;
                lines.emplace_back(i, e);
                i = j + 1;
            }
        if (i < n) lines.emplace_back(i, n);  // last line without a terminator
    }
    // (one ParsedLine per line, 136 bytes: left uninitialised — parse_line sets every field — so that millions of short rows do
    // not start with one thread zeroing hundreds of MB)
    std::unique_ptr<ParsedLine[]> parsed_store(new ParsedLine[lines.size()]);
    ParsedLine* parsed = parsed_store.get();
    const unsigned nt = (unsigned)std::min<size_t>(n < (8u << 20) ? 1 : hw, std::max<size_t>(1, lines.size()));
    if (nt <= 1) {
        for (size_t k = 0; k < lines.size(); k++) parse_line(text, lines[k].first, lines[k].second, parsed[k]);
    } else {
        std::atomic<size_t> next{0};
        std::vector<std::thread> pool;
        for (unsigned t = 0; t < nt; t++)
            pool.emplace_back([&] {
                for (;;) {  // (a few hundred lines per grab: short rows would otherwise fight over the counter)
                    const size_t k0 = next.fetch_add(256);
                    if (k0 >= lines.size()) break;
                    const size_t k1 = std::min(lines.size(), k0 + 256);
                    for (size_t k = k0; k < k1; k++) parse_line(text, lines[k].first, lines[k].second, parsed[k]);
                }
            });
        for (auto& th : pool) th.join();
    }
    // kept records: their index and the place of their CIGAR payload (one serial pass of additions; the first panic in file
    // order is the one reported, like the serial loop of the reference)
    const size_t n_lines = lines.size();
    if (n_lines > 0xFFFFFFFFull) throw Panic("more than 2^32 lines");
    std::vector<uint32_t> kept;  // line index of record r
    kept.reserve(n_lines);
    size_t total_cg = 0;
    for (size_t k = 0; k < n_lines; k++) {
        const ParsedLine& L = parsed[k];
        if (L.state == 2) throw Panic("assertion failed: t.len() >= 12");
        if (L.state == 3) throw Panic("assertion failed: PAF_TAG.is_match(token)");
        if (L.state == 4) throw Panic("Unable to parse cigar string.");
        if (L.state == 1) { paf.skipped++; continue; }
        kept.push_back((uint32_t)k);
        total_cg += L.cg_n;
    }
    const size_t n_ok = kept.size();
    paf.cigar.resize(total_cg);
    paf.cigar_off.resize(n_ok + 1);
    for (std::vector<uint64_t>* v : {&paf.q_len, &paf.q_st, &paf.q_en, &paf.t_len, &paf.t_st, &paf.t_en, &paf.mapq}) v->resize(n_ok);
    paf.strand.resize(n_ok); paf.q_id.resize(n_ok); paf.t_id.resize(n_ok);
    {   // payload offsets (serial additions), then ranges of ~4 MB of payload / 4 096 records for the threads
        size_t off = 0;
        paf.cigar_off[0] = 0;
        for (size_t r = 0; r < n_ok; r++) { off += parsed[kept[r]].cg_n; paf.cigar_off[r + 1] = off; }
    }
    std::vector<size_t> grabs(1, 0);
    for (size_t r = 0, acc = 0, cnt = 0; r < n_ok; r++) {
        acc += parsed[kept[r]].cg_n; cnt++;
        if (acc >= (4u << 20) || cnt >= 4096 || r + 1 == n_ok) { grabs.push_back(r + 1); acc = 0; cnt = 0; }
    }
    auto fill_range = [&](size_t a, size_t b) {  // numeric columns, strand and the CIGAR payload of records [a, b)
        for (size_t r = a; r < b; r++) {
            const ParsedLine& L = parsed[kept[r]];
            paf.q_len[r] = L.v[0]; paf.q_st[r] = L.v[1]; paf.q_en[r] = L.v[2];
            paf.t_len[r] = L.v[3]; paf.t_st[r] = L.v[4]; paf.t_en[r] = L.v[5];
            paf.mapq[r] = L.v[8];
            paf.strand[r] = L.strand;
            if (L.cg_n) memcpy(paf.cigar.data() + paf.cigar_off[r], L.cg, L.cg_n);
        }
    };
    std::vector<std::thread> pool;
    std::atomic<size_t> next{0};
    if (nt > 1 && n_ok >= 2)
        for (unsigned t = 0; t + 1 < nt; t++)
            pool.emplace_back([&] {
                for (;;) {
                    const size_t g = next.fetch_add(1);
                    if (g + 1 >= grabs.size()) break;
                    fill_range(grabs[g], grabs[g + 1]);
                }
            });
    // names meanwhile, on this thread, in file order (ids are handed out by first appearance)
    rbn::intern_record_names(
        n_ok, [&](size_t r) { const ParsedLine& L = parsed[kept[r]]; return std::make_pair(L.q_name, L.q_name_n); },
        [&](size_t r) { const ParsedLine& L = parsed[kept[r]]; return std::make_pair(L.t_name, L.t_name_n); },
        [&](const char* p, size_t len) { return paf.name_id(std::string(p, len)); }, paf.q_id.data(), paf.t_id.data());
    for (;;) {  // ... then it helps with what is left
        const size_t g = next.fetch_add(1);
        if (g + 1 >= grabs.size()) break;
        fill_range(grabs[g], grabs[g + 1]);
    }
    for (auto& th : pool) th.join();
    return paf;
}

// paf.rs:62-78 Paf::from_file.  An uncompressed file is mapped and parsed in place: the lines are only ever read once (the CIGAR
// payloads are copied into the packed buffer by all threads), so a private copy of many GB — allocated, zeroed and filled by one
// thread — would cost more than the parse itself.
Paf Paf::from_file(const std::string& path) {
    auto ends_with = [&](const char* suf) {
        const size_t n = strlen(suf);
        return path.size() >= n && path.compare(path.size() - n, n, suf) == 0;
    };
    if (path != "-" && !ends_with(".gz") && !ends_with(".bgz")) {
        const int fd = ::open(path.c_str(), O_RDONLY);
        if (fd < 0) throw Panic("Error: cannot read input file " + path);
        struct stat st;
        if (fstat(fd, &st) == 0 && S_ISREG(st.st_mode) && st.st_size > 0) {
            void* p = mmap(nullptr, (size_t)st.st_size, PROT_READ, MAP_PRIVATE, fd, 0);
            if (p != MAP_FAILED) {
                madvise(p, (size_t)st.st_size, MADV_WILLNEED);
                try {
                    Paf paf = from_text(static_cast<const char*>(p), (size_t)st.st_size);
                    munmap(p, (size_t)st.st_size);
                    ::close(fd);
                    return paf;
                } catch (...) {
                    munmap(p, (size_t)st.st_size);
                    ::close(fd);
                    throw;
                }
            }
        }
        ::close(fd);
    }
    std::string t = read_all(path);
    return from_text(t.data(), t.size());
}

rb_records Paf::view() {
    names_blob.clear();
    names_off.assign(1, 0);
    for (const std::string& s : names) {
        names_blob.insert(names_blob.end(), s.begin(), s.end());
        names_off.push_back(names_blob.size());
    }
    if (names_blob.empty()) names_blob.push_back(0);
    rb_records r{};
    r.n_rec = (uint32_t)size();
    r.cigar = cigar.data(); r.cigar_nbytes = cigar.size(); r.cigar_off = cigar_off.data();
    r.q_len = q_len.data(); r.q_st = q_st.data(); r.q_en = q_en.data();
    r.t_len = t_len.data(); r.t_st = t_st.data(); r.t_en = t_en.data(); r.mapq = mapq.data();
    r.strand = strand.data(); r.q_id = q_id.data(); r.t_id = t_id.data();
    r.names = names_blob.data(); r.names_off = names_off.data(); r.n_names = (uint32_t)names.size();
    return r;
}

// ---------------------------------------------------------------------------------------------
// BED — bed.rs:140-194 over bio 1.6.0 bed::Reader (csv: tab, '#' comments, fixed field count)
// ---------------------------------------------------------------------------------------------
std::vector<Region> parse_bed_text(const char* text, size_t n) {
    std::vector<Region> out;
    size_t i = 0, nf0 = 0;
    std::vector<std::pair<size_t, size_t>> f;
    while (i < n) {
        size_t j = i;
        while (j < n && text[j] != '\n' && text[j] != '\r') j++;
        const size_t a = i, b = j;
        i = j;
        while (i < n && (text[i] == '\n' || text[i] == '\r')) i++;
        if (a == b || text[a] == '#') continue;
        f.clear();
        size_t p = a;
        for (;;) {
            const char* tab = (const char*)memchr(text + p, '\t', b - p);
            if (!tab) { f.emplace_back(p, b - p); break; }
            f.emplace_back(p, (size_t)(tab - text) - p);
            p = (size_t)(tab - text) + 1;
        }
        if (nf0 == 0) nf0 = f.size();
        else if (f.size() != nf0) continue;
        if (f.size() < 3) continue;
        Region r;
        auto strict = [&](std::pair<size_t, size_t> s, uint64_t& v) {
            if (s.second == 0) return false;
            uint64_t x = 0;
            for (size_t k = 0; k < s.second; k++) {
                const char c = text[s.first + k];
                if (c < '0' || c > '9') return false;
                const uint64_t d = (uint64_t)(c - '0');
                if (x > (UINT64_MAX - d) / 10) return false;
                x = x * 10 + d;
            }
            v = x;
            return true;
        };
        if (!strict(f[1], r.st) || !strict(f[2], r.en)) continue;
        r.name.assign(text + f[0].first, f[0].second);
        if (f.size() > 3) r.id.assign(text + f[3].first, f[3].second);
        else { r.id = r.name + ":" + std::to_string(r.st + 1) + "-" + std::to_string(r.en); r.default_id = true; }  // bed.rs:150-153
        out.push_back(std::move(r));
    }
    return out;
}

Windows Windows::pack(const std::vector<Region>& rgns, const Paf& paf) {
    struct Row { uint32_t t; uint64_t st; uint32_t row; };
    std::vector<Row> rows;
    rows.reserve(rgns.size());
    for (size_t i = 0; i < rgns.size(); i++) {
        const int64_t id = paf.find_name(rgns[i].name);
        if (id < 0) continue;  // BED rows on contigs absent from the PAF are never visited (liftover.rs:151-164)
        rows.push_back(Row{(uint32_t)id, rgns[i].st, (uint32_t)i});
    }
    std::stable_sort(rows.begin(), rows.end(), [](const Row& a, const Row& b) { return a.t != b.t ? a.t < b.t : a.st < b.st; });
    Windows w;
    w.default_ids = true;
    for (const Row& r : rows) w.default_ids = w.default_ids && rgns[r.row].default_id;
    if (!w.default_ids) w.ids_off.push_back(0);
    for (const Row& r : rows) {
        const Region& g = rgns[r.row];
        w.t_id.push_back(r.t); w.st.push_back(g.st); w.en.push_back(g.en); w.bed_row.push_back(r.row);
        if (!w.default_ids) {
            w.ids.insert(w.ids.end(), g.id.begin(), g.id.end());
            w.ids_off.push_back(w.ids.size());
        }
    }
    if (w.ids.empty()) w.ids.push_back(0);
    return w;
}
// parse_bed_text + pack in one pass over the text, without a std::string per row and on all host threads: what `rb liftover`
// does with a 3-million-row BED (1 kb windows: 74 MB of text) before the GPU sees anything.  Same rows, same bed_row numbers
// (position among the rows that parse, whether or not their contig occurs in the PAF), same ids as the two-step form.
Windows Windows::pack_text(const char* text, size_t n, const Paf& paf) {
    // A line ends at \n or \r, runs of them separate lines, lines starting with '#' are comments (bio's bed::Reader over csv).
    // Every thread takes a byte range of the text, starts at the first line that BEGINS in it and parses line by line: no global
    // line table, no serial pass over the text.
    auto is_eol = [](char c) { return c == '\n' || c == '\r'; };
    auto line_end = [&](size_t i) {  // first \n or \r at or after i
        const char* q = (const char*)memchr(text + i, '\n', n - i);
        const size_t e = q ? (size_t)(q - text) : n;
        const char* r = (const char*)memchr(text + i, '\r', e - i);
        return r ? (size_t)(r - text) : e;
    };
    auto n_fields = [&](size_t a, size_t b) {
        size_t c = 1;
        for (const char* p = text + a; (p = (const char*)memchr(p, '\t', (size_t)(text + b - p))) != nullptr; p++) c++;
        return c;
    };
    size_t nf0 = 0;  // the first record fixes the field count
    for (size_t i = 0; i < n;) {
        while (i < n && is_eol(text[i])) i++;
        if (i >= n) break;
        const size_t j = line_end(i);
        if (text[i] != '#') { nf0 = n_fields(i, j); break; }
        i = j;
    }
    struct Row { uint32_t t; uint32_t row; uint64_t st, en; size_t id_at; uint32_t id_n; };
    const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
    const unsigned nt = n < (4u << 20) ? 1u : hw;
    std::vector<std::vector<Row>> part(nt);
    std::vector<size_t> parsed(nt, 0);  // rows of the part that parse (present contig or not): they number the BED rows
    auto work = [&](unsigned t) {
        size_t i = n / nt * t;
        const size_t stop = (t + 1 == nt) ? n : n / nt * (t + 1);
        if (t > 0) {  // a line that began before this range belongs to the thread in front
            if (!is_eol(text[i - 1])) i = line_end(i);
        }
        std::vector<Row>& out = part[t];
        out.reserve((stop - std::min(i, stop)) / 16 + 16);
        const char* last_name = nullptr;
        size_t last_n = 0;
        int64_t last_id = -1;
        size_t k_parsed = 0;
        for (;;) {
            while (i < n && is_eol(text[i])) i++;
            if (i >= stop || i >= n) break;  // (a line is owned by the range its first byte lies in)
            const size_t a = i, b = line_end(i);
            i = b;
            if (text[a] == '#') continue;
            size_t f[5][2];
            size_t nf = 0, p = a;
            for (;;) {  // the first four fields; the rest only counted
                const char* tab = (const char*)memchr(text + p, '\t', b - p);
                const size_t e = tab ? (size_t)(tab - text) : b;
                if (nf < 4) { f[nf][0] = p; f[nf][1] = e - p; }
                nf++;
                if (!tab) break;
                p = e + 1;
            }
            if (nf != nf0 || nf < 3) continue;
            auto strict = [&](size_t at, size_t len, uint64_t& v) {
                if (len == 0) return false;
                uint64_t x = 0;
                for (size_t k = 0; k < len; k++) {
                    const char c = text[at + k];
                    if (c < '0' || c > '9') return false;
                    const uint64_t d = (uint64_t)(c - '0');
                    if (x > (UINT64_MAX - d) / 10) return false;
                    x = x * 10 + d;
                }
                v = x;
                return true;
            };
            Row r{};
            if (!strict(f[1][0], f[1][1], r.st) || !strict(f[2][0], f[2][1], r.en)) continue;
            r.row = (uint32_t)k_parsed++;  // (relative to the part; rebased below)
            if (!(last_name && last_n == f[0][1] && memcmp(last_name, text + f[0][0], last_n) == 0)) {
                last_name = text + f[0][0]; last_n = f[0][1];
                last_id = paf.find_name(std::string(last_name, last_n));
            }
            if (last_id < 0) continue;  // BED rows on contigs absent from the PAF are never visited (liftover.rs:151-164)
            r.t = (uint32_t)last_id;
            if (nf > 3) { r.id_at = f[3][0]; r.id_n = (uint32_t)f[3][1]; }
            out.push_back(r);
        }
        parsed[t] = k_parsed;
    };
    if (nt <= 1) work(0);
    else {
        std::vector<std::thread> pool;
        for (unsigned t = 0; t < nt; t++) pool.emplace_back(work, t);
        for (auto& th : pool) th.join();
    }
    auto less = [](const Row& a, const Row& b) { return a.t != b.t ? a.t < b.t : a.st < b.st; };
    std::vector<size_t> at(nt + 1, 0), base(nt + 1, 0);  // where a part's rows go / what its row numbers start at
    for (unsigned t = 0; t < nt; t++) { at[t + 1] = at[t] + part[t].size(); base[t + 1] = base[t] + parsed[t]; }
    const size_t total = at[nt];
    bool sorted = true;  // (the usual case: bedtools makewindows output) — then the parts are written out where they are
    {
        const Row* prev = nullptr;
        for (unsigned t = 0; t < nt && sorted; t++) {
            if (part[t].empty()) continue;
            if (prev && less(part[t].front(), *prev)) sorted = false;
            if (!std::is_sorted(part[t].begin(), part[t].end(), less)) sorted = false;
            prev = &part[t].back();
        }
    }
    std::vector<Row> rows;
    if (!sorted) {
        rows.reserve(total);
        for (unsigned t = 0; t < nt; t++) {
            for (Row r : part[t]) { r.row += (uint32_t)base[t]; rows.push_back(r); }
            std::vector<Row>().swap(part[t]);
        }
        std::stable_sort(rows.begin(), rows.end(), less);
    }
    Windows w;
    w.default_ids = nf0 <= 3;
    w.t_id.resize(total); w.st.resize(total); w.en.resize(total); w.bed_row.resize(total);
    auto fill = [&](const Row* src, size_t cnt, size_t dst, uint32_t rebase) {
        for (size_t k = 0; k < cnt; k++) {
            const Row& r = src[k];
            w.t_id[dst + k] = r.t; w.st[dst + k] = r.st; w.en[dst + k] = r.en; w.bed_row[dst + k] = r.row + rebase;
        }
    };
    if (!sorted) fill(rows.data(), total, 0, 0u);
    else if (nt <= 1) fill(part[0].data(), part[0].size(), 0, 0u);
    else {
        std::vector<std::thread> pool;
        for (unsigned t = 0; t < nt; t++) pool.emplace_back([&, t] { fill(part[t].data(), part[t].size(), at[t], (uint32_t)base[t]); });
        for (auto& th : pool) th.join();
    }
    if (!w.default_ids) {  // (explicit ids: the byte offsets are a serial prefix sum)
        w.ids_off.push_back(0);
        auto add = [&](const Row& r) {
            w.ids.insert(w.ids.end(), text + r.id_at, text + r.id_at + r.id_n);
            w.ids_off.push_back(w.ids.size());
        };
        if (!sorted) for (const Row& r : rows) add(r);
        else for (unsigned t = 0; t < nt; t++) for (const Row& r : part[t]) add(r);
    }
    if (w.ids.empty()) w.ids.push_back(0);
    return w;
}

rb_windows Windows::view() const {
    rb_windows v{};
    v.n_win = (uint32_t)t_id.size();
    v.t_id = t_id.data(); v.st = st.data(); v.en = en.data(); v.bed_row = bed_row.data();
    v.ids = default_ids ? nullptr : ids.data(); v.ids_off = default_ids ? nullptr : ids_off.data();
    return v;
}

// rows [0, n) formatted by append(out, i) on all host threads, written to `f` in row order
template <class Append>
static void write_rows(FILE* f, size_t n, Append append) {
    const size_t block = 1u << 15;  // rows per work item
    const size_t n_blocks = (n + block - 1) / block;
    const unsigned nt = (unsigned)std::min<size_t>(std::max(1u, std::thread::hardware_concurrency()), std::max<size_t>(1, n_blocks));
    if (nt <= 1) {
        std::string out;
        for (size_t i = 0; i < n; i++) {
            append(out, i);
            if (out.size() > (1u << 20)) { fwrite(out.data(), 1, out.size(), f); out.clear(); }
        }
        fwrite(out.data(), 1, out.size(), f);
        return;
    }
    // waves of nt blocks: formatted in parallel, written in order
    std::vector<std::string> bufs(nt);
    for (size_t b0 = 0; b0 < n_blocks; b0 += nt) {
        const size_t nb = std::min<size_t>(nt, n_blocks - b0);
        std::vector<std::thread> pool;
        for (size_t k = 0; k < nb; k++)
            pool.emplace_back([&, k] {
                std::string& out = bufs[k];
                out.clear();
                const size_t lo = (b0 + k) * block, hi = std::min(n, lo + block);
                for (size_t i = lo; i < hi; i++) append(out, i);
            });
        for (auto& th : pool) th.join();
        for (size_t k = 0; k < nb; k++) fwrite(bufs[k].data(), 1, bufs[k].size(), f);
    }
}

void write_stats_rows(FILE* f, const Paf& paf, const rb_stats_out& st, bool qbed) {
    write_rows(f, paf.size(), [&](std::string& out, size_t i) { append_stats_row(out, paf, i, st, qbed); });
}

// ---------------------------------------------------------------------------------------------
// --largest (host-side post-filter over the rows the GPU produced; needs RB_WANT_TEXT | RB_WANT_NUMERIC)
// ---------------------------------------------------------------------------------------------
std::string largest_rows(const rb_lift_out& out) {
    struct Row { const uint8_t* id; size_t id_n; uint64_t span; uint64_t i; };
    std::vector<Row> rows((size_t)out.n_out);
    for (uint64_t i = 0; i < out.n_out; i++) {
        const uint8_t* ln = out.paf_text + out.line_off[i];
        const uint8_t* end = out.paf_text + out.line_off[i + 1];
        const uint8_t* p = ln;
        for (int tabs = 0; tabs < 12 && p < end; p++) tabs += (*p == '\t');  // 13th column: id:Z:<id>
        const uint8_t* id = p + 5;
        const uint8_t* q = id;
        while (q < end && *q != '\t') q++;
        rows[(size_t)i] = Row{id, (size_t)(q - id), out.t_en[i] - out.t_st[i], i};
    }
    std::stable_sort(rows.begin(), rows.end(), [](const Row& a, const Row& b) {
        const int c = memcmp(a.id, b.id, std::min(a.id_n, b.id_n));
        return c ? c < 0 : a.id_n < b.id_n;
    });
    std::string res;
    size_t i = 0;
    while (i < rows.size()) {
        size_t j = i, best = i;
        while (j < rows.size() && rows[j].id_n == rows[i].id_n && memcmp(rows[j].id, rows[i].id, rows[i].id_n) == 0) {
            if (rows[j].span >= rows[best].span) best = j;  // max_by_key keeps the last maximum
            j++;
        }
        const uint64_t k = rows[best].i;
        res.append(reinterpret_cast<const char*>(out.paf_text + out.line_off[k]), (size_t)(out.line_off[k + 1] - out.line_off[k]));
        i = j;
    }
    return res;
}

// ---------------------------------------------------------------------------------------------
// printing
// ---------------------------------------------------------------------------------------------
std::string fmt_f32(float v) {
    // Rust's `{}` for f32: shortest round-trip digits, closest to the value, an exact tie rounded UP (flt2dec's Dragon; Ryu /
    // std::to_chars round such ties to even): std::to_chars unless the value is exactly such a tie, then csrc/f32_fmt.cuh
    return f32_display_fast(v);
}

std::string stats_header(bool qbed) {
    std::string s = qbed ? "#query_name\tquery_start\tquery_end\tquery_length\tstrand\treference_name\treference_start\treference_end\treference_length\t"
                         : "#reference_name\treference_start\treference_end\treference_length\tstrand\tquery_name\tquery_start\tquery_end\tquery_length\t";
    s += "perID_by_matches\tperID_by_events\tperID_by_all\tmatches\tmismatches\tdeletion_events\tinsertion_events\tdeletions\tinsertions\n";
    return s;
}

void append_row(std::string& s, const std::string& q_name, const std::string& t_name, uint8_t strand, uint64_t q_st, uint64_t q_en,
                uint64_t q_len, uint64_t t_st, uint64_t t_en, uint64_t t_len, const rb_stats_out& st, size_t i, bool qbed) {
    auto q = [&] {
        s += q_name; s += '\t'; s += std::to_string((int64_t)q_st); s += '\t';
        s += std::to_string((int64_t)q_en); s += '\t'; s += std::to_string((int64_t)q_len); s += '\t';
    };
    auto r = [&] {
        s += t_name; s += '\t'; s += std::to_string((int64_t)t_st); s += '\t';
        s += std::to_string((int64_t)t_en); s += '\t'; s += std::to_string((int64_t)t_len); s += '\t';
    };
    if (qbed) { q(); s += (char)strand; s += '\t'; r(); }
    else { r(); s += (char)strand; s += '\t'; q(); }
    s += fmt_f32(st.id_by_matches[i]); s += '\t';
    s += fmt_f32(st.id_by_events[i]); s += '\t';
    s += fmt_f32(st.id_by_all[i]); s += '\t';
    s += std::to_string(st.equal[i]); s += '\t';
    s += std::to_string(st.diff[i]); s += '\t';
    s += std::to_string(st.del_events[i]); s += '\t';
    s += std::to_string(st.ins_events[i]); s += '\t';
    s += std::to_string(st.del[i]); s += '\t';
    s += std::to_string(st.ins[i]); s += '\n';
}

void append_stats_row(std::string& s, const Paf& paf, size_t i, const rb_stats_out& st, bool qbed) {
    append_row(s, paf.names[paf.q_id[i]], paf.names[paf.t_id[i]], paf.strand[i], paf.q_st[i], paf.q_en[i], paf.q_len[i], paf.t_st[i],
               paf.t_en[i], paf.t_len[i], st, i, qbed);
}

std::string paf_text(const Paf& paf, size_t lo, size_t hi) {
    std::string s;
    for (size_t i = lo; i < hi && i < paf.size(); i++) {
        s += paf.names[paf.q_id[i]]; s += '\t';
        s += std::to_string(paf.q_len[i]); s += '\t'; s += std::to_string(paf.q_st[i]); s += '\t';
        s += std::to_string(paf.q_en[i]); s += '\t'; s += (char)paf.strand[i]; s += '\t';
        s += paf.names[paf.t_id[i]]; s += '\t';
        s += std::to_string(paf.t_len[i]); s += '\t'; s += std::to_string(paf.t_st[i]); s += '\t';
        s += std::to_string(paf.t_en[i]); s += "\t0\t0\t"; s += std::to_string(paf.mapq[i]);
        s += "\tcg:Z:";
        s.append((const char*)paf.cigar.data() + paf.cigar_off[i], paf.cigar_off[i + 1] - paf.cigar_off[i]);
        s += '\n';
    }
    return s;
}

std::string bed_text(const std::vector<Region>& rgns, bool with_ids) {
    std::string s;
    for (const Region& r : rgns) {
        s += r.name; s += '\t'; s += std::to_string(r.st); s += '\t'; s += std::to_string(r.en);
        if (with_ids) { s += '\t'; s += r.id; }
        s += '\n';
    }
    return s;
}

}  // namespace rbh
