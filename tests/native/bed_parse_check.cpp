// The __host__ __device__ line rules of csrc/bed_parse_core.cuh, driven the way bed_parse_kernels.cu drives them (line starts,
// one bed_line per line, the first non-comment line's field count, row_parses, a name lookup, bed_row / window numbering, a stable
// sort by (t_id, st)), against the host packer rbh::Windows::pack_text on the same seeded random BED texts: t_id, st, en,
// bed_row, ids, the parsed-row count (parse_bed_text) and the field count.
//   bed_parse_check <seed> <n_lines>      prints "lines=.. kept=.. skipped=.. absent=.. comments=.. files=.. FAIL=<count>"
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>
#include <string>
#include <unordered_map>
#include <vector>

#include "bed_parse_core.cuh"
#include "rbhost.hpp"

namespace {

std::mt19937_64 rng;
uint64_t rnd(uint64_t n) { return n ? rng() % n : 0; }

const char* const TARGETS[] = {"chr1", "chr2", "chr3", "chrX", "ctg 7"};
const char* const QUERIES[] = {"q1", "read/2", "hap1#chr1"};  // in the name table as query names only
const char* const ABSENT[] = {"chrUn", "chr", "chr11", "Chr1", ""};

std::string num() {
    switch (rnd(14)) {
        case 0: return "+5";
        case 1: return "";
        case 2: return " 12";
        case 3: return "12 ";
        case 4: return "18446744073709551615";   // u64::MAX
        case 5: return "18446744073709551616";   // overflows
        case 6: return "99999999999999999999";   // 20 digits, overflows
        case 7: return "00000000000000000000042";
        case 8: return "-3";
        case 9: return "1e3";
        default: return std::to_string(rnd(100000));
    }
}

std::string name() {
    const uint64_t k = rnd(20);
    if (k < 13) return TARGETS[rnd(5)];
    if (k < 16) return QUERIES[rnd(3)];
    return ABSENT[rnd(5)];
}

std::string eol() {
    switch (rnd(10)) {
        case 0: return "\r\n";
        case 1: return "\r";
        case 2: return "\n\n\n";
        case 3: return "\r\n\r\n\n";
        default: return "\n";
    }
}

// one BED file: nf fields per row, with quirks
std::string bed_file(long n_lines, int nf, std::vector<std::string>& rows_seen) {
    std::string t;
    if (rnd(4) == 0) t += rnd(2) ? "\n\r\n" : "\r";                  // leading line ends
    if (rnd(6) == 0) t += "track name=x" + eol();                     // a 1-field header: fixes the field count to 1
    else if (rnd(6) == 0) t += "browser\tposition\tchr1:1-100\textra\textra2" + eol();  // a 5-field header line that does not parse
    std::string prev;
    for (long i = 0; i < n_lines; i++) {
        std::string l;
        const uint64_t k = rnd(60);
        if (k == 0) l = "#comment\twith\ttabs";
        else if (k == 1) l = "#";
        else if (k == 2 && !prev.empty()) l = prev;                   // a duplicate row
        else {
            int f = nf;
            if (rnd(25) == 0) f = (int)(2 + rnd(4));                   // 2 / 3 / 4 / 5 fields
            std::vector<std::string> c;
            c.push_back(name());
            c.push_back(rnd(10) ? std::to_string(rnd(100000)) : num());
            c.push_back(rnd(10) ? std::to_string(rnd(100000)) : num());
            if (f > 3) c.push_back(rnd(10) == 0 ? std::string() : rnd(8) == 0 ? "id with spaces" : "w" + std::to_string(rnd(1000)));
            while ((int)c.size() < f) c.push_back(rnd(3) ? "+" : "");
            for (int j = 0; j < f; j++) l += (j ? "\t" : "") + c[(size_t)j];
            if (rnd(40) == 0) l += "\t";                               // a trailing empty field
        }
        prev = l;
        rows_seen.push_back(l);
        t += l;
        if (i + 1 < n_lines || rnd(2)) t += eol();                    // with and without a final line end
    }
    return t;
}

struct Row { uint32_t t; uint64_t st, en; uint32_t row; uint64_t id_off, id_len; };

}  // namespace

int main(int argc, char** argv) {
    rng.seed(argc > 1 ? strtoull(argv[1], nullptr, 10) : 1);
    const long n = argc > 2 ? atol(argv[2]) : 1000;
    rbh::Paf paf;  // the batch's name table: query and target names
    for (const char* q : QUERIES) paf.name_id(q);
    for (const char* c : TARGETS) paf.name_id(c);
    std::unordered_map<std::string, uint32_t> index;
    for (size_t i = 0; i < paf.names.size(); i++) index.emplace(paf.names[i], (uint32_t)i);
    long fails = 0, kept = 0, skipped = 0, absent = 0, comments = 0, files = 0, lines = 0;
    auto bad = [&](long f, const char* what) {
        if (fails++ < 20) printf("FAIL file %ld: %s\n", f, what);
    };
    while (lines < n) {
        const int nf = (int)(3 + rnd(3));
        const long nl = std::min<long>(n - lines, 1 + (long)rnd(3000));
        std::vector<std::string> seen;
        const std::string text = bed_file(nl, nf, seen);
        lines += nl;
        files++;
        const uint8_t* tx = reinterpret_cast<const uint8_t*>(text.data());
        const uint64_t tn = text.size();
        // line starts (k_paf_lines_count / _fill, LINES_BED), one bed_line each (k_bed_fields)
        std::vector<uint64_t> starts;
        for (uint64_t p = 0; p < tn; p++)
            if (!rbbp::is_eol(tx[p]) && (p == 0 || rbbp::is_eol(tx[p - 1]))) starts.push_back(p);
        std::vector<rbbp::BedLine> L(starts.size());
        uint64_t first = UINT64_MAX;
        for (size_t i = 0; i < starts.size(); i++) {
            uint64_t b = starts[i];
            while (b < tn && !rbbp::is_eol(tx[b])) b++;
            rbbp::bed_line(tx, starts[i], b, L[i]);
            if (!L[i].comment) first = std::min<uint64_t>(first, i);
        }
        // k_bed_judge + scans + k_bed_compact
        const uint64_t nf0 = first < L.size() ? L[first].n_fields : 0;
        std::vector<Row> rows;
        uint32_t n_parsed = 0;
        for (size_t i = 0; i < L.size(); i++) {
            if (L[i].comment) { comments++; continue; }
            if (!rbbp::row_parses(L[i], nf0)) { skipped++; continue; }
            const uint32_t row = n_parsed++;
            const auto it = index.find(std::string(text, starts[i], L[i].name_len));
            if (it == index.end()) { absent++; continue; }
            kept++;
            rows.push_back(Row{it->second, L[i].st, L[i].en, row, L[i].id_off, L[i].id_len});
        }
        std::stable_sort(rows.begin(), rows.end(), [](const Row& a, const Row& b) { return a.t != b.t ? a.t < b.t : a.st < b.st; });
        // the host packer on the same text
        const rbh::Windows w = rbh::Windows::pack_text(text.data(), text.size(), paf);
        if (w.t_id.size() != rows.size()) { bad(files, "row count"); continue; }
        if (rbh::parse_bed_text(text.data(), text.size()).size() != n_parsed) bad(files, "n_parsed");
        // the field count of the first non-comment line, split the plain way
        uint64_t want_nf = 0;
        for (size_t p = 0; p < text.size();) {
            while (p < text.size() && (text[p] == '\n' || text[p] == '\r')) p++;
            if (p >= text.size()) break;
            size_t q = p;
            while (q < text.size() && text[q] != '\n' && text[q] != '\r') q++;
            if (text[p] != '#') { want_nf = 1 + (uint64_t)std::count(text.begin() + (long)p, text.begin() + (long)q, '\t'); break; }
            p = q;
        }
        if (want_nf != nf0) bad(files, "n_fields");
        if (w.default_ids != (nf0 <= 3)) bad(files, "default ids");
        uint64_t id_at = 0;
        for (size_t k = 0; k < rows.size(); k++) {
            const Row& r = rows[k];
            if (w.t_id[k] != r.t || w.st[k] != r.st || w.en[k] != r.en || w.bed_row[k] != r.row) { bad(files, "row"); break; }
            if (!w.default_ids) {
                const uint64_t len = w.ids_off[k + 1] - w.ids_off[k];
                if (len != r.id_len || memcmp(w.ids.data() + id_at, text.data() + r.id_off, len) != 0) { bad(files, "id"); break; }
                id_at += len;
            }
        }
    }
    printf("lines=%ld kept=%ld skipped=%ld absent=%ld comments=%ld files=%ld FAIL=%ld\n", lines, kept, skipped, absent, comments, files, fails);
    return fails ? 1 : 0;
}
