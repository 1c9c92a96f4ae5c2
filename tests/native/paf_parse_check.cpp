// The __host__ __device__ line rules of csrc/paf_parse_core.cuh (what k_paf_fields applies on the GPU) against the host reader,
// rbh::Paf::from_text, over seeded random and mutated PAF lines: kept columns, names and cg payload, every skip and every panic.
//   paf_parse_check <seed> <n_lines>      prints "lines=.. kept=.. skipped=.. panics=.. FAIL=<count>"
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>
#include <string>
#include <vector>

#include "paf_parse_core.cuh"
#include "rbhost.hpp"

namespace {

std::mt19937_64 rng;
uint64_t rnd(uint64_t n) { return n ? rng() % n : 0; }

std::string num() {
    switch (rnd(12)) {
        case 0: return "+17";
        case 1: return "18446744073709551615";          // u64::MAX
        case 2: return "18446744073709551616";          // overflows
        case 3: return "99999999999999999999";          // 20 digits, overflows
        case 4: return "00000000000000000000000042";    // leading zeros
        case 5: return "1x";
        case 6: return "+";
        case 7: return "-3";
        default: return std::to_string(rnd(1000000));
    }
}
std::string cigar() {
    static const char ops[] = "MIDX=NSHP";
    std::string s;
    const int n = (int)rnd(6);
    for (int i = 0; i < n; i++) { s += std::to_string(1 + rnd(500)); s += ops[rnd(rnd(3) ? 5 : 9)]; }
    if (rnd(10) == 0) s += "12";                        // ends in a number
    if (rnd(12) == 0) s = "5M" + std::string("3H") + "4M";  // H in the middle
    if (rnd(15) == 0) s += "99999999999M";              // op length beyond u32
    return s;
}
std::string sep() {
    if (rnd(6)) return "\t";
    static const char ws[] = " \t\x0C";
    std::string s;
    const int n = 1 + (int)rnd(4);
    for (int i = 0; i < n; i++) s += ws[rnd(3)];
    return s;
}

std::string line() {
    std::vector<std::string> t;
    static const char* names[] = {"q1", "q2", "chr1", "contig_7", "read/1", "x"};
    t.push_back(names[rnd(6)]);
    for (int k = 0; k < 3; k++) t.push_back(rnd(8) ? std::to_string(rnd(100000)) : num());
    t.push_back(rnd(20) ? (rnd(2) ? "+" : "-") : (rnd(2) ? "+-" : "."));
    t.push_back(names[rnd(6)]);
    for (int k = 0; k < 6; k++) t.push_back(rnd(8) ? std::to_string(rnd(100000)) : num());
    const int ntags = (int)rnd(4);
    bool cg = false;
    for (int k = 0; k < ntags; k++) {
        switch (rnd(8)) {
            case 0: t.push_back("NM:i:" + std::to_string(rnd(50))); break;
            case 1: t.push_back("cs:Z::10*ag:5+tt"); break;
            case 2: t.push_back("xxcg:Z:" + cigar()); break;   // a prefixed cg tag is a cg tag
            case 3: t.push_back("notatag"); break;
            case 4: t.push_back("cg:Z:"); break;               // empty payload: a later cg replaces it
            case 5: t.push_back("ab:c:d"); break;              // too short to match
            default: t.push_back("cg:Z:" + cigar()); cg = true; break;
        }
    }
    if (!cg && rnd(4)) t.push_back("cg:Z:" + cigar());
    if (rnd(15) == 0) t.erase(t.begin() + (long)rnd(12));  // 11 columns
    if (rnd(30) == 0) t.resize(rnd(4));
    std::string s = rnd(20) ? "" : sep();
    for (size_t i = 0; i < t.size(); i++) {
        if (i) s += sep();
        s += t[i];
    }
    if (rnd(15) == 0) s.insert(rnd(s.size() + 1), "\x0C");  // a stray form feed anywhere
    if (rnd(10) == 0) s += sep();
    if (rnd(8) == 0) s += "\r";
    if (rnd(40) == 0) s.clear();  // an empty line
    return s;
}

}  // namespace

int main(int argc, char** argv) {
    rng.seed(argc > 1 ? strtoull(argv[1], nullptr, 10) : 1);
    const long n = argc > 2 ? atol(argv[2]) : 1000;
    long fails = 0, kept = 0, skipped = 0, panics = 0;
    auto bad = [&](long i, const std::string& l, const char* what) {
        if (fails++ < 20) printf("FAIL line %ld (%s): [%s]\n", i, what, l.c_str());
    };
    std::string file;
    std::vector<rbpp::LineOut> outs;
    std::vector<std::string> lines;
    for (long i = 0; i < n; i++) {
        const std::string l = line();
        const std::string text = l + (rnd(2) || l.empty() ? "\n" : "");  // with and without a terminator (no byte at all is no line)
        // the host reader on this one line
        int host_state = 0;
        rbh::Paf paf;
        try {
            paf = rbh::Paf::from_text(text.data(), text.size());
            host_state = paf.skipped ? 1 : 0;
        } catch (const rbh::Panic& e) {
            const std::string m = e.what();
            host_state = m.find("t.len() >= 12") != std::string::npos ? 2 : m.find("PAF_TAG") != std::string::npos ? 3 : 4;
        }
        // the shared core: line split as k_paf_lines / k_paf_fields do it
        uint64_t e = l.size();
        if (e > 0 && l[e - 1] == '\r') e--;
        rbpp::LineOut o;
        rbpp::parse_line_serial(reinterpret_cast<const uint8_t*>(l.data()), 0, e, o);
        if (o.state != host_state) { bad(i, l, "state"); continue; }
        if (o.state >= 2) { panics++; continue; }
        if (o.state == 1) { skipped++; continue; }
        kept++;
        if (paf.size() != 1) { bad(i, l, "record count"); continue; }
        const uint64_t want[7] = {paf.q_len[0], paf.q_st[0], paf.q_en[0], paf.t_len[0], paf.t_st[0], paf.t_en[0], paf.mapq[0]};
        for (int k = 0; k < 7; k++)
            if (o.v[k] != want[k]) { bad(i, l, "column"); break; }
        if (o.strand != paf.strand[0]) bad(i, l, "strand");
        if (l.substr(o.qn_off, o.qn_len) != paf.names[paf.q_id[0]] || l.substr(o.tn_off, o.tn_len) != paf.names[paf.t_id[0]]) bad(i, l, "names");
        const std::string cg(reinterpret_cast<const char*>(paf.cigar.data()), paf.cigar.size());
        if (l.substr(o.cg_off, o.cg_len) != cg) bad(i, l, "cg");
        if (o.state == 0) { file += l + "\n"; lines.push_back(l); outs.push_back(o); }
    }
    // the kept lines as one file, the last one once more without a terminator: the same records
    file += lines.empty() ? std::string() : lines.back();
    const rbh::Paf all = rbh::Paf::from_text(file.data(), file.size());
    if (all.size() != outs.size() + (lines.empty() ? 0 : 1) || all.skipped != 0) { fails++; printf("FAIL file: %zu records\n", all.size()); }
    printf("lines=%ld kept=%ld skipped=%ld panics=%ld FAIL=%ld\n", n, kept, skipped, panics, fails);
    return fails ? 1 : 0;
}
