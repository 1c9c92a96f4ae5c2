// Fuzzes rbt::plan_line_split (csrc/text_split.hpp) against a direct split of random byte strings: the text is cut into 1-9 ranges
// (some empty), each range reports its first '\n' as the device kernel does, and the planned buffers must hold every line of the
// text exactly once, whole and in order, each on the device whose range holds its first byte.  Seeded cases: ranges without a newline, one line across several ranges, a newline as the
// first or last byte of a range, runs of empty lines, no final newline, empty text.
//     text_split_check <seed> <cases>   -> "cases=.. lines=.. FAIL=n"
#include <cstdio>
#include <algorithm>
#include <cstdlib>
#include <random>
#include <string>
#include <vector>

#include "text_split.hpp"

static std::vector<std::string> lines_of(const std::string& t) {  // each line with its '\n'; a last line without one as it is
    std::vector<std::string> v;
    size_t at = 0;
    while (at < t.size()) {
        const size_t e = t.find('\n', at);
        const size_t end = e == std::string::npos ? t.size() : e + 1;
        v.push_back(t.substr(at, end - at));
        at = end;
    }
    return v;
}

static int fails = 0;
static uint64_t n_lines = 0;

static void check(const std::string& text, const std::vector<uint64_t>& cut, const char* what) {
    const int D = (int)cut.size() - 1;
    std::vector<uint64_t> size((size_t)D), nl((size_t)D);
    std::vector<uint8_t> ends_nl((size_t)D);
    for (int d = 0; d < D; d++) {
        size[(size_t)d] = cut[(size_t)d + 1] - cut[(size_t)d];
        ends_nl[(size_t)d] = size[(size_t)d] && text[cut[(size_t)d + 1] - 1] == '\n';
        const size_t p = text.find('\n', cut[(size_t)d]);
        nl[(size_t)d] = (p != std::string::npos && p < cut[(size_t)d + 1]) ? p - cut[(size_t)d] : rbt::NO_NEWLINE;
    }
    const std::vector<rbt::Owned> own = rbt::plan_line_split(size, nl, ends_nl);
    std::string all;
    std::vector<std::string> got;
    int last_nonempty = -1;
    for (int d = 0; d < D; d++) {
        std::string buf;
        for (const rbt::Piece& p : own[(size_t)d].pieces) {
            if (p.src < 0 || p.src >= D || p.off + p.len > size[(size_t)p.src]) { fails++; printf("FAIL %s: piece out of range\n", what); return; }
            buf += text.substr(cut[(size_t)p.src] + p.off, p.len);
        }
        if (buf.size() != own[(size_t)d].bytes) { fails++; printf("FAIL %s: byte count\n", what); return; }
        if (!buf.empty()) last_nonempty = d;
        // every line of the buffer starts inside range d (the ownership rule)
        const uint64_t g0 = all.size();
        for (size_t i = 0; i < buf.size(); i++)
            if ((i == 0 || buf[i - 1] == '\n') && (g0 + i < cut[(size_t)d] || g0 + i >= cut[(size_t)d + 1])) {
                fails++; printf("FAIL %s: device %d holds a line that starts at %llu, outside its range\n", what, d, (unsigned long long)(g0 + i));
                return;
            }
        // every buffer starts at a line start of the text
        if (!buf.empty() && all.size() && all.back() != '\n') { fails++; printf("FAIL %s: device %d starts inside a line\n", what, d); return; }
        all += buf;
        for (const std::string& l : lines_of(buf)) got.push_back(l);
    }
    for (int d = 0; d < last_nonempty; d++) {  // (a buffer that ends without '\n' must be the last one with bytes)
        std::string buf;
        for (const rbt::Piece& p : own[(size_t)d].pieces) buf += text.substr(cut[(size_t)p.src] + p.off, p.len);
        if (!buf.empty() && buf.back() != '\n') { fails++; printf("FAIL %s: device %d cuts a line\n", what, d); return; }
    }
    if (all != text) { fails++; printf("FAIL %s: buffers do not concatenate to the text\n", what); return; }
    const std::vector<std::string> want = lines_of(text);
    if (got != want) { fails++; printf("FAIL %s: lines differ (%zu vs %zu)\n", what, got.size(), want.size()); return; }
    n_lines += want.size();
}

static std::vector<uint64_t> equal_cuts(uint64_t n, int D) {
    std::vector<uint64_t> c;
    for (int d = 0; d <= D; d++) c.push_back(n * (uint64_t)d / (uint64_t)D);
    return c;
}

int main(int argc, char** argv) {
    const unsigned seed = argc > 1 ? (unsigned)atoi(argv[1]) : 1;
    const int cases = argc > 2 ? atoi(argv[2]) : 1000;
    int done = 0;
    // seeded shapes
    const std::string fixed[] = {"", "\n", "\n\n\n\n", "abc", "abc\n", "a\nb", "a\n\n\nb\n", "0123456789abcdefghij",
                                 std::string(40, 'x') + "\n" + "y\n", "a\nb\nc\nd\ne\nf\ng\nh\ni\n"};
    for (const std::string& t : fixed)
        for (int D = 1; D <= 9; D++) {
            check(t, equal_cuts(t.size(), D), "fixed");
            done++;
            for (uint64_t i = 0; i <= t.size(); i++) {  // one cut anywhere, the other ranges empty at either end
                std::vector<uint64_t> c(1, 0);
                for (int d = 1; d < D; d++) c.push_back(d <= D / 2 ? i : t.size());
                c.push_back(t.size());
                for (size_t k = 1; k < c.size(); k++) if (c[k] < c[k - 1]) c[k] = c[k - 1];
                check(t, c, "one-cut");
                done++;
            }
        }
    // a newline as the first / last byte of a range
    {
        const std::string t = "aaaa\nbbbb\ncccc\n";
        check(t, {0, 5, 10, 15}, "nl-last");
        check(t, {0, 4, 9, 14, 15}, "nl-first");
        check(t, {0, 4, 5, 9, 10, 15}, "nl-alone");
        done += 3;
    }
    std::mt19937_64 rng(seed);
    for (int c = 0; c < cases; c++) {
        const int mode = (int)(rng() % 4);
        const size_t n = (size_t)(rng() % (mode == 3 ? 400 : 80));
        const unsigned nl_per_mille = mode == 0 ? 20u : mode == 1 ? 300u : mode == 2 ? 900u : 5u;  // sparse / dense / empty-line runs / long lines
        std::string t(n, 'a');
        for (size_t i = 0; i < n; i++) {
            if (rng() % 1000 < nl_per_mille) t[i] = '\n';
            else t[i] = (char)('a' + rng() % 3);
        }
        if (rng() % 2 && n) t[n - 1] = '\n';
        const int D = 1 + (int)(rng() % 9);
        std::vector<uint64_t> cut;
        if (rng() % 3 == 0) cut = equal_cuts(n, D);
        else {
            cut.push_back(0);
            for (int d = 1; d < D; d++) cut.push_back(rng() % (n + 1));
            cut.push_back(n);
            std::sort(cut.begin() + 1, cut.end() - 1);
        }
        check(t, cut, "random");
        done++;
    }
    printf("cases=%d lines=%llu FAIL=%d\n", done, (unsigned long long)n_lines, fails);
    return fails ? 1 : 0;
}
