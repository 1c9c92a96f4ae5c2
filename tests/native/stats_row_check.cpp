// Fuzzes rb::stats_row_len / rb::stats_row_put (csrc/stats_row.cuh, the row composer of k_stats_rows) against the host formatter
// rbh::append_row: random names (1 byte to 3 KB), coordinates up to u64 max (>= 2^63 prints negative, as the reference's i64 does),
// digit-count edges, random counters, identities from random bits in [0, 100], from random counters as bamstats.rs computes them,
// exact decimal ties (found by comparing the composer's digits with std::to_chars, which rounds ties to even), NaN, 0 and 100,
// both strands and both column orders.  stats_row_len must equal the bytes stats_row_put writes.
//     stats_row_check <seed> <cases>   -> "cases=.. ties=.. long_names=.. negative=.. FAIL=n"
#include <charconv>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>
#include <string>
#include <vector>

#include "rbhost.hpp"
#include "stats_row.cuh"

static uint32_t bits_of(float v) { uint32_t b; memcpy(&b, &v, 4); return b; }
static float float_of(uint32_t b) { float v; memcpy(&v, &b, 4); return v; }

static std::string core_digits(float v) {
    uint8_t buf[96];
    return std::string((const char*)buf, (size_t)rb::f32_display(v, buf));
}
static std::string to_chars_digits(float v) {
    char buf[128];
    auto r = std::to_chars(buf, buf + sizeof buf, v, std::chars_format::fixed);
    return std::string(buf, r.ptr);
}

int main(int argc, char** argv) {
    const uint64_t seed = argc > 1 ? strtoull(argv[1], nullptr, 10) : 1;
    const uint64_t cases = argc > 2 ? strtoull(argv[2], nullptr, 10) : 10000;
    std::mt19937_64 rng(seed);
    auto below = [&](uint64_t n) { return n ? rng() % n : 0; };

    // exact ties in [0, 100]: dyadic values i / 2^k whose shortest digits round up where std::to_chars rounds to even
    std::vector<uint32_t> ties;
    for (int k = 5; k <= 12; k++)
        for (uint32_t i = 1; i <= (100u << k); i++) {
            const float v = std::ldexp((float)i, -k);
            if (core_digits(v) != to_chars_digits(v)) ties.push_back(bits_of(v));
        }

    auto rand_u64 = [&]() -> uint64_t {
        switch (below(6)) {
            case 0: return below(1000);
            case 1: return rng();                                     // anything, half of them >= 2^63
            case 2: { uint64_t p = 1; for (uint64_t e = below(20); e; e--) p *= 10; return p - below(2); }  // 10^k and 10^k - 1
            case 3: return UINT64_MAX - below(3);
            case 4: return (1ull << 63) - 1 + below(3);               // around i64 max
            default: return below(1ull << 32);
        }
    };
    auto rand_u32 = [&]() -> uint32_t {
        switch (below(4)) {
            case 0: return (uint32_t)below(100);
            case 1: return (uint32_t)rng();
            case 2: return UINT32_MAX - (uint32_t)below(2);
            default: return (uint32_t)below(1u << 20);
        }
    };
    auto rand_name = [&](bool& long_name) {
        const uint64_t len = below(50) == 0 ? 1000 + below(2200) : 1 + below(40);
        long_name = len >= 1000;
        std::string s(len, 'a');
        for (char& c : s) c = (char)(33 + below(94));  // printable, no tab / newline
        return s;
    };
    auto rand_id = [&](uint32_t eq, uint32_t tot) -> uint32_t {
        switch (below(8)) {
            case 0: return (uint32_t)below(0x42C80001u);                                  // random bits in [0, 100]
            case 1: return ties.empty() ? 0u : ties[below(ties.size())];                 // exact ties
            case 2: return bits_of(std::nanf(""));
            case 3: return below(2) ? 0u : bits_of(100.0f);
            default: {                                                                   // bamstats.rs:138-142: 100 * equal / total
                volatile float num = 100.0f * (float)eq;
                volatile float q = num / (float)tot;
                return bits_of(q);
            }
        }
    };

    uint64_t fails = 0, n_ties = 0, n_long = 0, n_neg = 0, n_bytes = 0;
    std::vector<uint8_t> buf;
    for (uint64_t c = 0; c < cases; c++) {
        bool lq = false, lt = false;
        const std::string qn = rand_name(lq), tn = rand_name(lt);
        rb::StatsRow r;
        r.q_name = reinterpret_cast<const uint8_t*>(qn.data()); r.q_name_len = (uint32_t)qn.size();
        r.t_name = reinterpret_cast<const uint8_t*>(tn.data()); r.t_name_len = (uint32_t)tn.size();
        r.q_st = rand_u64(); r.q_en = rand_u64(); r.q_len = rand_u64(); r.t_st = rand_u64(); r.t_en = rand_u64(); r.t_len = rand_u64();
        r.strand = below(2) ? '+' : '-';
        r.equal = rand_u32(); r.diff = rand_u32(); r.ins = rand_u32(); r.del = rand_u32();
        r.ins_events = rand_u32(); r.del_events = rand_u32(); r.matches = rand_u32();
        const uint32_t tot = (uint32_t)(below(3) == 0 ? r.equal : r.equal + r.diff);
        for (int k = 0; k < 3; k++) r.id_bits[k] = rand_id(r.equal, tot);
        rb::stats_row_digits(r);
        const bool qbed = below(2) != 0;
        for (int k = 0; k < 3; k++)
            for (uint32_t t : ties) if (t == r.id_bits[k]) { n_ties++; break; }
        n_long += (lq || lt);
        for (uint64_t v : {r.q_st, r.q_en, r.q_len, r.t_st, r.t_en, r.t_len}) n_neg += (int64_t)v < 0;

        uint32_t eq[1] = {r.equal}, df[1] = {r.diff}, in[1] = {r.ins}, dl[1] = {r.del}, ie[1] = {r.ins_events}, de[1] = {r.del_events},
                 mt[1] = {r.matches};
        float im[1] = {float_of(r.id_bits[0])}, iv[1] = {float_of(r.id_bits[1])}, ia[1] = {float_of(r.id_bits[2])};
        rb_stats_out st{};
        st.n = 1; st.equal = eq; st.diff = df; st.ins = in; st.del = dl; st.ins_events = ie; st.del_events = de; st.matches = mt;
        st.id_by_matches = im; st.id_by_events = iv; st.id_by_all = ia;
        std::string want;
        rbh::append_row(want, qn, tn, r.strand, r.q_st, r.q_en, r.q_len, r.t_st, r.t_en, r.t_len, st, 0, qbed);

        const uint32_t len = rb::stats_row_len(r);
        buf.assign((size_t)len + 64, 0xEE);
        const uint8_t* end = rb::stats_row_put(buf.data(), r, qbed);
        const std::string got(reinterpret_cast<const char*>(buf.data()), (size_t)(end - buf.data()));
        n_bytes += got.size();
        if (got != want || got.size() != len || buf[len] != 0xEE) {
            if (fails < 5)
                fprintf(stderr, "FAIL case %llu (qbed %d, len %u, wrote %zu):\n  want %s  got  %s\n", (unsigned long long)c, (int)qbed, len,
                        got.size(), want.c_str(), got.c_str());
            fails++;
        }
    }
    printf("cases=%llu bytes=%llu ties=%llu tie_values=%zu long_names=%llu negative=%llu FAIL=%llu\n", (unsigned long long)cases,
           (unsigned long long)n_bytes, (unsigned long long)n_ties, ties.size(), (unsigned long long)n_long, (unsigned long long)n_neg,
           (unsigned long long)fails);
    return fails ? 1 : 0;
}
