// rb — the host CLI for the two subcommands on the hot path, same flags as the reference
// (src/cli.rs:16-27,49-60,100-115; drivers src/main.rs:50-58,186-214):
//     rb [-t N] [--gpus G] liftover --bed <BED> [--qbed] [--largest] [PAF|-]  (alias lo, cli.rs visible_aliases; --qbed: inversion on the
//                                                          GPU; --largest: host filter; --gpus G: spread the records over G B200s)
//                                                          --stats: print the rows `| rb stats --paf` would print — formatted on the GPU)
//     rb [-t N] stats --paf [--qbed] [PAF|-]
//     rb [-t N] break-paf [--max-size N] [PAF|-]        (aliases breakpaf, bp; src/cli.rs:155-165, main.rs:271-281)
//     rb [-t N] invert [PAF|-]                          (src/cli.rs:89-94, main.rs:176-182)
//     rb [-t N] trim-paf [-m M] [-d D] [-i I] [-r] [PAF|-]   (aliases trim, tp; src/cli.rs:117-138, main.rs:218-230)
// Text (plain / .gz / .bgz / stdin) is read and split on the host; CIGAR tokenising, liftover,
// trimming, serialisation and identity counting run on the B200 through include/rbcuda.h.
// Exit status 101 where the reference panics.  There is no CPU fallback: without an sm_100
// device the program fails.
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>

#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include "rbhost.hpp"

static int usage() {
    fprintf(stderr, "usage: rb [-t N] [--gpus G] liftover --bed <BED> [PAF]\n       rb [-t N] stats --paf [--qbed] [PAF]\n"
                    "       rb [-t N] break-paf [--max-size N] [PAF]\n       rb [-t N] invert [PAF]\n"
                    "       rb [-t N] trim-paf [-m M] [-d D] [-i I] [-r] [PAF]\n");
    return 2;
}

int main(int argc, char** argv) {
    std::string cmd, bed, input = "-";
    bool qbed = false, largest = false, paf_flag = false;
    int policy = RB_POLICY_RIGHTMOST;
    unsigned long max_size = 100;  // cli.rs:163
    int match_score = 1, diff_score = 1, indel_score = 1;  // cli.rs:126-134
    bool remove_contained = false;
    bool is_trim = false;
    bool stats_rows = false;
    int n_gpus = 1;  // --gpus G (not in the reference): a multi-device rb_ctx, records spread over devices 0 .. G-1
    for (int i = 1; i < argc; i++) {
        const std::string a = argv[i];
        if (a == "--gpus" && i + 1 < argc) { n_gpus = atoi(argv[++i]); continue; }
        if (cmd.empty() && a == "lo") { cmd = "liftover"; continue; }  // cli.rs: visible_aliases = ["lo"]
        if (cmd.empty() && (a == "trim-paf" || a == "trim" || a == "tp")) { cmd = "trim-paf"; is_trim = true; continue; }
        if (is_trim) {  // trim-paf reuses short flags of other subcommands (-m, -i, -d, -r)
            if ((a == "-m" || a == "--match-score") && i + 1 < argc) { match_score = atoi(argv[++i]); continue; }
            if ((a == "-d" || a == "--diff-score") && i + 1 < argc) { diff_score = atoi(argv[++i]); continue; }
            if ((a == "-i" || a == "--indel-score") && i + 1 < argc) { indel_score = atoi(argv[++i]); continue; }
            if (a == "-r" || a == "--remove-contained") { remove_contained = true; continue; }
        }
        if ((a == "-t" || a == "--threads") && i + 1 < argc) i++;  // accepted for compatibility; the GPU path has no thread knob
        else if (a == "-v" || a == "-vv" || a == "-vvv") {}
        else if ((a == "--bed" || a == "-b") && i + 1 < argc) bed = argv[++i];
        else if (a == "--qbed" || a == "-q") qbed = true;
        else if (a == "--largest" || a == "-l") largest = true;
        else if (a == "--stats") stats_rows = true;  // (not in the reference) liftover: print what `| rb stats --paf` would print
        else if (a == "--paf" || a == "-p") paf_flag = true;
        else if ((a == "--max-size" || a == "-m") && i + 1 < argc) max_size = strtoul(argv[++i], nullptr, 10);
        else if (a == "--policy" && i + 1 < argc) policy = strcmp(argv[++i], "early-exit") == 0 ? RB_POLICY_EARLY_EXIT : RB_POLICY_RIGHTMOST;
        else if (cmd.empty()) cmd = a;
        else input = a;
    }
    const bool brk = (cmd == "break-paf" || cmd == "breakpaf" || cmd == "bp");
    const bool inv = (cmd == "invert");
    if (cmd != "liftover" && !(cmd == "stats" && paf_flag) && !brk && !inv && !is_trim) return usage();
    int status = 0;
    if (n_gpus < 1 || n_gpus > 64) return usage();
    // RB_TIMING=1: wall-clock of the phases of this (one-shot, cold) process as one JSON line on stderr
    const bool timing = getenv("RB_TIMING") != nullptr;
    const auto t_start = std::chrono::steady_clock::now();
    auto t_last = t_start;
    std::string phases;
    auto mark = [&](const char* name) {
        if (!timing) return;
        const auto now = std::chrono::steady_clock::now();
        char buf[96];
        snprintf(buf, sizeof buf, "%s\"%s_ms\": %.1f", phases.empty() ? "" : ", ", name, std::chrono::duration<double, std::milli>(now - t_last).count());
        phases += buf;
        t_last = now;
    };
    int ids[64];
    for (int d = 0; d < n_gpus; d++) ids[d] = d;
    rb_ctx* ctx = rb_ctx_create(ids, n_gpus, &status);
    if (!ctx) {
        fprintf(stderr, "rb: no usable sm_100 CUDA device (status %d); this build has no CPU path\n", status);
        return 3;
    }
    mark("ctx_create");
    // PAF input (myio.rs:41-64): a `.bgz` / `.gz` file that is BGZF has its blocks inflated on the device (rb_inflate_bgzf) and the
    // lines are parsed out of the pinned buffer that comes back; RB_GPU_INFLATE=0 keeps the host's block-parallel zlib reader.
    // A plain gzip member, stdin and uncompressed files go through rbh::read_all as before.
    auto load_paf = [&](const std::string& path) {
        auto ends_with = [&](const char* suf) { const size_t n = strlen(suf); return path.size() >= n && path.compare(path.size() - n, n, suf) == 0; };
        const char* sw = getenv("RB_GPU_INFLATE");
        if (path != "-" && (ends_with(".bgz") || ends_with(".gz")) && !(sw && sw[0] == '0')) {
            const std::string raw = rbh::read_raw(path);
            if (rb_is_bgzf(reinterpret_cast<const uint8_t*>(raw.data()), raw.size())) {
                uint8_t* text = nullptr;
                uint64_t n = 0;
                if (rb_inflate_bgzf(ctx, reinterpret_cast<const uint8_t*>(raw.data()), raw.size(), &text, &n) != RB_OK)
                    throw rbh::Panic("error inflating " + path + ": " + rb_last_error(ctx));
                mark("gpu_inflate");
                rbh::Paf paf = rbh::Paf::from_text(reinterpret_cast<const char*>(text), (size_t)n);
                rb_free_text(ctx, text);
                return paf;
            }
        }
        return rbh::Paf::from_file(path);
    };
    // RB_DEVICE_PARSE=1: `rb [--gpus N] liftover` (plain, --stats, --largest) hands the bytes of the PAF and the BED to one
    // rb_liftover_text call, and `rb [--gpus N] stats --paf [--qbed]` the bytes of the PAF to one rb_stats_text call — lines are split
    // and parsed (and the stats rows formatted) on the device(s) instead of on the host.  A plain file is mapped, a .bgz / .gz that is
    // BGZF goes as it is (inflated on the device), a plain .gz and stdin are inflated / read by rbh::read_all first.
    const char* dp = getenv("RB_DEVICE_PARSE");
    const bool device_parse = dp && dp[0] == '1' && ((cmd == "liftover" && !qbed) || cmd == "stats");
    struct InputBytes {
        std::string owned;
        const uint8_t* data = nullptr;
        size_t n = 0;
        void* map = nullptr;
        ~InputBytes() { if (map) munmap(map, n); }
    };
    auto input_bytes = [&](const std::string& path, InputBytes& in) {
        auto ends_with = [&](const char* suf) { const size_t n = strlen(suf); return path.size() >= n && path.compare(path.size() - n, n, suf) == 0; };
        if (path != "-" && !ends_with(".gz") && !ends_with(".bgz")) {
            const int fd = ::open(path.c_str(), O_RDONLY);
            if (fd < 0) throw rbh::Panic("Error: cannot read input file " + path);
            struct stat st;
            if (fstat(fd, &st) == 0 && S_ISREG(st.st_mode) && st.st_size > 0) {
                in.map = mmap(nullptr, (size_t)st.st_size, PROT_READ, MAP_PRIVATE, fd, 0);
                if (in.map == MAP_FAILED) in.map = nullptr;
                else { in.data = static_cast<const uint8_t*>(in.map); in.n = (size_t)st.st_size; }
            }
            ::close(fd);
            if (!in.map) in.owned = rbh::read_raw(path);
        } else if (path != "-") {
            in.owned = rbh::read_raw(path);
            if (!rb_is_bgzf(reinterpret_cast<const uint8_t*>(in.owned.data()), in.owned.size())) in.owned = rbh::read_all(path);
        } else {
            in.owned = rbh::read_all(path);
        }
        if (!in.map) { in.data = reinterpret_cast<const uint8_t*>(in.owned.data()); in.n = in.owned.size(); }
    };
    int rc = 0;
    try {
        if (device_parse && cmd == "stats") {
            fputs(rbh::stats_header(qbed).c_str(), stdout);  // printed before the input is read (main.rs:51)
            fflush(stdout);
            rb_lift_out out{};
            rb_paf_info pinfo{};
            {
                InputBytes paf_in;
                input_bytes(input, paf_in);
                rc = rb_stats_text(ctx, paf_in.data, paf_in.n, qbed ? 1 : 0, RB_WANT_STATS_TEXT, &out, nullptr, &pinfo);
            }
            mark("rb_stats_text");
            if (pinfo.names_off && pinfo.skipped) fprintf(stderr, "\nUnable to parse %zu PAF record(s). Skipped.\n", (size_t)pinfo.skipped);
            if (rc == RB_OK) {
                fwrite(out.paf_text, 1, out.paf_nbytes, stdout);
                fflush(stdout);
                mark("write");
                rb_free_lift_out(ctx, &out);
            }
        } else if (device_parse) {
            if (bed.empty()) return usage();
            if (stats_rows && largest) return usage();
            InputBytes bed_in;
            input_bytes(bed, bed_in);
            mark("read_bed");
            const uint32_t want = (stats_rows ? RB_WANT_STATS_TEXT : RB_WANT_TEXT) | (largest ? RB_WANT_NUMERIC : 0u);
            rb_lift_out out{};
            rb_paf_info pinfo{};
            {
                InputBytes paf_in;
                input_bytes(input, paf_in);
                rc = rb_liftover_text(ctx, paf_in.data, paf_in.n, bed_in.data, bed_in.n, policy, want, &out, nullptr, &pinfo, nullptr);
            }
            mark("rb_liftover_text");
            if (pinfo.names_off) {  // the PAF parsed
                if (pinfo.skipped) fprintf(stderr, "\nUnable to parse %zu PAF record(s). Skipped.\n", (size_t)pinfo.skipped);
                if (stats_rows) { fputs(rbh::stats_header(false).c_str(), stdout); fflush(stdout); }  // main.rs:51
            }
            if (rc == RB_OK) {
                if (largest) {  // main.rs:200-208
                    const std::string rows = rbh::largest_rows(out);
                    fwrite(rows.data(), 1, rows.size(), stdout);
                } else {
                    fwrite(out.paf_text, 1, out.paf_nbytes, stdout);
                }
                fflush(stdout);
                mark("write");
                rb_free_lift_out(ctx, &out);
            }
        } else if (cmd == "stats") {
            fputs(rbh::stats_header(qbed).c_str(), stdout);  // printed before the input is read (main.rs:51)
            fflush(stdout);
            rbh::Paf paf = load_paf(input);
            mark("read_parse_paf");
            if (paf.skipped) fprintf(stderr, "\nUnable to parse %zu PAF record(s). Skipped.\n", paf.skipped);
            rb_records recs = paf.view();
            rb_stats_out st{};
            rc = rb_stats(ctx, &recs, &st);
            mark("rb_stats");
            if (rc == RB_OK) {
                rbh::write_stats_rows(stdout, paf, st, qbed);
                fflush(stdout);
                mark("format_write");
                rb_free_stats_out(ctx, &st);
            }
        } else if (brk) {
            rbh::Paf paf = load_paf(input);
            if (paf.skipped) fprintf(stderr, "\nUnable to parse %zu PAF record(s). Skipped.\n", paf.skipped);
            rb_records recs = paf.view();
            rb_lift_out out{};
            rc = rb_break_paf(ctx, &recs, (uint32_t)max_size, policy, RB_WANT_TEXT, &out, nullptr);
            if (rc == RB_OK) {
                fwrite(out.paf_text, 1, out.paf_nbytes, stdout);
                rb_free_lift_out(ctx, &out);
            }
        } else if (is_trim) {
            rbh::Paf paf = load_paf(input);
            if (paf.skipped) fprintf(stderr, "\nUnable to parse %zu PAF record(s). Skipped.\n", paf.skipped);
            rb_records recs = paf.view();
            rb_lift_out out{};
            rc = rb_trim_paf(ctx, &recs, match_score, diff_score, indel_score, remove_contained ? 1 : 0, policy, RB_WANT_TEXT, &out, nullptr);
            if (rc == RB_OK) {
                fwrite(out.paf_text, 1, out.paf_nbytes, stdout);
                rb_free_lift_out(ctx, &out);
            }
        } else if (inv) {
            rbh::Paf paf = load_paf(input);
            if (paf.skipped) fprintf(stderr, "\nUnable to parse %zu PAF record(s). Skipped.\n", paf.skipped);
            rb_records recs = paf.view();
            rb_lift_out out{};
            rc = rb_invert(ctx, &recs, RB_WANT_TEXT, &out);
            if (rc == RB_OK) {
                fwrite(out.paf_text, 1, out.paf_nbytes, stdout);
                rb_free_lift_out(ctx, &out);
            }
        } else {
            if (bed.empty()) return usage();
            const std::string bed_text = rbh::read_all(bed);
            mark("read_bed");
            rbh::Paf paf = load_paf(input);
            mark("read_parse_paf");
            if (paf.skipped) fprintf(stderr, "\nUnable to parse %zu PAF record(s). Skipped.\n", paf.skipped);
            rbh::Windows wins = rbh::Windows::pack_text(bed_text.data(), bed_text.size(), paf);  // bed::parse_bed + sort, all host threads
            mark("pack_bed");
            rb_records recs = paf.view();
            rb_windows w = wins.view();
            rb_lift_out out{};
            if (stats_rows && largest) return usage();
            const uint32_t want = (stats_rows ? RB_WANT_STATS_TEXT : RB_WANT_TEXT) | (largest ? RB_WANT_NUMERIC : 0u) | (qbed ? RB_WANT_QBED : 0u);
            if (stats_rows) { fputs(rbh::stats_header(false).c_str(), stdout); fflush(stdout); }  // main.rs:51
            rc = rb_liftover(ctx, &recs, &w, policy, want, &out, nullptr);
            mark("rb_liftover");
            if (rc == RB_OK) {
                if (largest) {  // main.rs:200-208
                    const std::string rows = rbh::largest_rows(out);
                    fwrite(rows.data(), 1, rows.size(), stdout);
                } else {
                    fwrite(out.paf_text, 1, out.paf_nbytes, stdout);
                }
                fflush(stdout);
                mark("write");
                rb_free_lift_out(ctx, &out);
            }
        }
    } catch (const rbh::Panic& e) {
        fprintf(stderr, "thread 'main' panicked: %s\n", e.what());
        rb_ctx_destroy(ctx);
        return 101;
    }
    if (rc != RB_OK) {
        fprintf(stderr, "rb: %s\n", rb_last_error(ctx));
        const bool ref_panic = (rc <= RB_ERR_REF_CIGAR_PARSE && rc >= RB_ERR_REF_INDEX) || rc == RB_ERR_REF_PAF_PARSE;
        rb_ctx_destroy(ctx);
        return ref_panic ? 101 : 1;
    }
    rb_ctx_destroy(ctx);
    mark("destroy");
    if (timing)
        fprintf(stderr, "{\"rb_timing\": {%s, \"total_ms\": %.1f}}\n", phases.c_str(),
                std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_start).count());
    return 0;
}
