// rbhost.hpp — C++ host side above the C ABI (include/rbcuda.h): text I/O stays on the host.
//
// Mirrors the reference's host-facing pieces for this path (file:line into the reference):
//   src/myio.rs:41-64        reader(): plain / .gz / .bgz / stdin          -> read_all()
//   src/paf.rs:62-78,379-430 Paf::from_file / PafRecord::new               -> Paf::from_text / from_file
//   src/bed.rs:140-194       parse_bed (bio bed::Reader semantics)         -> parse_bed_text / parse_bed
//   src/liftover.rs:134-167  trim_paf_by_rgns                              -> trim_paf_by_rgns (GPU, via rb_liftover)
//   src/bamstats.rs:91-105   stats_from_paf, :225-270 printers             -> stats_from_paf (GPU, via rb_stats) + printers
//   src/main.rs:50-58,186-214 `rb stats --paf`, `rb liftover`              -> rb_main.cpp
// CIGAR text is never tokenised here: the cg:Z: payload bytes are packed verbatim for the GPU.
#pragma once
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <new>
#include <stdexcept>
#include <string>
#include <unordered_map>
#include <utility>
#include <vector>

#include "rbcuda.h"

namespace rbh {

// Allocator of the big buffers that cross the C ABI (CIGAR text, window tables): page-aligned and padded to whole pages,
// so that rb_host_register() page-locks memory this buffer owns alone (a neighbouring heap object sharing its first or
// last page would otherwise end up half page-locked, which the driver rejects on the next copy out of it).
template <class T>
struct PageAlloc {
    using value_type = T;
    PageAlloc() = default;
    template <class U> PageAlloc(const PageAlloc<U>&) {}
    T* allocate(size_t n) {
        const size_t bytes = (n * sizeof(T) + 4095) / 4096 * 4096;
        void* p = aligned_alloc(4096, bytes ? bytes : 4096);
        if (!p) throw std::bad_alloc();
        return static_cast<T*>(p);
    }
    void deallocate(T* p, size_t) { free(p); }
    template <class U> bool operator==(const PageAlloc<U>&) const { return true; }
    template <class U> bool operator!=(const PageAlloc<U>&) const { return false; }
};
template <class T> using PagedVec = std::vector<T, PageAlloc<T>>;
// the same for the one buffer of many GB (the packed CIGAR text): resize() default-initialises, i.e. leaves the bytes alone, so
// the pages are first touched by the threads that copy the payloads in instead of being zeroed by one thread beforehand
template <class T>
struct PageAllocNoInit : PageAlloc<T> {
    template <class U> struct rebind { using other = PageAllocNoInit<U>; };
    PageAllocNoInit() = default;
    template <class U> PageAllocNoInit(const PageAllocNoInit<U>&) {}
    template <class U, class... A> void construct(U* p, A&&... a) {
        if constexpr (sizeof...(A) == 0) ::new (static_cast<void*>(p)) U;
        else ::new (static_cast<void*>(p)) U(std::forward<A>(a)...);
    }
};
using PagedBytes = std::vector<uint8_t, PageAllocNoInit<uint8_t>>;

struct Panic : std::runtime_error {  // the reference would panic (exit status 101)
    explicit Panic(const std::string& m) : std::runtime_error(m) {}
};

std::string read_all(const std::string& path);  // "-" = stdin; .gz/.bgz inflated with zlib
std::string read_raw(const std::string& path);  // the file's bytes as they are (the caller inflates: rb_inflate_bgzf)

// Packed records (what rb_records points into).  Name ids are shared by query and target names.
struct Paf {
    PagedBytes cigar;
    std::vector<uint64_t> cigar_off{0};
    std::vector<uint64_t> q_len, q_st, q_en, t_len, t_st, t_en, mapq;
    std::vector<uint8_t> strand;
    std::vector<uint32_t> q_id, t_id;
    std::vector<std::string> names;
    std::vector<uint8_t> names_blob;
    std::vector<uint64_t> names_off;
    size_t skipped = 0;

    size_t size() const { return q_id.size(); }
    uint32_t name_id(const std::string& s);            // interns
    int64_t find_name(const std::string& s) const;     // -1 if absent
    static Paf from_text(const char* text, size_t n);  // throws Panic like PafRecord::new's asserts
    static Paf from_file(const std::string& path);     // plain files are mapped, not copied; "-", .gz, .bgz go through read_all
    rb_records view();  // finalises the name table and returns the SoA view

   private:
    std::unordered_map<std::string, uint32_t> index_;  // name -> id; read-level PAFs intern millions of query names
};

struct Region {
    std::string name;
    uint64_t st = 0, en = 0;
    std::string id;
    bool default_id = false;  // no 4th BED column: id == "{name}:{st+1}-{en}" (bed.rs:150-153)
};
std::vector<Region> parse_bed_text(const char* text, size_t n);
inline std::vector<Region> parse_bed(const std::string& path) {
    std::string t = read_all(path);
    return parse_bed_text(t.data(), t.size());
}

// rb_windows builder: drops rows on contigs absent from the PAF, sorts by (t_id, st) keeping bed_row
struct Windows {
    PagedVec<uint32_t> t_id, bed_row;
    PagedVec<uint64_t> st, en, ids_off;
    PagedVec<uint8_t> ids;
    bool default_ids = false;  // every row carries the default id: ids / ids_off stay empty and the GPU formats them
    rb_windows view() const;
    static Windows pack(const std::vector<Region>& rgns, const Paf& paf);
    static Windows pack_text(const char* bed_text, size_t n, const Paf& paf);  // == pack(parse_bed_text(..), paf), parallel, no per-row strings
};

// `rb liftover --largest` (main.rs:200-208): rows stably sorted by id, one row per id: the LAST one of maximal target span
std::string largest_rows(const rb_lift_out& out);

std::string fmt_f32(float v);                 // Rust `{}` for f32 (shortest round trip, positional)
std::string stats_header(bool qbed);          // bamstats.rs:225-236
// bamstats.rs:239-270 for row i of `paf` with the GPU counters of row i
void append_stats_row(std::string& out, const Paf& paf, size_t i, const rb_stats_out& st, bool qbed);
// one row from its fields (what append_stats_row formats for a record of `paf`)
void append_row(std::string& out, const std::string& q_name, const std::string& t_name, uint8_t strand, uint64_t q_st, uint64_t q_en,
                uint64_t q_len, uint64_t t_st, uint64_t t_en, uint64_t t_len, const rb_stats_out& st, size_t i, bool qbed);
// every row of `paf` (bamstats.rs:239-270), formatted on all host threads, written to `f` in row order
void write_stats_rows(FILE* f, const Paf& paf, const rb_stats_out& st, bool qbed);

// ---- synthetic whole-genome-scale eqx PAF (SURVEY §8d, configs C2-C5) ----
struct SynthParams {
    uint64_t seed = 20261017;
    double scale = 1.0;   // multiplies the CHM13-like contig lengths
    int n_hap = 1;        // haplotypes (independent streams) concatenated
    int threads = 8;
    uint32_t contig_mask = 0xFFFFFFFFu;  // bit c: generate contig c of the CHM13-like table (a GPU's share of a multi-GPU job)
};
Paf synth_paf(const SynthParams& p);
// `bedtools makewindows`-style tiling of every target contig of `paf`, 3 columns (id = chrom:st+1-en), sorted
std::vector<Region> tiling_windows(const Paf& paf, uint64_t width);
Windows tiling_windows_packed(const Paf& paf, uint64_t width);
// PAF text of records [lo, hi) (12 columns + cg:Z:) — input for the CPU oracle / reference
std::string paf_text(const Paf& paf, size_t lo, size_t hi);
std::string bed_text(const std::vector<Region>& rgns, bool with_ids);

}  // namespace rbh
