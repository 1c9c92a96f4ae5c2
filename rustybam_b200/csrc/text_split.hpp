// text_split.hpp — which bytes each device parses when a text is cut into D consecutive byte ranges (rb_liftover_text).  A cut falls
// anywhere, so the lines that straddle cuts are moved whole: a line belongs to the device whose range holds its first byte.  Range
// d > 0 that does not start at a line start (the byte before it is not '\n') gives away its head — its bytes up to and including its
// first '\n', or all of them when it holds none — to the owner of the line they continue, the nearest range before it that starts a
// line or holds a '\n' (range 0 at the latest).  What a device keeps of its own range comes first in its buffer, then the pieces it
// receives, in text order; the buffers of devices 0 .. D-1 concatenated are the text again, and every buffer but the last non-empty
// one ends with '\n'.  Pure host code (tests/native/text_split_check.cpp fuzzes it).
#pragma once
#include <cstdint>
#include <vector>

namespace rbt {

constexpr uint64_t NO_NEWLINE = ~0ull;

struct Piece {
    int src;        // range the bytes come from
    uint64_t off;   // offset in that range
    uint64_t len;
};
struct Owned {
    std::vector<Piece> pieces;  // in text order; they go one after the other into the owner's buffer
    uint64_t bytes = 0;
};

// size[d]: bytes of range d; first_nl[d]: offset of the first '\n' in range d, or NO_NEWLINE; ends_nl[d]: range d is not empty and
// its last byte is '\n'
inline std::vector<Owned> plan_line_split(const std::vector<uint64_t>& size, const std::vector<uint64_t>& first_nl,
                                          const std::vector<uint8_t>& ends_nl) {
    const int D = (int)size.size();
    std::vector<Owned> own((size_t)D);
    int owner = 0;
    bool line_start = true;  // the text in front of range d is empty or ends with '\n'
    for (int d = 0; d < D; d++) {
        const uint64_t n = size[(size_t)d], nl = first_nl[(size_t)d];
        if (n == 0) continue;
        if (line_start) {
            owner = d;
            own[(size_t)d].pieces.push_back({d, 0, n});
        } else if (nl == NO_NEWLINE) {
            own[(size_t)owner].pieces.push_back({d, 0, n});
        } else {
            own[(size_t)owner].pieces.push_back({d, 0, nl + 1});
            owner = d;
            if (n > nl + 1) own[(size_t)d].pieces.push_back({d, nl + 1, n - nl - 1});
        }
        line_start = ends_nl[(size_t)d] != 0;
    }
    for (Owned& o : own)
        for (const Piece& p : o.pieces) o.bytes += p.len;
    return own;
}

}  // namespace rbt
