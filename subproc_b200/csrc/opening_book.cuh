// opening_book.cuh -- the game tree of the first OB_PLAYOUT_BOOK_DEPTH plies from the standard opening, which the
// random playout kernel walks instead of playing those plies (playout.cu).
//
// Every game from the standard opening with Black to move goes through the same few positions at first (4 after one
// ply, 244 move paths after four, 390 216 after eight).  A random ply there is a step down this tree: the draw that
// picks the k-th legal move picks the k-th child, because the children of a node are its legal moves in ascending
// square order (puttables() order, board.py:46-52).  So a book ply costs the draw, one load and the trajectory stores
// instead of a move generation, the k-th-bit search and put().
//
// Layout: breadth first, the children of a node contiguous and in ascending square order, one node per 32-byte
// sector.  No node above the last ply is without a legal move, so the tree holds no pass (build_book checks it), and
// Black moves at even depths.  The host builder uses the rules primitives of fastboard.cuh, so a g++ test can compare
// the tree with the oracle (tests/test_opening_book_host.py).
#pragma once
#include <stdint.h>
#include <vector>
#include "fastboard.cuh"

// Plies taken from the book; 0 = none.  Even, so that White's and Black's plies keep alternating in the unrolled loop
// of the kernel after it.  Depth 8 is 455 221 nodes (14.6 MB).
#if !defined(OB_PLAYOUT_BOOK_DEPTH)
#define OB_PLAYOUT_BOOK_DEPTH 8
#endif

namespace obb {

using obf::u64;
using obf::u32;

constexpr int kBookDepth = OB_PLAYOUT_BOOK_DEPTH;
static_assert(kBookDepth >= 0 && kBookDepth <= 8 && kBookDepth % 2 == 0, "OB_PLAYOUT_BOOK_DEPTH: 0, 2, 4, 6 or 8");

struct alignas(32) BookNode {
    u64 black, white;       // the position
    u32 first;              // index of the first child (nodes above the last ply)
    u32 info;               // bits 0..7: number of children (0 at the last ply); bits 8..15: the move that led here
    u32 pad[2];
};
static_assert(sizeof(BookNode) == 32, "one node per 32-byte sector");

// The line tables of obf::flips_lut, on the host.
struct HostLines {
    u64 t[obf::kRayTable64];
    HostLines() { for (int i = 0; i < obf::kRayTable64; i++) t[i] = obf::make_table_word(i); }
    OBF_HD u64 word(u32 i) const { return t[i]; }
    OBF_HD u32 byte(u32 i) const { return ((const unsigned char *)t)[i]; }      // (little-endian host)
};

// The tree to `depth` plies in `nodes`.  False if a position above the last ply has no legal move: the kernel's walk
// has no pass.
inline bool build_book(int depth, std::vector<BookNode> &nodes)
{
    static const HostLines lines;
    nodes.assign(1, BookNode{0x0000000810000000ull, 0x0000001008000000ull, 0, 0, {0, 0}});   // board.py:22-27
    size_t begin = 0;
    for (int d = 0; d < depth; d++) {
        const size_t end = nodes.size();
        for (size_t i = begin; i < end; i++) {
            const bool black = d % 2 == 0;
            const u64 own = black ? nodes[i].black : nodes[i].white, opp = black ? nodes[i].white : nodes[i].black;
            u64 legal = obf::legal_moves(own, opp);
            if (legal == 0) return false;
            nodes[i].first = (u32)nodes.size();
            nodes[i].info |= (u32)obf::popc64(legal);
            for (; legal; legal &= legal - 1) {
                const int s = __builtin_ctzll(legal);
                const u64 f = obf::flips_lut(s, own, opp, lines, 1u);
                const u64 mover = own | f | (1ull << s), other = opp & ~f;
                nodes.push_back(BookNode{black ? mover : other, black ? other : mover, 0, (u32)s << 8, {0, 0}});
            }
        }
        begin = end;
    }
    return true;
}

}  // namespace obb
