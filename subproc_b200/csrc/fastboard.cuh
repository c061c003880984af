// fastboard.cuh -- the rules primitives every kernel uses: Board.puttables (board.py:46-52) and
// Board.put (board.py:161-174) on a pair of 64-bit bitboards held in registers.
//
// The formulation is shaped by what ncu showed on the first, textbook version (8-direction
// Kogge-Stone floods in both shift directions): the playout kernel was bound by the INT32 ALU pipe
// (sm__inst_executed_pipe_alu 96 %, profiles/playout_r01_ncu_summary.txt) while the FMA pipe (IMAD)
// and the XU pipe (BREV/POPC) idled.  On B200 a 64-bit RIGHT shift costs two ALU instructions, a
// LEFT shift one ALU + one IMAD.SHL; BREV runs on the XU pipe.  So:
//
//   * every flood runs to the LEFT: the four "down" directions are evaluated as "up" directions
//     on the bit-reversed board (BREV64 = 2 XU instructions), results reversed back once;
//   * the two horizontal directions use the carry of an integer ADD instead of a flood:
//     adding the run-start bits to the opponent row makes the carry ripple through the run and
//     land on the square behind it (3 instructions per 32-bit half instead of 24);
//   * put(): the flipped run of each of the 8 rays is found with one 64-bit ADD per ray:
//     (opp | ~ray) + move_bit ripples through the opponent discs on the ray and stops on the first
//     square that is not one; if that square is own, the rippled-through discs are the flips.
//     Ray masks come from a 2 KB table in shared memory ([direction][square], 8 LDS.64 per move).
//
// All functions are host+device so tests/ can compile this very file with g++ and compare it with
// the oracle on the CPU (tests/test_fastboard_host.py); the host build is test scaffolding only.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define OBF_HD __host__ __device__ __forceinline__
#else
#define OBF_HD inline
#endif

namespace obf {

typedef unsigned long long u64;
typedef unsigned int u32;

constexpr u64 kInner64 = 0x7E7E7E7E7E7E7E7Eull;   // files b..g (see bitboard.cuh)
constexpr u32 kInner32 = 0x7E7E7E7Eu;

OBF_HD u32 lo32(u64 v) { return (u32)v; }
OBF_HD u32 hi32(u64 v) { return (u32)(v >> 32); }
OBF_HD u64 pack(u32 lo, u32 hi) { return ((u64)hi << 32) | lo; }

OBF_HD u32 brev32(u32 v)
{
#if defined(__CUDA_ARCH__)
    return __brev(v);
#else
    v = ((v >> 1) & 0x55555555u) | ((v & 0x55555555u) << 1);
    v = ((v >> 2) & 0x33333333u) | ((v & 0x33333333u) << 2);
    v = ((v >> 4) & 0x0F0F0F0Fu) | ((v & 0x0F0F0F0Fu) << 4);
    v = ((v >> 8) & 0x00FF00FFu) | ((v & 0x00FF00FFu) << 8);
    return (v >> 16) | (v << 16);
#endif
}

// square s <-> square 63 - s: a 180 degree rotation of the board
OBF_HD u64 rev64(u64 v) { return pack(brev32(hi32(v)), brev32(lo32(v))); }

OBF_HD int popc64(u64 v)
{
#if defined(__CUDA_ARCH__)
    return __popcll(v);
#else
    return __builtin_popcountll(v);
#endif
}

// ---- move generation in the row-interleaved layout ------------------------------------------------
// A 64-bit shift that crosses the two 32-bit halves costs an ALU-pipe funnel (SHF.L.U64.HI).  With
// word a = ranks 1,3,5,7 and word b = ranks 2,4,6,8 (one rank per byte) "one rank down" swaps the
// words, so every shift of the +8 and +9 floods and half of the +7 ones is a plain 32-bit LEFT shift
// (IMAD.SHL on the FMA pipe) and "+8" costs one instruction instead of two:
//     +8: (a, b) -> (b << 8, a)      +16: (a << 8,  b << 8)
//     +9: (a, b) -> (b << 9, a << 1) +18: (a << 10, b << 10)
//     +7: (a, b) -> (b << 7, a >> 1) +14: (a << 6,  b << 6)
// Converting to and from the standard layout is two byte permutes (PRMT) per bitboard; the 180-degree
// rotation is still two BREVs: rev{a, b} = {brev(b), brev(a)}.
struct Inter { u32 a, b; };

OBF_HD u32 byte_perm(u32 x, u32 y, u32 sel)
{
#if defined(__CUDA_ARCH__)
    return __byte_perm(x, y, sel);
#else
    const u64 v = pack(x, y);
    u32 r = 0;
    for (int i = 0; i < 4; i++) r |= (u32)((v >> (8 * ((sel >> (4 * i)) & 7))) & 0xFF) << (8 * i);
    return r;
#endif
}

OBF_HD Inter to_inter(u64 v) { return Inter{byte_perm(lo32(v), hi32(v), 0x6420u), byte_perm(lo32(v), hi32(v), 0x7531u)}; }
OBF_HD u64 from_inter(Inter v) { return pack(byte_perm(v.a, v.b, 0x5140u), byte_perm(v.a, v.b, 0x7362u)); }
OBF_HD Inter rev_inter(Inter v) { return Inter{brev32(v.b), brev32(v.a)}; }
OBF_HD Inter iand(Inter x, Inter y) { return Inter{x.a & y.a, x.b & y.b}; }
OBF_HD Inter ior(Inter x, Inter y) { return Inter{x.a | y.a, x.b | y.b}; }

#if defined(__CUDACC__)
// An integer 1 the compiler cannot see through: multiplying by it keeps an addition on the FMA pipe
// (IMAD) instead of the saturated ALU pipe (IADD3 / SEL / LOP3).
static __device__ __constant__ u32 kOpaqueOne = 1u;
#endif

template <int D> OBF_HD Inter ishift(Inter v)        // D squares up (towards higher squares), D in {7, 8, 9}
{
    return D == 8 ? Inter{v.b << 8, v.a} : D == 9 ? Inter{v.b << 9, v.a << 1} : Inter{v.b << 7, v.a >> 1};
}
template <int D> OBF_HD Inter ishift2(Inter v)       // 2 * D squares up
{
    return D == 8 ? Inter{v.a << 8, v.b << 8} : D == 9 ? Inter{v.a << 10, v.b << 10} : Inter{v.a << 6, v.b << 6};
}

// Flood to the LEFT (towards higher squares) by D: squares just beyond a run of `m` discs that
// starts right after an `own` disc.  Kogge-Stone: 1 + 1 + 2 + 2 = up to 6 discs.  p = pairs(m): discs of m
// whose neighbour D squares down is in m as well.
template <int D> OBF_HD Inter pairs(Inter m) { return iand(m, ishift<D>(m)); }
template <int D> OBF_HD Inter flood_up(Inter own, Inter m, Inter p)
{
    Inter f = iand(m, ishift<D>(own));
    f = ior(f, iand(m, ishift<D>(f)));
    f = ior(f, iand(p, ishift2<D>(f)));
    f = ior(f, iand(p, ishift2<D>(f)));
    return ishift<D>(f);
}

// Horizontal direction towards higher squares, per 32-bit word (a rank never straddles a word and
// `m` has no a/h-file bits, so no carry and no shifted bit crosses a rank): the carry of m + a
// ripples through each opponent run that starts right after an own disc and lands behind it.
OBF_HD u32 row_up32(u32 own, u32 m)
{
    const u32 a = (own << 1) & m;       // run starts
    return (m + a) & ~m;                // carry-out squares (bits set by the add that were clear in m)
}

// the pair masks of the three flood directions
struct Pairs { Inter p8, p7, p9; };
OBF_HD Pairs make_pairs(Inter opp, Inter m) { return Pairs{pairs<8>(opp), pairs<7>(m), pairs<9>(m)}; }
// ... of the board rotated by 180 degrees, from those of the board as it stands: a pair (s - D, s) is the pair
// (63 - s, 63 - s + D) of the rotated board, so the rotated mask is the rotation shifted up by D -- two BREVs
// (XU pipe) instead of two LOP3 (the saturated ALU pipe) per direction
OBF_HD Pairs rotated_pairs(const Pairs &q)
{
    return Pairs{ishift<8>(rev_inter(q.p8)), ishift<7>(rev_inter(q.p7)), ishift<9>(rev_inter(q.p9))};
}

// the four "up" directions (+1, +7, +8, +9) of one board; m = opp without the a/h files
OBF_HD Inter moves_up(Inter own, Inter opp, Inter m, const Pairs &q)
{
    Inter r = Inter{row_up32(own.a, m.a), row_up32(own.b, m.b)};
    r = ior(r, flood_up<8>(own, opp, q.p8));
    r = ior(r, flood_up<7>(own, m, q.p7));
    r = ior(r, flood_up<9>(own, m, q.p9));
    return r;
}

// A position prepared for move generation: both colours in the row-interleaved layout, as they stand
// and rotated by 180 degrees.  Swapping the roles of the colours is free (swap the members), and a
// successor position is two ORs / AND-NOTs away (see child_mobility).
struct Pos4 { Inter o, p, ro, rp; };

OBF_HD Pos4 make_pos4(u64 own, u64 opp)
{
    const Inter o = to_inter(own), p = to_inter(opp);
    return Pos4{o, p, rev_inter(o), rev_inter(p)};
}
OBF_HD Pos4 swapped(const Pos4 &q) { return Pos4{q.p, q.o, q.rp, q.ro}; }

// legal moves of colour `o`, still in the interleaved layout (popcount it, or from_inter() it)
OBF_HD Inter legal_inter(const Pos4 &q)
{
    // kInner32 is a palindrome, so the rotated inner mask is the same constant
    const Inter m = Inter{q.p.a & kInner32, q.p.b & kInner32}, mr = Inter{q.rp.a & kInner32, q.rp.b & kInner32};
    const Pairs pu = make_pairs(q.p, m);
    const Pairs pd = rotated_pairs(pu);                                       // BREV (XU pipe) instead of LOP3 (ALU pipe)
    const Inter up = moves_up(q.o, q.p, m, pu);
    const Inter down = moves_up(q.ro, q.rp, mr, pd);                          // the rotated board
    return iand(ior(up, rev_inter(down)), Inter{~(q.o.a | q.p.a), ~(q.o.b | q.p.b)});
}

OBF_HD int popc_inter(Inter v)
{
#if defined(__CUDA_ARCH__)
    return __popc(v.a) + __popc(v.b);
#else
    return __builtin_popcount(v.a) + __builtin_popcount(v.b);
#endif
}

// Board.puttables(piece) as a mask (board.py:46-52).
OBF_HD u64 legal_moves(u64 own, u64 opp) { return from_inter(legal_inter(make_pos4(own, opp))); }
// n_puttable_for(piece) (board.py:54-55): a popcount does not care about the layout, so the mask is not converted back
// (two PRMT on the ALU pipe fewer than __popcll(legal_moves()))
OBF_HD int mobility(u64 own, u64 opp) { return popc_inter(legal_inter(make_pos4(own, opp))); }

// n_puttable_for(mover) AFTER the mover has played: `placed` = the new disc + the discs it flipped.  The
// successor is built from the prepared parent (own' = own | placed, opp' = opp & ~placed), so a child costs one
// layout conversion and one rotation of `placed` instead of two of each for two full boards, and nothing is
// converted back (a popcount does not care about the layout).
OBF_HD int child_mobility(const Pos4 &parent, u64 placed)
{
    const Inter d = to_inter(placed), rd = rev_inter(d);
    const Pos4 c = Pos4{ior(parent.o, d), Inter{parent.p.a & ~d.a, parent.p.b & ~d.b},
                        ior(parent.ro, rd), Inter{parent.rp.a & ~rd.a, parent.rp.b & ~rd.b}};
    return popc_inter(legal_inter(c));
}

// n_puttable_for() of BOTH colours of one position (the mobility feature of counts(),
// parameter_progress_position_moves_learn.py:8): the layout conversions and rotations of the two
// boards are shared, and a popcount does not care about the layout, so nothing is converted back.
OBF_HD void mobility_both(u64 black, u64 white, int &mob_black, int &mob_white)
{
    const Pos4 q = make_pos4(black, white);
    mob_black = popc_inter(legal_inter(q));
    mob_white = popc_inter(legal_inter(swapped(q)));
}

// ---- move generation for four boards at once: the rank-sliced layout ----------------------------
// Word r of a sliced board holds rank r of four games, game j in byte j; bit x of a byte is still file x.  One rank up
// or down is the next or previous word, so a flood along a vertical or diagonal direction is one pass over the ranks
// (one LOP3 per rank for four games, plus a 1-bit shift inside the bytes for a diagonal) instead of a Kogge-Stone
// flood per game; a rank never straddles a byte, so the horizontal directions are row_up32 as above, the one towards
// lower files on the bit-reversed word (BREV32 also reverses the order of the games, which does not matter).  The
// inner mask keeps files a and h out of every diagonal and horizontal run, so no shifted bit or carry crosses into a
// neighbouring game's byte.  Going in and out of the layout is a 4x4 byte transpose per half-board (8 PRMT).

// byte i of word j <-> byte j of word i (its own inverse)
OBF_HD void transpose4(u32 &w0, u32 &w1, u32 &w2, u32 &w3)
{
    const u32 a = byte_perm(w0, w1, 0x5140u), b = byte_perm(w0, w1, 0x7362u);
    const u32 c = byte_perm(w2, w3, 0x5140u), d = byte_perm(w2, w3, 0x7362u);
    w0 = byte_perm(a, c, 0x5410u);
    w1 = byte_perm(a, c, 0x7632u);
    w2 = byte_perm(b, d, 0x5410u);
    w3 = byte_perm(b, d, 0x7632u);
}
OBF_HD void to_sliced(const u64 v[4], u32 s[8])
{
    for (int j = 0; j < 4; j++) { s[j] = lo32(v[j]); s[4 + j] = hi32(v[j]); }
    transpose4(s[0], s[1], s[2], s[3]);
    transpose4(s[4], s[5], s[6], s[7]);
}
OBF_HD void from_sliced(u32 s[8], u64 v[4])
{
    transpose4(s[0], s[1], s[2], s[3]);
    transpose4(s[4], s[5], s[6], s[7]);
    for (int j = 0; j < 4; j++) v[j] = pack(s[j], s[4 + j]);
}

// Board.puttables (board.py:46-52) of four positions: legal[j] = legal_moves(own[j], opp[j])
OBF_HD void legal_moves4(const u64 own[4], const u64 opp[4], u64 legal[4])
{
    u32 o[8], p[8], m[8], mv[8];
    to_sliced(own, o);
    to_sliced(opp, p);
#if defined(__CUDACC__)
#pragma unroll
#endif
    for (int r = 0; r < 8; r++) {
        m[r] = p[r] & kInner32;
        mv[r] = row_up32(o[r], m[r]) | brev32(row_up32(brev32(o[r]), brev32(m[r])));
    }
    // Up the board: u8 / u9 / u7 = the squares of rank r + 1 just beyond a run that starts after an own disc and
    // reaches rank r, along +8 / +9 (towards file h) / +7 (towards file a); each is also the run carried into rank r + 1.
    u32 u8 = 0, u9 = 0, u7 = 0;
#if defined(__CUDACC__)
#pragma unroll
#endif
    for (int r = 1; r < 7; r++) {
        u8 = p[r] & (o[r - 1] | u8);
        u9 = (m[r] & ((o[r - 1] << 1) | u9)) << 1;
        u7 = (m[r] & ((o[r - 1] >> 1) | u7)) >> 1;
        mv[r + 1] |= u8 | u9 | u7;
    }
    // ... and down the board: -8, -9 (towards file a), -7 (towards file h)
    u32 d8 = 0, d9 = 0, d7 = 0;
#if defined(__CUDACC__)
#pragma unroll
#endif
    for (int r = 6; r > 0; r--) {
        d8 = p[r] & (o[r + 1] | d8);
        d9 = (m[r] & ((o[r + 1] >> 1) | d9)) >> 1;
        d7 = (m[r] & ((o[r + 1] << 1) | d7)) << 1;
        mv[r - 1] |= d8 | d9 | d7;
    }
#if defined(__CUDACC__)
#pragma unroll
#endif
    for (int r = 0; r < 8; r++) mv[r] &= ~(o[r] | p[r]);
    from_sliced(mv, legal);
}


// ---- put(): flips through carry propagation along rays -----------------------------------------
// ray table: ray[d][s] = squares strictly beyond s in direction d in {+1, +7, +8, +9}, up to the edge; behind the
// four ray rows: a row of single-square masks, and the tables of the rank look-up (row_flips below)
constexpr int kRayDirs = 4;
constexpr int kRayBasic64 = (kRayDirs + 1) * 64;       // what the carry-chain form of put() needs: rays + single squares
constexpr int kRankMul64 = kRayBasic64;                // [8]: 1 << 8 * rank
constexpr int kFileMul64 = kRankMul64 + 8;             // [8]: low word 1 << (7 - file), high word 1 << file
constexpr int kDiag9_64 = kFileMul64 + 8;              // [64]: the whole +9 / -9 diagonal through a square
constexpr int kDiag7_64 = kDiag9_64 + 64;              // [64]: the whole +7 / -7 diagonal
constexpr int kRowOutflank64 = kDiag7_64 + 64;         // bytes [position on the line][opponent discs of the line]
// The two line tables are rows of 256 bytes, one per position on the line, kLineStride bytes apart.  With rows 256 bytes
// apart the shared-memory bank of an entry would depend on the pattern alone, and the patterns are anything but uniform
// (the second look-up is indexed by at most two closing discs: 0, 1, 2, 4 ...): lanes with different positions and the
// same pattern -- different addresses in ONE bank -- made these byte loads 6 to 7.6 wavefronts each, and the greedy kernel,
// which does eight of them per successor, ran at 87 % of the shared-memory pipe (profiles/greedy_r02_ncu_summary.txt).
// 276 = 256 + 20 moves every row on by five banks.
constexpr int kLineStride = 276;
constexpr int kLineTable64 = (8 * kLineStride + 7) / 8;
constexpr int kRowFlip64 = kRowOutflank64 + kLineTable64;  // bytes [position on the line][outflanking own discs]
constexpr int kKthBit64 = kRowFlip64 + kLineTable64;   // bytes [byte value][k]: position of the k-th set bit of a byte
constexpr int kSpread64 = kKthBit64 + 256 * 8 / 8;     // [256]: bit k of the index on bit 8 * k (a file-a column)
constexpr int kLine9_64 = kSpread64 + 256;             // [15]: the +9 / -9 diagonal number x - y + 7
constexpr int kLine7_64 = kLine9_64 + 15;              // [15]: the +7 / -7 diagonal number x + y
constexpr int kRayTable64 = kLine7_64 + 15;            // table entries (u64): 12.2 KB
OBF_HD constexpr u64 make_ray(int d, int s)
{
    if (d == kRayDirs) return 1ull << s;                               // row 4: the square itself (1 << s as a table load)
    const int dx = (d == 0) ? 1 : (d == 1) ? -1 : (d == 2) ? 0 : 1;   // +1: E, +7: SW, +8: S, +9: SE (y grows with s)
    const int dy = (d == 0) ? 0 : 1;
    u64 r = 0;
    int x = (s & 7) + dx, y = (s >> 3) + dy;
    while (x >= 0 && x < 8 && y < 8) { r |= 1ull << (x + 8 * y); x += dx; y += dy; }
    return r;
}
// A move on file x of a rank whose opponent discs are `opp` (8 bits): the squares on which an own disc would
// close a run of opponent discs that starts next to x (at most one on either side).
OBF_HD constexpr u32 row_outflank(int x, u32 opp)
{
    u32 r = 0;
    int i = x + 1;
    while (i <= 6 && ((opp >> i) & 1u)) i++;
    if (i > x + 1) r |= 1u << i;
    i = x - 1;
    while (i >= 1 && ((opp >> i) & 1u)) i--;
    if (i < x - 1) r |= 1u << i;
    return r;
}
// ... and the discs flipped when own discs stand on `closing` of those squares: everything between x and the
// nearest closing disc on either side.
OBF_HD constexpr u32 row_flipped(int x, u32 closing)
{
    u32 r = 0;
    for (int i = x + 1; i < 8; i++)
        if ((closing >> i) & 1u) { r |= ((1u << i) - 1u) & ~((2u << x) - 1u); break; }
    for (int i = x - 1; i >= 0; i--)
        if ((closing >> i) & 1u) { r |= ((1u << x) - 1u) & ~((2u << i) - 1u); break; }
    return r;
}
// position of the k-th (0-based, ascending) set bit of an 8-bit value (0 if it has fewer)
OBF_HD constexpr u32 kth_bit_of_byte(u32 v, int k)
{
    for (int i = 0; i < 8; i++)
        if ((v >> i) & 1u) { if (k == 0) return (u32)i; k--; }
    return 0;
}
// every square of the diagonal through s (s included), step 9 or 7
OBF_HD constexpr u64 make_diagonal(int step, int s)
{
    const int dx = step == 9 ? 1 : -1;
    u64 r = 0;
    for (int k = -7; k <= 7; k++) {
        const int x = (s & 7) + k * dx, y = (s >> 3) + k;
        if (x >= 0 && x < 8 && y >= 0 && y < 8) r |= 1ull << (x + 8 * y);
    }
    return r;
}
// word i of the whole table
OBF_HD constexpr u64 make_table_word(int i)
{
    if (i < kRankMul64) return make_ray(i >> 6, i & 63);
    if (i < kFileMul64) return 1ull << (8 * (i - kRankMul64));
    if (i < kDiag9_64) return ((1ull << (i - kFileMul64)) << 32) | (1ull << (7 - (i - kFileMul64)));
    if (i < kDiag7_64) return make_diagonal(9, i - kDiag9_64);
    if (i < kRowOutflank64) return make_diagonal(7, i - kDiag7_64);
    if (i >= kLine7_64) { const int n = i - kLine7_64; return make_diagonal(7, n < 8 ? n : 8 * (n - 7) + 7); }   // a square with x + y = n
    if (i >= kLine9_64) { const int n = i - kLine9_64; return make_diagonal(9, n < 8 ? 8 * (7 - n) : n - 7); }   // ... x - y + 7 = n
    u64 w = 0;
    for (int j = 0; j < 8; j++) {
        if (i >= kSpread64) {
            w |= (u64)(((i - kSpread64) >> j) & 1) << (8 * j);
        } else if (i >= kKthBit64) {
            w |= (u64)kth_bit_of_byte((u32)(i - kKthBit64), j) << (8 * j);
        } else if (i < kRowFlip64) {
            const int e = (i - kRowOutflank64) * 8 + j, x = e / kLineStride, v = e % kLineStride;
            if (x < 8 && v < 256) w |= (u64)row_outflank(x, (u32)v) << (8 * j);
        } else {
            const int e = (i - kRowFlip64) * 8 + j, x = e / kLineStride, v = e % kLineStride;
            if (x < 8 && v < 256) w |= (u64)row_flipped(x, (u32)v) << (8 * j);
        }
    }
    return w;
}

// The two horizontal rays of a move by table look-up instead of two carry chains: the rank of the move is a BYTE
// of the bitboards, so extracting it is one PRMT per colour; [file][opponent discs] gives the squares where an own
// disc would outflank, [file][those that are own] the flipped discs, which a multiply puts back on the rank.  6
// ALU-pipe instructions instead of 16 + 2 POPC; the look-ups run on the LSU pipe, idle in the playout kernel.
// rays.byte(i) = byte i of the table, rays.word(i) = word i.
template <typename RayTable>
OBF_HD void row_flips(int s, u64 own, u64 opp, const RayTable &rays, u32 &f_lo, u32 &f_hi)
{
    const u32 y = (u32)s >> 3, x = (u32)s & 7u;
    const u32 ob = byte_perm(lo32(own), hi32(own), y);       // byte 0 = the rank of the move (bytes 1..3: the first rank)
    const u32 pb = byte_perm(lo32(opp), hi32(opp), y);
    const u32 cand = rays.byte(kRowOutflank64 * 8 + x * kLineStride + (pb & 0xffu));
    const u32 flip = rays.byte(kRowFlip64 * 8 + x * kLineStride + (cand & ob));
    const u64 mul = rays.word(kRankMul64 + y);
    f_lo += flip * lo32(mul);
    f_hi += flip * hi32(mul);
}

// one ray: x = move bit, R = ray mask beyond it.  Returns the opponent run that an own disc closes.
OBF_HD u64 ray_flips(u64 x, u64 R, u64 own, u64 opp)
{
    const u64 sum = (opp | ~R) + x;            // ripples from x through the opponent discs on the ray
    const u64 closed = sum & own & R;          // the square where it stopped, if that square is own
    const u64 run = R & opp & ~sum;            // the discs it rippled through
    return closed ? run : 0ull;
}

#if defined(__CUDACC__)
// acc += run when the ray is closed.  The flipped runs of the 8 rays are pairwise disjoint, so the
// OR-accumulation of put() is an ADD.  `closed` has at most one bit set, so the sum of its two halves is
// non-zero exactly when the ray is closed; POPC (XU pipe) turns that into 0 / 1 and the run is added through
// a multiply by it (IMAD, FMA pipe): the test costs the saturated ALU pipe nothing (it used to be an OR of the
// halves + a compare per ray, 16 ALU instructions per move).
__device__ __forceinline__ void ray_accumulate(u32 &acc_lo, u32 &acc_hi, u64 x, u64 R, u64 own, u64 opp, u32 one)
{
    const u64 sum = (opp | ~R) + x;
    const u64 closed = sum & own & R;
    const u64 run = R & opp & ~sum;
    u32 any;
    asm("mad.lo.u32 %0, %1, %3, %2;" : "=r"(any) : "r"(lo32(closed)), "r"(hi32(closed)), "r"(one));
    const u32 valid = (u32)__popc(any);
    asm("mad.lo.u32 %0, %2, %4, %0;\n\tmad.lo.u32 %1, %3, %4, %1;"
        : "+r"(acc_lo), "+r"(acc_hi) : "r"(lo32(run)), "r"(hi32(run)), "r"(valid));
}
#endif

#if defined(__CUDACC__)
// index of the k-th (0-based, ascending) set bit of a non-empty mask, k < popc(mask): puttables()[k]
// (board.py:48-51).  Binary search on POPC (XU pipe); the conditional updates of k and of the bit
// base are predicated IMADs (FMA pipe), so a step costs the ALU pipe three instructions.
template <bool BYTE_LUT, typename RayTable>
__device__ __forceinline__ int kth_set_bit(u64 mask, int k, const RayTable &rays)
{
    const u32 one = kOpaqueOne;
    u32 v = lo32(mask);
    int base = 0;
    {
        const int c = __popc(v);
        const u32 hi = hi32(mask);
        asm("{\n\t.reg .pred p;\n\tsetp.ge.s32 p, %1, %3;\n\t@p mov.b32 %0, %4;\n\t@p mad.lo.s32 %2, %5, 32, %2;\n\t"
            "@p mad.lo.s32 %1, %3, %6, %1;\n\t}"
            : "+r"(v), "+r"(k), "+r"(base) : "r"(c), "r"(hi), "r"(one), "r"(0u - one));
    }
#define OBF_KTH_STEP(W)                                                                                            \
    {                                                                                                              \
        /* set bits among the low W of the window: shifted to the top (IMAD.SHL, FMA pipe) instead of masked (LOP3) */ \
        const int c = __popc(v << (32 - (W)));                                                                     \
        asm("{\n\t.reg .pred p;\n\tsetp.ge.s32 p, %1, %3;\n\t@p shr.u32 %0, %0, " #W ";\n\t"                        \
            "@p mad.lo.s32 %2, %4, " #W ", %2;\n\t@p mad.lo.s32 %1, %3, %5, %1;\n\t}"                                \
            : "+r"(v), "+r"(k), "+r"(base) : "r"(c), "r"(one), "r"(0u - one));                                     \
    }
    OBF_KTH_STEP(16)
    OBF_KTH_STEP(8)
    if (BYTE_LUT) {
        // the byte that holds the bit is the low byte of the window: its k-th set bit from [byte][k] (one LDS instead
        // of three more rounds of POPC + compare + shift)
        return base + (int)rays.byte(kKthBit64 * 8 + (v & 0xffu) * 8 + (u32)k);
    }
    OBF_KTH_STEP(4)
    OBF_KTH_STEP(2)
#undef OBF_KTH_STEP
    return base + ((k >= (int)(v & 1u)) ? 1 : 0);
}
struct NoTable { __device__ __forceinline__ u32 byte(u32) const { return 0; } };
__device__ __forceinline__ int kth_set_bit(u64 mask, int k) { return kth_set_bit<false>(mask, k, NoTable()); }
#endif

OBF_HD u32 umulhi32(u32 a, u32 b)
{
#if defined(__CUDA_ARCH__)
    return __umulhi(a, b);
#else
    return (u32)(((u64)a * b) >> 32);
#endif
}
// umulhi32(a, b) + c in one IMAD.HI
OBF_HD u32 madhi32(u32 a, u32 b, u32 c)
{
#if defined(__CUDA_ARCH__)
    u32 d;
    asm("mad.hi.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
#else
    return umulhi32(a, b) + c;
#endif
}
// byte y (0..7) of the pair (lo, hi) in byte 0 of the result; bytes 1..3 are junk (byte 0 of lo)
OBF_HD u32 byte_of(u32 lo, u32 hi, u32 y)
{
#if defined(__CUDA_ARCH__)
    u32 d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(lo), "r"(hi), "r"(y));     // (no masking of the selector: y < 8)
    return d;
#else
    return byte_perm(lo, hi, y);
#endif
}

// put() entirely by table look-up: the FOUR lines through the move (rank, file, two diagonals) instead of eight rays.
// Each line is gathered into a byte per colour, [position][opponent byte] gives the squares where an own disc would
// outflank, [position][those that are own] the flipped discs of the line, which are scattered back.  What makes this
// pay on a 32-bit machine whose ALU pipe is the bottleneck is that gather and scatter are multiplies (FMA pipe):
//   rank      the byte itself (PRMT); scatter = multiply by 1 << 8 * rank
//   file      multiply by 1 << (7 - file) moves the file onto bit 7 of every byte (no other bit lands there), the
//             high half of a multiply by 2^25 + 2^18 + 2^11 + 2^4 collects the four bits of a word (all 16 partial
//             products fall on different bits, so nothing carries); scatter = [byte] -> file-a column, times 1 << file
//   diagonal  a diagonal has one square per file: mask it, OR the two words, multiply by 0x01010101 -- the top byte is
//             the OR of the four bytes, bit j = file j; scatter = the byte times 0x01010101, masked with the diagonal
// and a byte with junk above it needs no cleaning where it is ANDed with a clean table byte.  27 ALU-pipe
// instructions for a move instead of 52, no rotated board, no POPC.  `one` = kOpaqueOne on the device (keeps the
// shifts and address additions on the FMA pipe), 1 on the host.
// LINE_DIAG: fetch the diagonal masks by diagonal number (15 entries each: lanes on the same diagonal share a word and
// the rest fall into different banks) instead of by square (64 entries: 4.8 wavefronts per load in the greedy kernel, which
// is bound by the shared-memory pipe); costs two IMADs, so the random playout kernel, whose LSU pipe idles, keeps the squares.
template <bool LINE_DIAG = false, typename RayTable>
OBF_HD u64 flips_lut(int s, u64 own, u64 opp, const RayTable &T, u32 one)
{
    const u32 y = (u32)s >> 3, x = (u32)s & 7u;
    const u32 olo = lo32(own), ohi = hi32(own), plo = lo32(opp), phi = hi32(opp);
    const u32 t1x = kRowOutflank64 * 8 + x * kLineStride, t2x = kRowFlip64 * 8 + x * kLineStride;      // tables of position x
    const u32 t1y = kRowOutflank64 * 8 + y * kLineStride, t2y = kRowFlip64 * 8 + y * kLineStride;
    const u32 shr24 = one << 8;                                  // v >> 24 == umulhi(v, 1 << 8)
    u32 f_lo, f_hi;
    {   // the rank
        const u32 ob = byte_of(olo, ohi, y);                     // byte 0 = the rank (bytes 1..3: junk)
        const u32 pb = byte_of(plo, phi, y) & 0xffu;
        const u32 flip = T.byte((T.byte(pb * one + t1x) & ob) * one + t2x);
        const u64 mul = T.word(kRankMul64 + y);
        f_lo = flip * lo32(mul);
        f_hi = flip * hi32(mul);
    }
    {   // the file
        const u64 fm = T.word(kFileMul64 + x);
        const u32 up = lo32(fm);
        const u32 kLo = 0x02040810u, kHi = 0x20408100u;          // bits 8k+7 -> bit k / bit 4+k of the high half
        const u32 pb = madhi32((plo * up) & 0x80808080u, kLo, umulhi32((phi * up) & 0x80808080u, kHi)) & 0xffu;
        const u32 ob = madhi32((olo * up) & 0x80808080u, kLo, umulhi32((ohi * up) & 0x80808080u, kHi));   // (junk above bit 7)
        const u32 flip = T.byte((T.byte(pb * one + t1y) & ob) * one + t2y);
        const u64 col = T.word(kSpread64 + flip);
        f_lo += lo32(col) * hi32(fm);
        f_hi += hi32(col) * hi32(fm);
    }
#define OBF_DIAGONAL(INDEX)                                                                                        \
    {                                                                                                              \
        const u64 d = T.word(INDEX);                                                                               \
        const u32 pb = umulhi32(((plo & lo32(d)) | (phi & hi32(d))) * 0x01010101u, shr24);                         \
        const u32 ob = umulhi32(((olo & lo32(d)) | (ohi & hi32(d))) * 0x01010101u, shr24);                         \
        const u32 r = T.byte((T.byte(pb * one + t1x) & ob) * one + t2x) * 0x01010101u;                            \
        f_lo |= r & lo32(d);                                                                                       \
        f_hi |= r & hi32(d);                                                                                       \
    }
    OBF_DIAGONAL(LINE_DIAG ? (x * one + (kLine9_64 + 7)) - y * one : kDiag9_64 + (u32)s)
    OBF_DIAGONAL(LINE_DIAG ? x * one + (y * one + kLine7_64) : kDiag7_64 + (u32)s)
#undef OBF_DIAGONAL
    return pack(f_lo, f_hi);
}

// Discs flipped by an `own` disc on the EMPTY square s (board.py:161-174); rays = table [4][64].
// BIT_LUT: take the move bit and its rotation from the table's fifth row (two LDS) instead of a variable
// 64-bit shift (two ALU instructions) + two BREVs.  Pays in the random playout kernel, whose LSU pipe idles
// (+1.1 %); costs the greedy kernel 0.8 % (its LSU pipe also carries the work-item lists), so it is a choice.
// ROW_LUT: the two horizontal rays through row_flips.
template <bool BIT_LUT = false, bool ROW_LUT = false, typename RayTable>
OBF_HD u64 flips_for(int s, u64 own, u64 opp, u64 own_r, u64 opp_r, const RayTable &rays)
{
    const int sr = 63 - s;
#if defined(__CUDA_ARCH__)
    const u64 x = BIT_LUT ? rays(kRayDirs, s) : 1ull << s;
    const u64 xr = BIT_LUT ? rays(kRayDirs, sr) : rev64(x);   // (two BREVs on the XU pipe, not two more ALU shifts)
    const u32 one = kOpaqueOne;
    u32 f_lo = 0, f_hi = 0, r_lo = 0, r_hi = 0;
    if (ROW_LUT) row_flips(s, own, opp, rays, f_lo, f_hi);
#pragma unroll
    for (int d = ROW_LUT ? 1 : 0; d < kRayDirs; d++) {
        ray_accumulate(f_lo, f_hi, x, rays(d, s), own, opp, one);
        ray_accumulate(r_lo, r_hi, xr, rays(d, sr), own_r, opp_r, one);
    }
    return pack(f_lo, f_hi) | rev64(pack(r_lo, r_hi));
#else
    const u64 x = 1ull << s, xr = 1ull << sr;
    u64 f = 0, fr = 0;
    if (ROW_LUT) {
        u32 f_lo = 0, f_hi = 0;
        row_flips(s, own, opp, rays, f_lo, f_hi);
        f = pack(f_lo, f_hi);
    }
    for (int d = ROW_LUT ? 1 : 0; d < kRayDirs; d++) {
        f |= ray_flips(x, rays(d, s), own, opp);
        fr |= ray_flips(xr, rays(d, sr), own_r, opp_r);
    }
    return f | rev64(fr);
#endif
}

}  // namespace obf
