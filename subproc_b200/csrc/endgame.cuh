// endgame.cuh -- exact endgame search: the perfect-play value and best move of one position, in one lane.
//
// Semantics (include/othello_b200.h, othello_solve): value = own - opponent discs of the terminal position reached
// under perfect play, "own" = the side to move at the root; the game ends when neither side can move (board.py:57-58);
// a pass is a ply; empty squares left at the end are NOT given to the winner (the reference's own scoring,
// game_runner.py:194-199 and progress_position_moves_learn.py:55 -- not the Edax / WTHOR convention).  move = the
// lowest square among the moves that reach the value, OTHELLO_PASS when the mover must pass, OTHELLO_NO_MOVE when the
// game is over.
//
// Structure (DESIGN.md section 12):
//   * negamax with fail-soft alpha-beta;
//   * nodes with more than kLowEmpties empties live on an explicit stack of Frames (the caller's array: local memory
//     in the kernel); their moves are tried fewest-opponent-replies first (kSortEmpties and up), which changes the
//     node count and the time, never the value;
//   * nodes with at most kLowEmpties empties are searched by Low<E>, a template-unrolled recursion whose levels the
//     compiler keeps in registers (perft's Dfs<R> pattern), moves in ascending square order;
//   * the last empty square is scored from the flip count of its one move (or of the opponent's, if the mover must
//     pass) without generating moves;
//   * a pass never costs a stack level: the node swaps the colours and negates its window in place.
// The root tries its moves in ascending square order: the first with a full window, every later one with a null
// window around the best value so far (a later, higher square must be strictly better to replace it), and a move
// that is better is searched again with the window (best, +inf) -- so the value is exact and the move is the lowest
// square that reaches it.
//
// All functions are host+device like fastboard.cuh, so tests/ compiles this very file with g++ and checks it against
// the oracle's plain negamax; the host build is also the CPU figure of tools/bench_solve.py.
#pragma once
#include "fastboard.cuh"

namespace obe {

using obf::u64;
using obf::u32;

#ifndef OBE_MAX_EMPTIES
#define OBE_MAX_EMPTIES 24
#endif
constexpr int kMaxEmpties = OBE_MAX_EMPTIES;     // OTHELLO_SOLVE_MAX_EMPTIES (smaller only in tests/ host builds)
constexpr int kRefused = -128;         // OTHELLO_SOLVE_REFUSED
constexpr int kPass = 64;              // OTHELLO_PASS
constexpr int kNoMove = 255;           // OTHELLO_NO_MOVE
constexpr int kInf = 65;               // beyond every value (-64..64)

#ifndef OBE_LOW_EMPTIES
#define OBE_LOW_EMPTIES 6
#endif
#ifndef OBE_SORT_EMPTIES
#define OBE_SORT_EMPTIES 8
#endif
constexpr int kLowEmpties = OBE_LOW_EMPTIES;     // at most this many empties: register-resident Low<E>
constexpr int kSortEmpties = OBE_SORT_EMPTIES;   // stack nodes with at least this many empties order their moves
static_assert(kLowEmpties >= 1 && kLowEmpties < kMaxEmpties, "kLowEmpties");
// The root is not on the stack, and every child of the root has at most kMaxEmpties - 1 empties (a root pass is
// searched in place, see solve()); the stack holds the nodes with kLowEmpties + 1 .. kMaxEmpties - 1 empties of one
// path.  A pass inside the tree keeps the level it is found on.
constexpr int kFrames = kMaxEmpties - 1 - kLowEmpties;

// The host build (tests/) checks the stack bound on every push; the kernel relies on the argument above.
#if defined(__CUDA_ARCH__)
#define OBE_CHECK_FRAME(sp) ((void)0)
#else
#define OBE_CHECK_FRAME(sp) do { if ((sp) >= kFrames) __builtin_trap(); } while (0)
#endif

OBF_HD int ctz64(u64 v)
{
#if defined(__CUDA_ARCH__)
    return __ffsll((long long)v) - 1;
#else
    return __builtin_ctzll(v);
#endif
}

OBF_HD int disc_diff(u64 own, u64 opp) { return obf::popc64(own) - obf::popc64(opp); }
OBF_HD int empties(u64 own, u64 opp) { return 64 - obf::popc64(own | opp); }

template <typename RayTable>
OBF_HD u64 flips(int sq, u64 own, u64 opp, const RayTable &rays)
{
    return obf::flips_for(sq, own, opp, obf::rev64(own), obf::rev64(opp), rays);
}

// ---- the last few empties: register-resident, ascending squares -------------------------------------------------
template <int E> struct Low {
    template <typename RayTable>
    static OBF_HD int run(u64 own, u64 opp, int alpha, int beta, const RayTable &rays, u64 &nodes)
    {
        nodes++;
        u64 legal = obf::legal_moves(own, opp);
        int sign = 1;
        if (!legal) {                                  // pass in place: same level, colours swapped, window negated
            legal = obf::legal_moves(opp, own);
            if (!legal) return disc_diff(own, opp);
            const u64 t = own; own = opp; opp = t;
            const int a = alpha; alpha = -beta; beta = -a;
            sign = -1;
        }
        int best = -kInf;
        const u64 own_r = obf::rev64(own), opp_r = obf::rev64(opp);
        for (u64 rem = legal; rem; rem &= rem - 1) {
            const int sq = ctz64(rem);
            const u64 f = obf::flips_for(sq, own, opp, own_r, opp_r, rays);
            const int v = -Low<E - 1>::run(opp & ~f, own | f | (1ull << sq), -beta, -alpha, rays, nodes);
            if (v > best) {
                best = v;
                if (v > alpha) { alpha = v; if (alpha >= beta) break; }
            }
        }
        return sign * best;
    }
};

// one empty square: the move there, else the opponent's, else the game ends with it empty
template <> struct Low<1> {
    template <typename RayTable>
    static OBF_HD int run(u64 own, u64 opp, int, int, const RayTable &rays, u64 &nodes)
    {
        nodes++;
        const int sq = ctz64(~(own | opp));
        const int d = disc_diff(own, opp);
        u64 f = flips(sq, own, opp, rays);
        if (f) return d + 1 + 2 * obf::popc64(f);
        f = flips(sq, opp, own, rays);
        if (f) return d - 1 - 2 * obf::popc64(f);
        return d;
    }
};

template <> struct Low<0> {
    template <typename RayTable>
    static OBF_HD int run(u64 own, u64 opp, int, int, const RayTable &, u64 &nodes)
    {
        nodes++;
        return disc_diff(own, opp);
    }
};

// ---- the upper levels: an explicit stack ---------------------------------------------------------------------
struct Frame {
    u64 own, opp;                      // the mover's discs after a pass swap, if any
    int alpha, beta, best;             // window and best value, from `own`'s side
    int sign;                          // -1 when the node's mover passed (own / opp swapped, window negated)
    int n, i;                          // moves in `order`, next one to try
    unsigned char order[kMaxEmpties];  // squares, in the order they are tried
};

// Set up frame F for a position with more than kLowEmpties empties.  Returns true (and the value in `leaf`) when
// the game is over there.
template <typename RayTable>
OBF_HD bool enter(Frame &F, u64 own, u64 opp, int alpha, int beta, const RayTable &rays, u64 &nodes, int &leaf)
{
    nodes++;
    u64 legal = obf::legal_moves(own, opp);
    F.sign = 1;
    if (!legal) {
        legal = obf::legal_moves(opp, own);
        if (!legal) { leaf = disc_diff(own, opp); return true; }
        const u64 t = own; own = opp; opp = t;
        const int a = alpha; alpha = -beta; beta = -a;
        F.sign = -1;
    }
    F.own = own; F.opp = opp; F.alpha = alpha; F.beta = beta; F.best = -kInf; F.i = 0;
    int n = 0;
    if (empties(own, opp) >= kSortEmpties) {
        // fewest opponent replies first; ties in ascending square order (insertion sort on mobility * 64 + square)
        unsigned short key[kMaxEmpties];
        const u64 own_r = obf::rev64(own), opp_r = obf::rev64(opp);
        for (u64 rem = legal; rem; rem &= rem - 1) {
            const int sq = ctz64(rem);
            const u64 f = obf::flips_for(sq, own, opp, own_r, opp_r, rays);
            const unsigned short k = (unsigned short)(obf::mobility(opp & ~f, own | f | (1ull << sq)) * 64 + sq);
            int j = n++;
            for (; j > 0 && key[j - 1] > k; j--) key[j] = key[j - 1];
            key[j] = k;
        }
        for (int j = 0; j < n; j++) F.order[j] = (unsigned char)(key[j] & 63);
    } else {
        for (u64 rem = legal; rem; rem &= rem - 1) F.order[n++] = (unsigned char)ctz64(rem);
    }
    F.n = n;
    return false;
}

OBF_HD void record(Frame &F, int v)
{
    if (v > F.best) {
        F.best = v;
        if (v > F.alpha) F.alpha = v;
    }
}

// fail-soft alpha-beta value of a position with more than kLowEmpties empties; st: kFrames frames
template <typename RayTable>
OBF_HD int search_stack(u64 own, u64 opp, int alpha, int beta, const RayTable &rays, u64 &nodes, Frame *st)
{
    int leaf;
    if (enter(st[0], own, opp, alpha, beta, rays, nodes, leaf)) return leaf;
    int sp = 0;
    for (;;) {
        Frame &F = st[sp];
        if (F.i < F.n && F.alpha < F.beta) {
            const int sq = F.order[F.i++];
            const u64 f = flips(sq, F.own, F.opp, rays);
            const u64 c_own = F.opp & ~f, c_opp = F.own | f | (1ull << sq);
            int v;
            if (empties(c_own, c_opp) <= kLowEmpties) {
                v = Low<kLowEmpties>::run(c_own, c_opp, -F.beta, -F.alpha, rays, nodes);
            } else {
                OBE_CHECK_FRAME(sp + 1);
                if (!enter(st[sp + 1], c_own, c_opp, -F.beta, -F.alpha, rays, nodes, v)) {
                    sp++;
                    continue;
                }
            }
            record(F, -v);
            continue;
        }
        const int v = F.sign * F.best;                 // the node's value from the side that entered it
        if (sp == 0) return v;
        sp--;
        record(st[sp], -v);
    }
}

template <typename RayTable>
OBF_HD int search(u64 own, u64 opp, int alpha, int beta, const RayTable &rays, u64 &nodes, Frame *st)
{
    switch (empties(own, opp)) {
    case 0: return Low<0>::run(own, opp, alpha, beta, rays, nodes);
    case 1: return Low<1>::run(own, opp, alpha, beta, rays, nodes);
#if OBE_LOW_EMPTIES >= 2
    case 2: return Low<2>::run(own, opp, alpha, beta, rays, nodes);
#endif
#if OBE_LOW_EMPTIES >= 3
    case 3: return Low<3>::run(own, opp, alpha, beta, rays, nodes);
#endif
#if OBE_LOW_EMPTIES >= 4
    case 4: return Low<4>::run(own, opp, alpha, beta, rays, nodes);
#endif
#if OBE_LOW_EMPTIES >= 5
    case 5: return Low<5>::run(own, opp, alpha, beta, rays, nodes);
#endif
#if OBE_LOW_EMPTIES >= 6
    case 6: return Low<6>::run(own, opp, alpha, beta, rays, nodes);
#endif
#if OBE_LOW_EMPTIES >= 7
    case 7: return Low<7>::run(own, opp, alpha, beta, rays, nodes);
#endif
#if OBE_LOW_EMPTIES >= 8
    case 8: return Low<8>::run(own, opp, alpha, beta, rays, nodes);
#endif
    default: return search_stack(own, opp, alpha, beta, rays, nodes, st);
    }
}
static_assert(kLowEmpties <= 8, "search(): add the cases");

// The value and move of one root position (own to move).  nodes = positions the search visited (each one generated
// its moves, or scored its last empty square): a function of the position alone.
// A root whose mover must pass is searched in place, like every other pass: the opponent's moves are tried from the
// root itself and the value is negated, so every child of the root has fewer empties than the root (kFrames).
template <typename RayTable>
OBF_HD int solve(u64 own, u64 opp, const RayTable &rays, int &move, u64 &nodes, Frame *st)
{
    nodes = 0;
    move = kNoMove;
    if ((own & opp) || empties(own, opp) > kMaxEmpties) return kRefused;
    nodes = 1;
    u64 legal = obf::legal_moves(own, opp);
    const bool pass = !legal;
    if (pass) {
        legal = obf::legal_moves(opp, own);
        if (!legal) return disc_diff(own, opp);
        const u64 t = own; own = opp; opp = t;
    }
    int best = -kInf, best_sq = kNoMove;
    for (u64 rem = legal; rem; rem &= rem - 1) {
        if (best == 64) break;                         // nothing is strictly better
        const int sq = ctz64(rem);
        const u64 f = flips(sq, own, opp, rays);
        const u64 c_own = opp & ~f, c_opp = own | f | (1ull << sq);
        // root window (lo, hi): full for the first move, then (best, best + 1) -- is this higher square strictly
        // better? -- and, if it is, (best, +inf) for its exact value
        const int lo = best_sq == kNoMove ? -kInf : best;
        int hi = best_sq == kNoMove ? kInf : best + 1;
        int v;
        for (;;) {
            v = -search(c_own, c_opp, -hi, -lo, rays, nodes, st);
            if (hi == kInf || v <= best) break;
            hi = kInf;
        }
        if (v > best) { best = v; best_sq = sq; }
    }
    move = pass ? kPass : best_sq;
    return pass ? -best : best;
}

}  // namespace obe
