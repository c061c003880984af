// midgame.cuh -- depth-limited search on the linear evaluation: the minimax value and best move of one position, in
// one lane.
//
// Semantics (include/othello_b200.h, othello_search): every node is scored from the ROOT mover's side,
// score(P, O) = W[phase(P|O)] . (mobility(P), a..h of P) + W[phase][9] with P = the root mover's discs -- the fp32 value
// othello_eval returns, same fmaf order, intercept first.  Plies alternate from the root; a pass is a ply and uses one
// level of depth; a node is a leaf `depth` plies below the root or when neither side can move.  value = plain minimax
// over the leaf scores (max on the root mover's plies, min on the opponent's), -0.0 returned as +0.0; move = the lowest
// square whose subtree reaches the value, OTHELLO_PASS when the root mover must pass (value: the passed position
// searched to depth - 1), OTHELLO_NO_MOVE when the game is over (value: score(root)).  The weights are finite.
//
// Structure (DESIGN.md section 13):
//   * negamax over sgn * score (sgn = +1 where the root mover is to move) with fail-soft alpha-beta on floats; max and
//     min are exact, so pruning and move order change the node count and the time, never the value;
//   * nodes with more than kLowDepth plies below them live on an explicit stack of Frames (the caller's array: local
//     memory in the kernel); their moves are tried best shallow score first (kSortDepth plies and up), ties in
//     ascending square order;
//   * nodes with at most kLowDepth plies below them are searched by Low<R>, a template-unrolled recursion whose levels
//     the compiler keeps in registers (perft's Dfs<R> pattern), moves in ascending square order; a node one ply above
//     the leaves scores its children directly (Low<0> inlined: flip, the root mover's mobility, the 9-term dot
//     product -- the greedy kernel's work per child);
//   * the root tries its moves in the same order as a stack node.  The first gets a full window; every later one a
//     null window that asks whether it replaces the best so far -- strictly better for a higher square, at least as
//     good for a lower one -- and, if it does, the window (lo, +inf) for its exact value.  So the value is exact and
//     the move is the lowest square that reaches it, whatever the order.
//
// All functions are host+device like endgame.cuh, so tests/ compiles this very file with g++ (-std=c++17: no float
// contraction, only the explicit fmaf fuses) and checks it against the oracle's plain minimax; the host build is also
// the CPU figure of tools/bench_search.py.
#pragma once
#include <math.h>
#include <string.h>
#include "endgame.cuh"

namespace obm {

using obf::u64;
using obf::u32;

constexpr int kMaxDepth = 12;                    // OTHELLO_SEARCH_MAX_DEPTH
constexpr int kPass = obe::kPass;                // OTHELLO_PASS
constexpr int kNoMove = obe::kNoMove;            // OTHELLO_NO_MOVE
constexpr int kMaxMoves = 64;                    // legal moves of any position (at most its empty squares)

#ifndef OBM_LOW_DEPTH
#define OBM_LOW_DEPTH 3
#endif
#ifndef OBM_SORT_DEPTH
#define OBM_SORT_DEPTH 3
#endif
constexpr int kLowDepth = OBM_LOW_DEPTH;         // at most this many plies below: register-resident Low<R>
constexpr int kSortDepth = OBM_SORT_DEPTH;       // stack nodes and the root with at least this many plies below order
static_assert(kLowDepth >= 1 && kLowDepth < kMaxDepth && kLowDepth <= 4, "kLowDepth (search(): add the cases)");
// Frame 0 holds the root's move order.  A child of the root has at most kMaxDepth - 1 plies below it, so the stack
// holds the nodes with kLowDepth + 1 .. kMaxDepth - 1 plies below them of one path: frames 1 .. kFrames - 1.
constexpr int kFrames = kMaxDepth - kLowDepth;

#if defined(__CUDA_ARCH__)
#define OBM_CHECK_FRAME(sp) ((void)0)
#else
#define OBM_CHECK_FRAME(sp) do { if ((sp) >= kFrames) __builtin_trap(); } while (0)
#endif

// ---- the evaluation, host+device (ob::eval_linear is device-only) --------------------------------------------------
// square-class masks a..h (parameter_progress_position_moves_learn.py:9-16), the same as ob::kClassMask
OBF_HD constexpr u64 class_mask(int k)
{
    return k == 0 ? 0x8100000000000081ull : k == 1 ? 0x4281000000008142ull : k == 2 ? 0x0042000000004200ull
         : k == 3 ? 0x2400810000810024ull : k == 4 ? 0x1800008181000018ull : k == 5 ? 0x003C424242423C00ull
         : k == 6 ? 0x0000240000240000ull : 0x0000183C3C180000ull;
}

// phase row of a disc count: shards (0,16),(17,32),(33,48),(49,64) inclusive
OBF_HD int phase_row(int discs)
{
    const int r = ((discs + 15) >> 4) - 1;
    return r < 0 ? 0 : (r > 3 ? 3 : r);
}

// w[phase] . (mobility, a..h) + w[phase][9] of colour P: ob::eval_linear's operations in its order
OBF_HD float score(u64 P, u64 O, const float *w)
{
    const float *row = w + 10 * phase_row(obf::popc64(P | O));
    float acc = row[9];
    acc = fmaf(row[0], (float)obf::mobility(P, O), acc);
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int k = 0; k < 8; k++) acc = fmaf(row[1 + k], (float)obf::popc64(P & class_mask(k)), acc);
    return acc;
}

// the leaf value of a node, from its mover's (`own`) side: sgn = +1 when `own` is the root mover
OBF_HD float leaf(u64 own, u64 opp, int sgn, const float *w)
{
    return sgn > 0 ? score(own, opp, w) : -score(opp, own, w);
}

// order-preserving map float -> u32 (larger float <=> larger unsigned); -0.0 is folded into +0.0
OBF_HD u32 ordered_bits(float v)
{
    v += 0.0f;
#if defined(__CUDA_ARCH__)
    const u32 u = __float_as_uint(v);
#else
    u32 u;
    memcpy(&u, &v, sizeof u);
#endif
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// ---- the last plies: register-resident, ascending squares -----------------------------------------------------------
template <int R> struct Low {
    template <typename RayTable>
    static OBF_HD float run(u64 own, u64 opp, float alpha, float beta, int sgn, const float *w, const RayTable &rays,
                            u64 &nodes)
    {
        nodes++;
        const u64 legal = obf::legal_moves(own, opp);
        if (!legal) {
            if (!obf::legal_moves(opp, own)) return leaf(own, opp, sgn, w);
            return -Low<R - 1>::run(opp, own, -beta, -alpha, -sgn, w, rays, nodes);      // a pass: one ply
        }
        float best = -INFINITY;
        const u64 own_r = obf::rev64(own), opp_r = obf::rev64(opp);
        for (u64 rem = legal; rem; rem &= rem - 1) {
            const int sq = obe::ctz64(rem);
            const u64 f = obf::flips_for(sq, own, opp, own_r, opp_r, rays);
            const float v = -Low<R - 1>::run(opp & ~f, own | f | (1ull << sq), -beta, -alpha, -sgn, w, rays, nodes);
            if (v > best) {
                best = v;
                if (v > alpha) { alpha = v; if (alpha >= beta) break; }
            }
        }
        return best;
    }
};

template <> struct Low<0> {
    template <typename RayTable>
    static OBF_HD float run(u64 own, u64 opp, float, float, int sgn, const float *w, const RayTable &, u64 &nodes)
    {
        nodes++;
        return leaf(own, opp, sgn, w);
    }
};

// ---- the upper levels: an explicit stack ------------------------------------------------------------------------
struct Frame {
    u64 own, opp;                      // the node, `own` to move
    float alpha, beta, best;           // window and best value, from `own`'s side
    signed char sgn;                   // +1 when `own` is the root mover
    unsigned char rem;                 // plies below the node
    unsigned char n, i;                // moves in `order`, next one to try
    unsigned char order[kMaxMoves];    // squares (or kPass), in the order they are tried
};

// The legal moves of `own` into order[], best shallow score (the child's leaf value from `own`'s side) first, ties
// and unsorted lists in ascending square order.  Returns their number.
template <typename RayTable>
OBF_HD int order_moves(unsigned char *order, u64 own, u64 opp, u64 legal, int sgn, bool sort, const float *w,
                       const RayTable &rays)
{
    int n = 0;
    if (!sort) {
        for (u64 rem = legal; rem; rem &= rem - 1) order[n++] = (unsigned char)obe::ctz64(rem);
        return n;
    }
    // insertion sort on (descending score with its low 6 bits dropped, square): the order only steers pruning
    u32 key[kMaxMoves];
    const u64 own_r = obf::rev64(own), opp_r = obf::rev64(opp);
    for (u64 rem = legal; rem; rem &= rem - 1) {
        const int sq = obe::ctz64(rem);
        const u64 f = obf::flips_for(sq, own, opp, own_r, opp_r, rays);
        const float v = leaf(own | f | (1ull << sq), opp & ~f, sgn, w);
        const u32 k = (~ordered_bits(v) & ~63u) | (u32)sq;
        int j = n++;
        for (; j > 0 && key[j - 1] > k; j--) key[j] = key[j - 1];
        key[j] = k;
    }
    for (int j = 0; j < n; j++) order[j] = (unsigned char)(key[j] & 63u);
    return n;
}

// Set up frame F for a node with more than kLowDepth plies below it.  Returns true (and the value in `value`) when
// the game is over there.  A node whose mover must pass gets the one move kPass.
template <typename RayTable>
OBF_HD bool enter(Frame &F, u64 own, u64 opp, int rem, float alpha, float beta, int sgn, const float *w,
                  const RayTable &rays, u64 &nodes, float &value)
{
    nodes++;
    const u64 legal = obf::legal_moves(own, opp);
    F.own = own; F.opp = opp; F.alpha = alpha; F.beta = beta; F.best = -INFINITY;
    F.sgn = (signed char)sgn; F.rem = (unsigned char)rem; F.i = 0;
    if (!legal) {
        if (!obf::legal_moves(opp, own)) { value = leaf(own, opp, sgn, w); return true; }
        F.order[0] = (unsigned char)kPass;
        F.n = 1;
        return false;
    }
    F.n = (unsigned char)order_moves(F.order, own, opp, legal, sgn, rem >= kSortDepth, w, rays);
    return false;
}

OBF_HD void record(Frame &F, float v)
{
    if (v > F.best) {
        F.best = v;
        if (v > F.alpha) F.alpha = v;
    }
}

// fail-soft alpha-beta value of a node with more than kLowDepth plies below it; st: the frames of the stack
template <typename RayTable>
OBF_HD float search_stack(u64 own, u64 opp, int rem, float alpha, float beta, int sgn, const float *w,
                          const RayTable &rays, u64 &nodes, Frame *st)
{
    float value;
    if (enter(st[0], own, opp, rem, alpha, beta, sgn, w, rays, nodes, value)) return value;
    int sp = 0;
    for (;;) {
        Frame &F = st[sp];
        if (F.i < F.n && F.alpha < F.beta) {
            const int sq = F.order[F.i++];
            u64 c_own = F.own, c_opp = F.opp;
            if (sq != kPass) {
                const u64 f = obe::flips(sq, F.own, F.opp, rays);
                c_opp = F.own | f | (1ull << sq);
                c_own = F.opp & ~f;
            } else {
                c_own = F.opp; c_opp = F.own;
            }
            float v;                                   // the child's value, from its mover's side
            if (F.rem - 1 == kLowDepth) {
                v = Low<kLowDepth>::run(c_own, c_opp, -F.beta, -F.alpha, -F.sgn, w, rays, nodes);
            } else {
                OBM_CHECK_FRAME(sp + 2);               // (st = the caller's frames + 1)
                if (!enter(st[sp + 1], c_own, c_opp, F.rem - 1, -F.beta, -F.alpha, -F.sgn, w, rays, nodes, v)) {
                    sp++;
                    continue;
                }
            }
            record(F, -v);
            continue;
        }
        const float v = F.best;
        if (sp == 0) return v;
        sp--;
        record(st[sp], -v);
    }
}

template <typename RayTable>
OBF_HD float search(u64 own, u64 opp, int rem, float alpha, float beta, int sgn, const float *w, const RayTable &rays,
                    u64 &nodes, Frame *st)
{
    switch (rem) {
    case 0: return Low<0>::run(own, opp, alpha, beta, sgn, w, rays, nodes);
    case 1: return Low<1>::run(own, opp, alpha, beta, sgn, w, rays, nodes);
#if OBM_LOW_DEPTH >= 2
    case 2: return Low<2>::run(own, opp, alpha, beta, sgn, w, rays, nodes);
#endif
#if OBM_LOW_DEPTH >= 3
    case 3: return Low<3>::run(own, opp, alpha, beta, sgn, w, rays, nodes);
#endif
#if OBM_LOW_DEPTH >= 4
    case 4: return Low<4>::run(own, opp, alpha, beta, sgn, w, rays, nodes);
#endif
    default: return search_stack(own, opp, rem, alpha, beta, sgn, w, rays, nodes, st + 1);
    }
}

// The value and move of one root position (own to move), 1 <= depth <= kMaxDepth; st: kFrames frames.  nodes =
// positions the search visited (each one generated its moves, or was scored as a leaf): a function of the position,
// the depth and the weights alone.  Overlapping colours: NaN, kNoMove, 0 nodes.
template <typename RayTable>
OBF_HD float search_root(u64 own, u64 opp, int depth, const float *w, const RayTable &rays, int &move, u64 &nodes,
                         Frame *st)
{
    nodes = 0;
    move = kNoMove;
    if (own & opp) return NAN;
    nodes = 1;
    const u64 legal = obf::legal_moves(own, opp);
    if (!legal) {
        if (!obf::legal_moves(opp, own)) return score(own, opp, w) + 0.0f;
        move = kPass;
        return -search(opp, own, depth - 1, -INFINITY, INFINITY, -1, w, rays, nodes, st) + 0.0f;
    }
    unsigned char *order = st[0].order;
    const int n = order_moves(order, own, opp, legal, 1, depth >= kSortDepth, w, rays);
    float best = -INFINITY;
    int best_sq = kNoMove;
    for (int i = 0; i < n; i++) {
        const int sq = order[i];
        const u64 f = obe::flips(sq, own, opp, rays);
        const u64 c_own = opp & ~f, c_opp = own | f | (1ull << sq);
        // (lo, hi): the full window for the first move; then the null window above lo, where lo = the largest value
        // that does NOT replace the best (best itself for a higher square, the float below it for a lower one), and,
        // if the move does replace it, (lo, +inf) for its exact value
        const bool first = best_sq == kNoMove;
        const float lo = first ? -INFINITY : (sq > best_sq ? best : nextafterf(best, -INFINITY));
        float hi = first ? INFINITY : nextafterf(lo, INFINITY);
        float v;
        for (;;) {
            v = -search(c_own, c_opp, depth - 1, -hi, -lo, -1, w, rays, nodes, st);
            if (hi == INFINITY || v <= lo || depth == 1) break;      // (a leaf's value is exact in any window)
            hi = INFINITY;
        }
        if (first || v > lo) { best = v; best_sq = sq; }
    }
    move = best_sq;
    return best + 0.0f;
}

}  // namespace obm
