// move_values.cuh -- the value of every move of a position, one (position, slot) item at a time.
//
// A row has kSlots = 65 entries, indexed by the move code: squares 0..63 and kPass = 64 (include/othello_b200.h,
// othello_search_moves / othello_solve_moves).
//
//   * search_slot: the minimax value of the subtree after the move, searched to depth - 1 further plies with a full
//     window and every node scored from the ROOT mover's side, as in obm::search_root.  The pass slot is the passed
//     position searched the same way: exactly the value search_root returns with move == kPass.  A full window makes
//     the value exact, so the row's maximum is search_root's value and its lowest arg-max search_root's move.
//   * solve_slot: the perfect-play value after the move from the mover's side, = minus the child's solve.  The pass
//     slot is obe::solve of the root itself: a root at kMaxEmpties empties that must pass tries the opponent's moves in
//     place, without a child frame (endgame.cuh's stack holds the nodes below kMaxEmpties empties only).
//
// A slot that is not a move of the position (an illegal square, the pass slot when the mover has a move, every slot of
// a game-over position, of overlapping colours or, for the solver, of a position with more than kMaxEmpties empties)
// gets the sentinel (NaN / kRefused) and 0 nodes; telling costs one move generation.  nodes = the positions the slot's
// search visited: a function of (position, slot, depth, weights) alone.
//
// Host+device like midgame.cuh and endgame.cuh: tests/move_values_host.cpp compiles this file with g++.
#pragma once
#include "midgame.cuh"

namespace obv {

using obf::u64;

constexpr int kSlots = 65;

template <typename RayTable>
OBF_HD float search_slot(u64 own, u64 opp, int slot, int depth, const float *w, const RayTable &rays, u64 &nodes,
                         obm::Frame *st)
{
    nodes = 0;
    if (own & opp) return NAN;
    const u64 legal = obf::legal_moves(own, opp);
    u64 c_own = opp, c_opp = own;                      // the pass: the same discs, the opponent to move
    if (slot < 64) {
        if (!((legal >> slot) & 1)) return NAN;
        const u64 f = obe::flips(slot, own, opp, rays);
        c_own = opp & ~f;
        c_opp = own | f | (1ull << slot);
    } else if (legal || !obf::legal_moves(opp, own)) {
        return NAN;
    }
    return -obm::search(c_own, c_opp, depth - 1, -INFINITY, INFINITY, -1, w, rays, nodes, st) + 0.0f;
}

template <typename RayTable>
OBF_HD int solve_slot(u64 own, u64 opp, int slot, const RayTable &rays, u64 &nodes, obe::Frame *st)
{
    nodes = 0;
    if ((own & opp) || obe::empties(own, opp) > obe::kMaxEmpties) return obe::kRefused;
    const u64 legal = obf::legal_moves(own, opp);
    if (slot == obe::kPass) {
        if (legal || !obf::legal_moves(opp, own)) return obe::kRefused;
        int move;
        return obe::solve(own, opp, rays, move, nodes, st);
    }
    if (!((legal >> slot) & 1)) return obe::kRefused;
    const u64 f = obe::flips(slot, own, opp, rays);
    return -obe::search(opp & ~f, own | f | (1ull << slot), -obe::kInf, obe::kInf, rays, nodes, st);
}

}  // namespace obv
