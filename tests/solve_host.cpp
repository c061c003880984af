// tests/solve_host.cpp -- TEST SCAFFOLDING: compiles subproc_b200/csrc/endgame.cuh for the host so the exact search
// the solve kernel runs can be compared with the oracle without a GPU (and timed on one core by tools/bench_solve.py).
#include "../subproc_b200/csrc/endgame.cuh"
#include "host_rays.h"

// black, white, turn (1 = Black, anything else = White; NULL = Black) -> value, move, nodes (NULL = not wanted)
extern "C" void eg_solve(const unsigned long long *black, const unsigned long long *white, const unsigned char *turn,
                         int *value, unsigned char *move, unsigned long long *nodes, long n)
{
    obe::Frame st[obe::kFrames];
    for (long i = 0; i < n; i++) {
        const bool black_moves = turn ? turn[i] == 1 : true;
        int mv;
        unsigned long long cnt;
        value[i] = obe::solve(black_moves ? black[i] : white[i], black_moves ? white[i] : black[i], Rays(), mv, cnt, st);
        move[i] = (unsigned char)mv;
        if (nodes) nodes[i] = cnt;
    }
}
