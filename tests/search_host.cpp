// tests/search_host.cpp -- TEST SCAFFOLDING: compiles subproc_b200/csrc/midgame.cuh for the host so the search the
// search kernel runs can be compared with the oracle without a GPU (and timed on one core by tools/bench_search.py).
// Build it with -std=c++17 (not gnu++17): g++ then contracts no float expression, and only the explicit fmaf fuses,
// as on the device.
#include "../subproc_b200/csrc/midgame.cuh"
#include "host_rays.h"

// black, white, turn (1 = Black, anything else = White; NULL = Black), weights [4][10], depth -> value, move, nodes
// (NULL = not wanted)
extern "C" void mg_search(const unsigned long long *black, const unsigned long long *white, const unsigned char *turn,
                          const float *weights, int depth, float *value, unsigned char *move, unsigned long long *nodes,
                          long n)
{
    obm::Frame st[obm::kFrames];
    for (long i = 0; i < n; i++) {
        const bool black_moves = turn ? turn[i] == 1 : true;
        int mv;
        unsigned long long cnt;
        value[i] = obm::search_root(black_moves ? black[i] : white[i], black_moves ? white[i] : black[i], depth, weights,
                                    Rays(), mv, cnt, st);
        move[i] = (unsigned char)mv;
        if (nodes) nodes[i] = cnt;
    }
}

// score(P, O) of colour P, the evaluation every leaf gets
extern "C" float mg_score(unsigned long long P, unsigned long long O, const float *weights)
{
    return obm::score(P, O, weights);
}
