// tests/solve_host.cpp -- TEST SCAFFOLDING: compiles subproc_b200/csrc/endgame.cuh for the host so the exact search
// the solve kernel runs can be compared with the oracle without a GPU (and timed on one core by tools/bench_solve.py).
#include "../subproc_b200/csrc/endgame.cuh"

static unsigned long long g_rays[obf::kRayTable64];
static bool g_init = false;
struct Rays {
    unsigned long long operator()(int d, int s) const { return g_rays[d * 64 + s]; }
    unsigned long long word(unsigned i) const { return g_rays[i]; }
    unsigned byte(unsigned i) const { return ((const unsigned char *)g_rays)[i]; }     // (little-endian host)
};

// black, white, turn (1 = Black, anything else = White; NULL = Black) -> value, move, nodes (NULL = not wanted)
extern "C" void eg_solve(const unsigned long long *black, const unsigned long long *white, const unsigned char *turn,
                         int *value, unsigned char *move, unsigned long long *nodes, long n)
{
    if (!g_init) {
        for (int i = 0; i < obf::kRayTable64; i++) g_rays[i] = obf::make_table_word(i);
        g_init = true;
    }
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
