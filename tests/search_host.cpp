// tests/search_host.cpp -- TEST SCAFFOLDING: compiles subproc_b200/csrc/midgame.cuh for the host so the search the
// search kernel runs can be compared with the oracle without a GPU (and timed on one core by tools/bench_search.py).
// Build it with -std=c++17 (not gnu++17): g++ then contracts no float expression, and only the explicit fmaf fuses,
// as on the device.
#include "../subproc_b200/csrc/midgame.cuh"

static unsigned long long g_rays[obf::kRayTable64];
static bool g_init = false;
struct Rays {
    unsigned long long operator()(int d, int s) const { return g_rays[d * 64 + s]; }
    unsigned long long word(unsigned i) const { return g_rays[i]; }
    unsigned byte(unsigned i) const { return ((const unsigned char *)g_rays)[i]; }     // (little-endian host)
};

// black, white, turn (1 = Black, anything else = White; NULL = Black), weights [4][10], depth -> value, move, nodes
// (NULL = not wanted)
extern "C" void mg_search(const unsigned long long *black, const unsigned long long *white, const unsigned char *turn,
                          const float *weights, int depth, float *value, unsigned char *move, unsigned long long *nodes,
                          long n)
{
    if (!g_init) {
        for (int i = 0; i < obf::kRayTable64; i++) g_rays[i] = obf::make_table_word(i);
        g_init = true;
    }
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
