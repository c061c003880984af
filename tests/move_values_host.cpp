// tests/move_values_host.cpp -- TEST SCAFFOLDING: compiles subproc_b200/csrc/move_values.cuh for the host so the rows
// the move-value kernels write can be compared with the oracle without a GPU, and with the kernels bit for bit on one.
// Build it with -std=c++17 (not gnu++17), as tests/search_host.cpp: only the explicit fmaf fuses, as on the device.
#include "../subproc_b200/csrc/move_values.cuh"

static unsigned long long g_rays[obf::kRayTable64];
static bool g_init = false;
struct Rays {
    unsigned long long operator()(int d, int s) const { return g_rays[d * 64 + s]; }
    unsigned long long word(unsigned i) const { return g_rays[i]; }
    unsigned byte(unsigned i) const { return ((const unsigned char *)g_rays)[i]; }     // (little-endian host)
};

// the ray table; call once before the row functions run on several threads
extern "C" void mv_init(void)
{
    if (!g_init) {
        for (int i = 0; i < obf::kRayTable64; i++) g_rays[i] = obf::make_table_word(i);
        g_init = true;
    }
}

// black, white, turn (1 = Black, anything else = White; NULL = Black), weights [4][10], depth -> values [n][65],
// nodes [n][65] (NULL = not wanted)
extern "C" void mv_search_moves(const unsigned long long *black, const unsigned long long *white,
                                const unsigned char *turn, const float *weights, int depth, float *values,
                                unsigned long long *nodes, long n)
{
    mv_init();
    obm::Frame st[obm::kFrames];
    for (long i = 0; i < n; i++) {
        const bool black_moves = turn ? turn[i] == 1 : true;
        for (int s = 0; s < obv::kSlots; s++) {
            unsigned long long cnt;
            values[i * obv::kSlots + s] = obv::search_slot(black_moves ? black[i] : white[i],
                                                           black_moves ? white[i] : black[i], s, depth, weights, Rays(),
                                                           cnt, st);
            if (nodes) nodes[i * obv::kSlots + s] = cnt;
        }
    }
}

// black, white, turn -> values [n][65], nodes [n][65] (NULL = not wanted)
extern "C" void mv_solve_moves(const unsigned long long *black, const unsigned long long *white,
                               const unsigned char *turn, int *values, unsigned long long *nodes, long n)
{
    mv_init();
    obe::Frame st[obe::kFrames];
    for (long i = 0; i < n; i++) {
        const bool black_moves = turn ? turn[i] == 1 : true;
        for (int s = 0; s < obv::kSlots; s++) {
            unsigned long long cnt;
            values[i * obv::kSlots + s] = obv::solve_slot(black_moves ? black[i] : white[i],
                                                          black_moves ? white[i] : black[i], s, Rays(), cnt, st);
            if (nodes) nodes[i * obv::kSlots + s] = cnt;
        }
    }
}
