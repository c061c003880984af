// tests/fastboard_host.cpp -- TEST SCAFFOLDING: compiles subproc_b200/csrc/fastboard.cuh for the
// host so the exact source the kernels use can be compared with the oracle without a GPU.
#include "../subproc_b200/csrc/fastboard.cuh"
#include "host_rays.h"

extern "C" void fb_legal(const unsigned long long *own, const unsigned long long *opp, unsigned long long *out, long n)
{
    for (long i = 0; i < n; i++) out[i] = obf::legal_moves(own[i], opp[i]);
}

extern "C" void fb_flips(const unsigned long long *own, const unsigned long long *opp, const unsigned char *sq,
                         unsigned long long *out, long n)
{
    for (long i = 0; i < n; i++) {
        const unsigned long long x = 1ull << sq[i];
        out[i] = ((own[i] | opp[i]) & x) ? 0ull
                 : obf::flips_for(sq[i], own[i], opp[i], obf::rev64(own[i]), obf::rev64(opp[i]), Rays());
    }
}

// the same with the horizontal rays through the rank look-up (what the playout kernel runs)
extern "C" void fb_flips_rowlut(const unsigned long long *own, const unsigned long long *opp, const unsigned char *sq,
                                unsigned long long *out, long n)
{
    for (long i = 0; i < n; i++) {
        const unsigned long long x = 1ull << sq[i];
        out[i] = ((own[i] | opp[i]) & x) ? 0ull
                 : obf::flips_for<false, true>(sq[i], own[i], opp[i], obf::rev64(own[i]), obf::rev64(opp[i]), Rays());
    }
}

extern "C" void fb_mobility_both(const unsigned long long *black, const unsigned long long *white, int *mb, int *mw, long n)
{
    for (long i = 0; i < n; i++) obf::mobility_both(black[i], white[i], mb[i], mw[i]);
}

extern "C" void fb_mobility(const unsigned long long *own, const unsigned long long *opp, int *out, long n)
{
    for (long i = 0; i < n; i++) out[i] = obf::mobility(own[i], opp[i]);
}

extern "C" void fb_child_mobility(const unsigned long long *own, const unsigned long long *opp, const unsigned char *sq,
                                  int *out, long n)
{
    for (long i = 0; i < n; i++) {
        const unsigned long long x = 1ull << sq[i];
        const unsigned long long f = ((own[i] | opp[i]) & x) ? 0ull
                 : obf::flips_for(sq[i], own[i], opp[i], obf::rev64(own[i]), obf::rev64(opp[i]), Rays());
        out[i] = f ? obf::child_mobility(obf::make_pos4(own[i], opp[i]), f | x) : -1;
    }
}

// put() by four line look-ups (what the game kernels run)
extern "C" void fb_flips_lut(const unsigned long long *own, const unsigned long long *opp, const unsigned char *sq,
                             unsigned long long *out, long n)
{
    for (long i = 0; i < n; i++) {
        const unsigned long long x = 1ull << sq[i];
        out[i] = ((own[i] | opp[i]) & x) ? 0ull : obf::flips_lut(sq[i], own[i], opp[i], Rays(), 1u);
    }
}

// ... with the diagonal masks fetched by diagonal number (what the greedy kernel runs)
extern "C" void fb_flips_lut_line(const unsigned long long *own, const unsigned long long *opp, const unsigned char *sq,
                             unsigned long long *out, long n)
{
    for (long i = 0; i < n; i++) {
        const unsigned long long x = 1ull << sq[i];
        out[i] = ((own[i] | opp[i]) & x) ? 0ull : obf::flips_lut<true>(sq[i], own[i], opp[i], Rays(), 1u);
    }
}

// byte [value][k] of the k-th-set-bit table the playout kernel reads from shared memory
extern "C" int fb_kth_table(int value, int k)
{
    return (int)Rays().byte(obf::kKthBit64 * 8 + value * 8 + k);
}
