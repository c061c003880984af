// tests/legal4_host.cpp -- TEST SCAFFOLDING: compiles subproc_b200/csrc/fastboard.cuh for the host so that the
// rank-sliced move generator of four boards (obf::legal_moves4) can be compared with the oracle without a GPU.
#include "../subproc_b200/csrc/fastboard.cuh"

// n a multiple of 4: the positions 4i .. 4i + 3 are one call, position 4i + q in byte slot (q - rot) & 3
extern "C" void fb_legal4(const unsigned long long *own, const unsigned long long *opp, unsigned long long *out, long n,
                          int rot)
{
    for (long i = 0; i < n; i += 4) {
        unsigned long long o[4], p[4], l[4];
        for (int j = 0; j < 4; j++) {
            o[j] = own[i + ((j + rot) & 3)];
            p[j] = opp[i + ((j + rot) & 3)];
        }
        obf::legal_moves4(o, p, l);
        for (int j = 0; j < 4; j++) out[i + ((j + rot) & 3)] = l[j];
    }
}

extern "C" void fb_legal(const unsigned long long *own, const unsigned long long *opp, unsigned long long *out, long n)
{
    for (long i = 0; i < n; i++) out[i] = obf::legal_moves(own[i], opp[i]);
}

// the 4x4 byte transpose in and out of the layout: out = from_sliced(to_sliced(v))
extern "C" void fb_sliced_round_trip(const unsigned long long *v, unsigned long long *out, unsigned *words, long n)
{
    for (long i = 0; i < n; i += 4) {
        unsigned s[8];
        obf::to_sliced(v + i, s);
        for (int r = 0; r < 8; r++) words[2 * i + r] = s[r];
        obf::from_sliced(s, out + i);
    }
}
