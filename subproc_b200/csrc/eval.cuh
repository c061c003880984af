// eval.cuh -- the linear evaluation, host+device: the square classes, the phase rows and the dot product with which
// othello_eval, the greedy engine and the midgame search score a position.  One definition, so that all three agree
// bit for bit; tests/ compiles it with g++ through midgame.cuh.
#pragma once
#include <math.h>
#include <string.h>
#include "fastboard.cuh"

namespace ob {

typedef unsigned long long u64;
typedef unsigned int u32;

// square-class masks a..h (parameter_progress_position_moves_learn.py:9-16)
OBF_HD constexpr u64 class_mask(int k)
{
    return k == 0 ? 0x8100000000000081ull : k == 1 ? 0x4281000000008142ull : k == 2 ? 0x0042000000004200ull
         : k == 3 ? 0x2400810000810024ull : k == 4 ? 0x1800008181000018ull : k == 5 ? 0x003C424242423C00ull
         : k == 6 ? 0x0000240000240000ull : 0x0000183C3C180000ull;
}

// Board.mask_count(side, class k) (board.py:74-81) for the eight classes.  Every class mask is mirror symmetric and its
// low and high words occupy different bit positions, so the two halves of the board can be merged before counting:
// one POPC instead of two and no add.
OBF_HD int class_count(u64 bb, int k)
{
    const u32 m = ((u32)bb & (u32)class_mask(k)) | ((u32)(bb >> 32) & (u32)(class_mask(k) >> 32));
#if defined(__CUDA_ARCH__)
    return __popc(m);
#else
    return __builtin_popcount(m);
#endif
}
static_assert(((class_mask(0) >> 32) & class_mask(0) & 0xffffffffull) == 0 && ((class_mask(1) >> 32) & class_mask(1) & 0xffffffffull) == 0 &&
              ((class_mask(2) >> 32) & class_mask(2) & 0xffffffffull) == 0 && ((class_mask(3) >> 32) & class_mask(3) & 0xffffffffull) == 0 &&
              ((class_mask(4) >> 32) & class_mask(4) & 0xffffffffull) == 0 && ((class_mask(5) >> 32) & class_mask(5) & 0xffffffffull) == 0 &&
              ((class_mask(6) >> 32) & class_mask(6) & 0xffffffffull) == 0 && ((class_mask(7) >> 32) & class_mask(7) & 0xffffffffull) == 0,
              "class masks: low and high words must not share bit positions");

// phase row of a disc count: shards (0,16),(17,32),(33,48),(49,64) inclusive
// (progress_position_moves_learn.py:75,112-113)
OBF_HD int phase_row(int discs)
{
    int r = (discs + 15) >> 4;
    r -= 1;
    return r < 0 ? 0 : (r > 3 ? 3 : r);
}

// row . (mobility, a..h) + row[9] of colour `own`, where row = w + 10 * phase_row(discs): the intercept first, then
// fmaf in this order.  The greedy kernel passes the row itself: the children of one position all have its disc count
// + 1.
OBF_HD float eval_row(u64 own, u64 opp, const float *__restrict__ row)
{
    float acc = row[9];
    acc = fmaf(row[0], (float)obf::mobility(own, opp), acc);
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int k = 0; k < 8; k++) acc = fmaf(row[1 + k], (float)class_count(own, k), acc);
    return acc;
}

// w[phase] . (mobility, a..h) + w[phase][9] of colour `own`; w = [4][10] floats (shared or global)
OBF_HD float eval_linear(u64 own, u64 opp, const float *__restrict__ w)
{
    return eval_row(own, opp, w + 10 * phase_row(obf::popc64(own | opp)));
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

}  // namespace ob
