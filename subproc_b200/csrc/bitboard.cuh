// bitboard.cuh -- what every kernel shares besides the rules primitives of fastboard.cuh and the linear
// evaluation of eval.cuh: the counter-based RNG, counts(), and the shared-memory ray table that put() needs.
//
// The rules themselves -- the replacement of the reference's list-of-lists ray walks
// (board.py:124-174: hands_for_direc, is_puttable_at, put) -- are obf::legal_moves / obf::flips_for.
// Bit s = x + 8*y (board.py:79): +1 = one file to the right, +8 = one rank down the board.
#pragma once
#include <stdint.h>
#include "fastboard.cuh"
#include "eval.cuh"

namespace ob {

// ---- counter-based RNG (DESIGN.md "RNG"; oracle restatement: orc_rng_*) ----------------------
__device__ __forceinline__ u32 fmix32(u32 h)
{
    h ^= h >> 16; h *= 0x85EBCA6Bu; h ^= h >> 13; h *= 0xC2B2AE35u; h ^= h >> 16;
    return h;
}
__device__ __forceinline__ u32 rng_key(u64 seed, u64 gid)
{
    u32 h = fmix32((u32)seed ^ 0x9E3779B9u);
    h = fmix32(h ^ (u32)(seed >> 32));
    h = fmix32(h ^ (u32)gid);
    h = fmix32(h ^ (u32)(gid >> 32));
    return h;
}
__device__ __forceinline__ u32 rng_draw(u32 key, u32 ply, u32 stream)
{
    return fmix32(key + ply * 0x9E3779B9u + stream * 0x632BE5ABu);
}
__device__ __forceinline__ u32 rng_below(u32 r, u32 n) { return __umulhi(r, n); }

// rng_draw with its three right shifts issued as IMAD.HI (h >> k == umulhi(h, 2^(32-k))) on the FMA
// pipe; `one` is obf::kOpaqueOne so that ptxas cannot turn the multiplies back into ALU shifts
__device__ __forceinline__ u32 rng_draw_fma(u32 key, u32 ply, u32 stream, u32 one)
{
    const u32 c16 = one << 16, c19 = one << 19;
    u32 h = key + ply * 0x9E3779B9u + stream * 0x632BE5ABu;
    h ^= __umulhi(h, c16); h *= 0x85EBCA6Bu; h ^= __umulhi(h, c19); h *= 0xC2B2AE35u; h ^= __umulhi(h, c16);
    return h;
}

// ---- features --------------------------------------------------------------------------------
// counts(a_book, side) (parameter_progress_position_moves_learn.py:5-17) for side = `own`
__device__ __forceinline__ void features10(u64 own, u64 opp, int f[10])
{
    f[0] = __popcll(own | opp);
    f[1] = obf::mobility(own, opp);
#pragma unroll
    for (int k = 0; k < 8; k++) f[2 + k] = class_count(own, k);
}

// ray masks for obf::flips_for, [direction][square] so that lanes with different squares spread over
// the shared-memory banks (2 KB per CTA); filled once per CTA, then one __syncthreads()
struct Rays {
    const u64 *t;
    __device__ __forceinline__ u64 operator()(int d, int s) const { return t[d * 64 + s]; }
    __device__ __forceinline__ u64 word(u32 i) const { return t[i]; }
    __device__ __forceinline__ u32 byte(u32 i) const { return ((const uint8_t *)t)[i]; }
};

// the table is built at compile time and lives in global memory (L2-resident); a CTA copies its 2 KB
// into shared memory with two loads per thread instead of walking 256 rays
struct alignas(16) RayTableInit {
    u64 v[obf::kRayTable64];
    constexpr RayTableInit() : v()
    {
        for (int i = 0; i < obf::kRayTable64; i++) v[i] = obf::make_table_word(i);
    }
};
static __device__ const RayTableInit kRayTable = RayTableInit();

// N = obf::kRayBasic64: the ray masks of the carry-chain put() (2.5 KB); obf::kRayTable64: + the line look-up
// tables of the game kernels (12.2 KB)
template <int N = obf::kRayBasic64>
__device__ __forceinline__ void fill_rays(u64 *t)
{
    for (int i = threadIdx.x; i < N; i += blockDim.x) t[i] = kRayTable.v[i];
}

// The whole table for a game kernel, t 16-byte aligned, CTAs of at least MIN_THREADS threads: 16-byte loads, ALL of
// them issued before the first store.  A plain copy loop is one L2 round trip per 8 bytes and thread, twelve in a row
// for 11.9 KB and 128 threads: ncu's samples had the warps of the playout kernel spend 13 % of their life there.
template <int MIN_THREADS>
__device__ __forceinline__ void fill_tables(u64 *t)
{
    constexpr int kVec = obf::kRayTable64 / 2, kPer = (kVec + MIN_THREADS - 1) / MIN_THREADS;
    static_assert(obf::kRayTable64 % 2 == 0, "table size");
    const uint4 *src = reinterpret_cast<const uint4 *>(kRayTable.v);
    uint4 *dst = reinterpret_cast<uint4 *>(t);
    uint4 r[kPer];
#pragma unroll
    for (int j = 0; j < kPer; j++) {
        const int i = threadIdx.x + j * blockDim.x;
        if (i < kVec) r[j] = __ldg(src + i);
    }
#pragma unroll
    for (int j = 0; j < kPer; j++) {
        const int i = threadIdx.x + j * blockDim.x;
        if (i < kVec) dst[i] = r[j];
    }
}

// Board.put(piece, x, y) (board.py:161-174): flips of an own disc on EMPTY square s
__device__ __forceinline__ u64 put_flips(int s, u64 own, u64 opp, const Rays &rays)
{
    return obf::flips_for(s, own, opp, obf::rev64(own), obf::rev64(opp), rays);
}

}  // namespace ob
