// playout_common.cuh -- pieces shared by the random (playout.cu) and greedy (greedy.cu) game kernels
#pragma once
#include "common.cuh"
#include "fastboard.cuh"

namespace obp {

using ob::u64;
using ob::u32;

constexpr int kThreads = 128;

using ob::Rays;
using ob::fill_rays;

// go_for's substitution test (game_runner.py:134-135): with budget `rest` left, play a random move
// with probability 1/rest (stream 0 of the counter-based RNG)
__device__ __forceinline__ bool substitute_now(u32 key, int t, int rest)
{
    return rest > 0 && ob::rng_below(ob::rng_draw(key, (u32)t, 0u), (u32)rest) == 0;
}

// othello_playout_args.summary: plies in the low byte, n_black - n_white (int8) in the high byte
__device__ __forceinline__ uint16_t game_summary(int plies, int n_black, int n_white)
{
    return (uint16_t)(min(plies, 255) | (((n_black - n_white) & 0xff) << 8));
}

// End of a game kernel: what play_a_game reports per game (game_runner.py:194-199), summed over the
// launch (othello_playout_args.totals).  Every lane of the warp must arrive (live = false for lanes
// past the batch); one atomic per value per warp.
__device__ __forceinline__ void add_totals(unsigned long long *totals, bool live, int plies, int n_black, int n_white)
{
    if (totals == nullptr) return;                     // uniform over the launch
    constexpr unsigned kAll = 0xffffffffu;
    const int p = __reduce_add_sync(kAll, live ? plies : 0);
    const int d = __reduce_add_sync(kAll, live ? n_black - n_white : 0);
    const int bw = __popc(__ballot_sync(kAll, live && n_black > n_white));
    const int ww = __popc(__ballot_sync(kAll, live && n_white > n_black));
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(totals + 0, (unsigned long long)p);
        atomicAdd(totals + 1, (unsigned long long)(long long)d);
        atomicAdd(totals + 2, (unsigned long long)bw);
        atomicAdd(totals + 3, (unsigned long long)ww);
    }
}

}  // namespace obp

// greedy.cu
int ob_launch_greedy(const othello_playout_args &a, cudaStream_t s);
// search_playout.cu: depth_b / depth_w = 0 for a random side, 1 for a greedy one
int ob_launch_search_playout(const othello_playout_args &a, int depth_b, int depth_w, cudaStream_t s);
