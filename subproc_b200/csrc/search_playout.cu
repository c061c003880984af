// search_playout.cu -- self-play with the midgame search (OTHELLO_POLICY_SEARCH): GameRunner.play_a_game where the engine
// behind a colour answers 'go' with the move othello_search returns for the position, at that colour's depth, on that
// colour's table.
//
// One lane plays one whole game: the greedy kernel's per-lane logic (trajectory row, game-over test, random plies and
// go_for's substitution with the same draws), with obm::search_root in place of the arg-max over the children.  A
// position costs between a few and 10^5 nodes, so the lanes of a warp finish their games at very different times; the
// grid is persistent, as in search.cu, and a lane whose game ends takes the next game index from a counter in the
// caller's workspace (reset by the call itself).  Both colours' weight tables and the ray masks of put() are staged in
// shared memory.  A greedy side is a search side of depth 1, a random side one of depth 0.
//
// Nothing here depends on which lane plays a game or when: a game's moves depend only on (seed, gid0 + g), the
// arguments and the game's own positions, and the launch totals are integer sums.
#include "playout_common.cuh"
#include "midgame.cuh"

using namespace ob;

namespace {

constexpr int kThreads = 128;
constexpr int kWeights = OTHELLO_PHASES * OTHELLO_WEIGHTS;
static_assert(2 * kWeights <= kThreads, "weight tables");

__device__ __forceinline__ unsigned long long warp_sum(unsigned long long v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Left alone, ptxas gives the kernel 160 registers (3 CTAs per SM); 4 CTAs per SM caps it at 128 without spills.
#if !defined(OB_SEARCH_PLAYOUT_CTAS)
#define OB_SEARCH_PLAYOUT_CTAS 4
#endif

// depth_b / depth_w: 0 = the random engine, 1 = greedy, 2.. = search
__global__ void __launch_bounds__(kThreads, OB_SEARCH_PLAYOUT_CTAS)
search_playout_kernel(const othello_playout_args a, int depth_b, int depth_w, unsigned long long *next)
{
    __shared__ u64 ray_s[obf::kRayBasic64];
    __shared__ float w_s[2 * kWeights];                       // Black's table, then White's
    fill_rays(ray_s);
    if (threadIdx.x < 2 * kWeights) {
        const float *src = threadIdx.x < kWeights ? (a.weights ? a.weights : a.weights_white)
                                                  : (a.weights_white ? a.weights_white : a.weights);
        // (a random side may come without a table: its row is never read)
        w_s[threadIdx.x] = src ? src[threadIdx.x % kWeights] : 0.0f;
    }
    __syncthreads();
    const Rays rays = {ray_s};
    // the root's move order and the stack of the upper levels of the search, in local memory (see search.cu)
    obm::Frame st[obm::kFrames];
    const bool traj = a.traj_black != nullptr;
    const int t_max = a.t_max;
    const int64_t stride = a.stride;
    // this lane's share of the launch totals, reduced over the warp once at exit
    unsigned long long plies_sum = 0, diff_sum = 0, black_wins = 0, white_wins = 0;
    for (;;) {
        const unsigned long long i = atomicAdd(next, 1ull);
        if (i >= (unsigned long long)a.n_games) break;
        const int64_t g = (int64_t)i;
        const u64 b0 = a.black0 ? a.black0[g] : OTHELLO_START_BLACK;
        const u64 w0 = a.white0 ? a.white0[g] : OTHELLO_START_WHITE;
        bool black_moves = a.turn0 ? (a.turn0[g] == OTHELLO_BLACK) : true;
        u64 own = black_moves ? b0 : w0, opp = black_moves ? w0 : b0;
        const u32 key = rng_key(a.seed, a.gid0 + (u64)g);
        // n_rand_rest = min(n_rand_hands, N_RAND_HAND_UNTIL = 10) (game_runner.py:6,118-119)
        int rest_b = min(a.n_rand_black, 10), rest_w = min(a.n_rand_white, 10);
        for (int t = 0;; t++) {
            if (traj && t <= t_max) {
                __stcs((u64 *)a.traj_black + (int64_t)t * stride + g, black_moves ? own : opp);
                __stcs((u64 *)a.traj_white + (int64_t)t * stride + g, black_moves ? opp : own);
            }
            const u64 legal = obf::legal_moves(own, opp);
            // is_game_over (board.py:57-58); a full board needs no second move generation
            if (legal == 0 && (~(own | opp) == 0 || obf::legal_moves(opp, own) == 0)) {
                const u64 fb = black_moves ? own : opp, fw = black_moves ? opp : own;
                const int n_black = __popcll(fb), n_white = __popcll(fw);
                a.nplies[g] = t;
                a.final_black[g] = fb;
                a.final_white[g] = fw;
                if (a.summary) a.summary[g] = obp::game_summary(t, n_black, n_white);
                plies_sum += (unsigned long long)t;
                diff_sum += (unsigned long long)(long long)(n_black - n_white);
                black_wins += n_black > n_white;
                white_wins += n_white > n_black;
                break;
            }
            int move = OTHELLO_PASS;
            u64 f = 0, x = 0;
            if (legal) {
                const int n = __popcll(legal);
                const int depth = black_moves ? depth_b : depth_w;
                bool random_now = t < a.random_plies || depth == 0;
                if (obp::substitute_now(key, t, black_moves ? rest_b : rest_w)) {   // game_runner.py:134-150
                    random_now = true;
                    if (black_moves) rest_b--; else rest_w--;
                }
                if (random_now) {
                    move = obf::kth_set_bit(legal, (int)rng_below(rng_draw(key, (u32)t, 1u), (u32)n));
                } else if (n == 1) {                                                // a forced move needs no search
                    move = __ffsll((long long)legal) - 1;
                } else {
                    u64 nodes;
                    obm::search_root(own, opp, depth, w_s + (black_moves ? 0 : kWeights), rays, move, nodes, st);
                    // no square (overlapping colours, NaN scores): the lowest legal one, never a ray-table index >= 64
                    if (move >= 64) move = __ffsll((long long)legal) - 1;
                }
                x = 1ull << move;
                f = obe::flips(move, own, opp, rays);
            }
            if (traj && t < t_max) __stcs(a.traj_move + (int64_t)t * stride + g, (uint8_t)move);
            const u64 moved = own | f | x;                    // put_s (board.py:203-208)
            own = opp & ~f;
            opp = moved;
            black_moves = !black_moves;
        }
    }
    // every lane of the warp gets here (the CTAs are whole warps): one atomic per value per warp
    if (a.totals == nullptr) return;
    plies_sum = warp_sum(plies_sum);
    diff_sum = warp_sum(diff_sum);
    black_wins = warp_sum(black_wins);
    white_wins = warp_sum(white_wins);
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(a.totals + 0, plies_sum);
        atomicAdd(a.totals + 1, diff_sum);
        atomicAdd(a.totals + 2, black_wins);
        atomicAdd(a.totals + 3, white_wins);
    }
}

}  // namespace

// othello_playout with a search side, its arguments already checked (playout.cu)
int ob_launch_search_playout(const othello_playout_args &a, int depth_b, int depth_w, cudaStream_t s)
{
    unsigned long long *next = (unsigned long long *)a.workspace;
    OB_CUDA(cudaMemsetAsync(next, 0, sizeof *next, s));
    unsigned blocks;
    if (const int e = ob_persistent_blocks(search_playout_kernel, kThreads, a.n_games, blocks)) return e;
    search_playout_kernel<<<blocks, kThreads, 0, s>>>(a, depth_b, depth_w, next);
    return ob_launch_status();
}
