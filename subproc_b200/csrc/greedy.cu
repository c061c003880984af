// greedy.cu -- greedy self-play (BASELINE config 4): GameRunner.play_a_game where the engine behind
// both players answers 'go' with the arg-max, over puttables(), of the linear evaluation of the
// successor position from the mover's side (ties -> lowest square).
//
// A lane owns a game, but the expensive part -- one flip + one move generation + one evaluation
// per CHILD, ~9.5 children per position, 1..33 per game -- is flattened over the warp: every ply
// the 32 games of a warp publish their positions and enumerate their (game, square) work items
// into shared memory; the warp then evaluates 32 items per round, whatever game they belong to,
// and reduces per game with two native 32-bit shared-memory atomics (ATOMS.MAX on the order-
// preserving bits of the score, ATOMS.MIN on the square among the lanes that hold the maximum).
// This keeps the lanes ~90 % busy; one-thread-per-game loops run at the pace of the warp's
// largest move list (~45 % busy).  Weight rows and ray masks are staged in shared memory.
//
// go_for's substitution rule (game_runner.py:133-152) and the `random_plies` opening are decided
// per lane exactly as in the oracle; such plies and forced moves (one legal move) skip evaluation.
#include "playout_common.cuh"

using namespace ob;
using namespace obp;

namespace {

constexpr int kWarps = kThreads / 32;
constexpr int kMaxItems = 32 * 60;            // 32 games x at most 60 empty squares: holds ANY pair of bitboards, not only
                                              // positions reachable from the opening (<= 33 legal moves)
constexpr unsigned kFull = 0xffffffffu;

struct WarpScratch {
    u64 own[32], opp[32];                     // positions of the 32 games (mover-relative)
    unsigned best_key[32];                    // arg-max state per game
    unsigned best_sq[32];
    unsigned row[32];                         // float offset of the children's weight row: colour table + 10 * phase
    unsigned short item[kMaxItems];           // (White to move << 15) | (game lane << 8) | square
};

template <bool SUBST, bool TRAJ>
#if !defined(OB_GREEDY_CTAS)
#define OB_GREEDY_CTAS 7
#endif
__global__ void __launch_bounds__(kThreads, OB_GREEDY_CTAS) greedy_kernel(const othello_playout_args a)
{
    constexpr int kW = OTHELLO_PHASES * OTHELLO_WEIGHTS;
    __shared__ float w_s[2 * kW];                             // Black's table, then White's
    __shared__ __align__(16) u64 ray_s[obf::kRayTable64];
    __shared__ WarpScratch scratch[kWarps];
    for (int i = threadIdx.x; i < 2 * kW; i += blockDim.x) {    // (a CTA is 2 or 4 warps, see ob_launch_greedy)
        const float *src = i < kW ? (a.weights ? a.weights : a.weights_white)
                                  : (a.weights_white ? a.weights_white : a.weights);
        w_s[i] = src[i % kW];
    }
    // which colours are served by the greedy engine (the other answers uniformly at random)
    const bool greedy_b = a.policy == OTHELLO_POLICY_GREEDY;
    const bool greedy_w = (a.policy_white == -1 ? a.policy : a.policy_white) == OTHELLO_POLICY_GREEDY;
    ob::fill_tables<kThreads / 2>(ray_s);                     // (a CTA is 2 or 4 warps)
    __syncthreads();
    const Rays rays = {ray_s};
    WarpScratch &ws = scratch[threadIdx.x >> 5];
    const int lane = threadIdx.x & 31;

    // a warp plays `gpw` games (one per lane, lanes >= gpw only help evaluating children): 32 for large
    // batches; fewer for small ones, so that a batch of 2^16 games still fills every SM with warps
    const int gpw = a.games_per_warp;
    const int64_t g = ((int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * gpw + lane;
    bool done = lane >= gpw || g >= a.n_games;                // lanes without a game only help evaluating
    const int64_t gi = done ? 0 : g;
    const u64 b0 = a.black0 ? a.black0[gi] : OTHELLO_START_BLACK;
    const u64 w0 = a.white0 ? a.white0[gi] : OTHELLO_START_WHITE;
    bool black_moves = a.turn0 ? (a.turn0[gi] == OTHELLO_BLACK) : true;
    u64 own = black_moves ? b0 : w0, opp = black_moves ? w0 : b0;
    const u32 key = rng_key(a.seed, a.gid0 + (u64)gi);
    // n_rand_rest = min(n_rand_hands, N_RAND_HAND_UNTIL = 10) (game_runner.py:6,118-119)
    int rest_b = SUBST ? min(a.n_rand_black, 10) : 0, rest_w = SUBST ? min(a.n_rand_white, 10) : 0;

    u64 *tb = TRAJ ? (u64 *)a.traj_black + gi : nullptr;
    u64 *tw = TRAJ ? (u64 *)a.traj_white + gi : nullptr;
    uint8_t *tm = TRAJ ? a.traj_move + gi : nullptr;
    const int t_max = a.t_max;
    const int64_t stride = a.stride;

    int t = 0;
    const bool live = !done;
    int plies = 0, n_black = 0, n_white = 0;               // the game's result, for the launch totals
    while (__any_sync(kFull, !done)) {
        u64 legal = 0;
        if (!done) {
            if (TRAJ && t <= t_max) {
                __stcs(tb, black_moves ? own : opp);
                __stcs(tw, black_moves ? opp : own);
                tb += stride; tw += stride;
            }
            legal = obf::legal_moves(own, opp);
            // is_game_over (board.py:57-58); a full board needs no second move generation
            if (legal == 0 && (~(own | opp) == 0 || obf::legal_moves(opp, own) == 0)) {
                done = true;
                const u64 fb = black_moves ? own : opp, fw = black_moves ? opp : own;
                a.nplies[g] = t;
                a.final_black[g] = fb;
                a.final_white[g] = fw;
                plies = t; n_black = __popcll(fb); n_white = __popcll(fw);
                if (a.summary) a.summary[g] = game_summary(plies, n_black, n_white);
            }
        }
        const bool moving = !done && legal != 0;              // otherwise: finished, or this ply is a pass
        const int n = __popcll(legal);
        bool random_now = t < a.random_plies || !(black_moves ? greedy_b : greedy_w);
        if (SUBST && moving) {
            if (substitute_now(key, t, black_moves ? rest_b : rest_w)) {           // game_runner.py:134-150
                random_now = true;
                if (black_moves) rest_b--; else rest_w--;
            }
        }
        const bool evaluate = moving && !random_now && n > 1;  // a forced move needs no evaluation
        // exclusive prefix of the children counts over the warp
        const int cnt = evaluate ? n : 0;
        int incl = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(kFull, incl, o);
            if (lane >= o) incl += v;
        }
        const int total = __shfl_sync(kFull, incl, 31);
        if (total > 0) {
            ws.own[lane] = own; ws.opp[lane] = opp;
            ws.best_key[lane] = 0u; ws.best_sq[lane] = 64u;
            ws.row[lane] = (black_moves ? 0 : kW) + 10 * phase_row(__popcll(own | opp) + 1);
            if (evaluate) {
                // one 32-bit half after the other: 9 instructions per square (lowest bit through POPC of the bits
                // below it) instead of the 21 of a 64-bit find-first-set + clear
                unsigned short *dst = ws.item + (incl - cnt);
                unsigned tag = (black_moves ? 0u : 0x8000u) | ((unsigned)lane << 8);
#pragma unroll
                for (int half = 0; half < 2; half++) {
                    for (u32 w = half ? obf::hi32(legal) : obf::lo32(legal); w;) {
                        const u32 below = w - 1u;
                        *dst++ = (unsigned short)(tag + (unsigned)__popc(~w & below));
                        w &= below;
                    }
                    tag += 32u;
                }
            }
            __syncwarp();
            for (int base = 0; base < total; base += 32) {
                const int j = base + lane;
                const bool have = j < total;
                unsigned owner = 0, sq = 0, kbits = 0, before = 0;
                if (have) {
                    const unsigned it = ws.item[j];
                    owner = (it >> 8) & 31u; sq = it & 63u;
                    const u64 o = ws.own[owner], p = ws.opp[owner];
                    
                    const u64 f = obf::flips_lut<true>((int)sq, o, p, rays, obf::kOpaqueOne);
                    kbits = ob::ordered_bits(ob::eval_row(o | f | (1ull << sq), p & ~f, w_s + ws.row[owner]));
                    before = ws.best_key[owner];
                }
                __syncwarp();
                if (have) atomicMax(&ws.best_key[owner], kbits);
                __syncwarp();
                // lanes that raised their game's maximum in this round restart its square, then the
                // lowest square among the lanes holding the maximum wins (items ascend with the square)
                const bool top = have && ws.best_key[owner] == kbits && kbits > before;
                if (top) ws.best_sq[owner] = 64u;
                __syncwarp();
                if (top) atomicMin(&ws.best_sq[owner], sq);
                __syncwarp();
            }
        }
        if (!done) {
            int move = OTHELLO_PASS;
            u64 f = 0, x = 0;
            if (moving) {
                if (evaluate) {
                    move = (int)ws.best_sq[lane];
                    if (move >= 64) move = __ffsll((long long)legal) - 1;      // every score NaN (NaN weights): lowest square
                }
                else if (random_now) move = obf::kth_set_bit(legal, (int)rng_below(rng_draw(key, (u32)t, 1u), (u32)n));
                else move = __ffsll((long long)legal) - 1;
                x = 1ull << move;
                f = obf::flips_lut<true>(move, own, opp, rays, obf::kOpaqueOne);
            }
            if (TRAJ && t < t_max) { __stcs(tm, (uint8_t)move); tm += stride; }
            const u64 moved = own | f | x;                    // put_s (board.py:203-208)
            own = opp & ~f;
            opp = moved;
            black_moves = !black_moves;
            t++;
        }
        __syncwarp();
    }
    add_totals(a.totals, live, plies, n_black, n_white);
}

}  // namespace

int ob_launch_greedy(const othello_playout_args &args, cudaStream_t s)
{
    othello_playout_args a = args;
    if (a.games_per_warp != 8 && a.games_per_warp != 16 && a.games_per_warp != 32) {
        a.games_per_warp = 32;
    }
    // Small batches (less than two waves of 6 CTAs x 148 SMs) run as CTAs of 2 warps instead of 4: twice as
    // many CTAs spread evenly over the SMs (2^16 games: 6.9 per SM instead of 3.5, i.e. 7 vs 4 on the fullest)
    const int threads = a.n_games < 2 * 6 * 148 * kThreads ? kThreads / 2 : kThreads;
    const unsigned blocks = ob_blocks(a.n_games, a.games_per_warp * (threads / 32));
    const bool subst = a.n_rand_black > 0 || a.n_rand_white > 0;
    if (a.traj_black) {
        if (subst) greedy_kernel<true, true><<<blocks, threads, 0, s>>>(a);
        else greedy_kernel<false, true><<<blocks, threads, 0, s>>>(a);
    } else {
        if (subst) greedy_kernel<true, false><<<blocks, threads, 0, s>>>(a);
        else greedy_kernel<false, false><<<blocks, threads, 0, s>>>(a);
    }
    return ob_launch_status();
}
