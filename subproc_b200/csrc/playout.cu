// playout.cu -- GameRunner.play_a_game (game_runner.py:165-201) for millions of games at once.
//
// One thread owns four games from the first ply to the last: each position lives in four 32-bit
// registers (own/opp bitboards), the four move generations of a ply are one pass over the ranks of the
// four boards (obf::legal_moves4), a game-ply is ~235 integer instructions (fastboard.cuh) and touches
// memory only to append the position and the move to the SoA trajectory [t][game] (a warp writes
// 32 consecutive u64 = 256 B per array per slot and ply).  The warp runs in lock step; games that end
// early idle until the longest of the warp's 128 games is over.  A warp whose games all start from the
// standard opening with Black to move takes its first OB_PLAYOUT_BOOK_DEPTH plies from the opening
// book (opening_book.cuh): per ply the loads of one 32-byte node of a 14.6 MB table; after that
// nothing is read from memory.
//
// The loop is the reference's: positions are recorded before every ply and once at the end
// (recorder.add, game_runner.py:170,159); the side to move asks go_for (game_runner.py:133-152),
// which may substitute a uniformly random move for the engine's, an engine with no move answers
// 'ps' and the pass is a ply of its own (board.py:194-195,203-208); the game stops when neither
// colour can move (board.py:57-58).
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <mutex>
#include <vector>
#include "playout_common.cuh"
#include "opening_book.cuh"

using namespace ob;
using namespace obp;
using obb::BookNode;
using obb::kBookDepth;

namespace {

// Table look-ups on the idle LSU pipe instead of ALU-pipe instructions (A/B on B200, profiles/playout_variants_r02.txt):
// put() as four line look-ups (obf::flips_lut, +15 % over eight carry-chain rays), the last three rounds of the
// k-th-set-bit search from the byte table (+2.3 %)
constexpr bool kKthLut = true;

// A thread plays kSlots games.  Their move generation is one call of obf::legal_moves4 (the rank-sliced layout: one
// pass over the ranks per direction for four boards instead of a Kogge-Stone flood per board); the rest of a ply --
// the draw, the k-th legal move, put() -- is per game, straight-line code whose effects are predicated on the game
// being live, so that ptxas interleaves the four independent chains.  Lane l, slot k of warp w plays game
// 128 w + 32 k + l: for each slot the 32 lanes store 32 consecutive games, as with one game per thread.
constexpr int kSlots = 4;
#if !defined(OB_PLAYOUT_THREADS)
#define OB_PLAYOUT_THREADS 64
#endif
constexpr int kPlayoutThreads = OB_PLAYOUT_THREADS;
constexpr int kGamesPerCta = kPlayoutThreads * kSlots;

// the random engine (uniform over puttables()); the greedy engine lives in greedy.cu
struct Game {
    u64 own, opp;
    int t;
    u32 key;
    bool live;                  // in the batch and not over
    bool passed;                // the previous ply was a pass
    bool black;                 // Black to move (read when the launch has per-game turns)
};

// One ply of every live game of the thread.  BLACK: 1 = Black moves, 0 = White moves (known at compile time when every
// game of the launch starts with the same colour: Black and White then alternate strictly, passes included, so the
// games of a thread are always at the same parity), -1 = read Game::black.  Returns whether a game of the thread is
// still live.
// TRAJ: 0 = no trajectory; 1 = trajectory with capacity checks; 2 = a trajectory that is known to fit, so the two
// checks per ply fall away: from the standard opening the first two plies are moves and a pass can only follow a move,
// so a game has at most 60 moves + 59 passes = 119 plies; with the pass that is taken back at the end of a game (below)
// the kernel writes position rows 0 .. plies + 1 <= 120 and move rows 0 .. plies <= 119, i.e. t_max >= 120 holds them.
// The three trajectory arrays are addressed with ONE 32-bit element index t * stride + game, computed from t (an IMAD
// instead of a register per game), hence (t_max + 2) * stride < 2^32 (othello_playout checks); game = g0 + 32 k.
template <int TRAJ, int BLACK>
__device__ __forceinline__ bool play_ply(Game (&g)[kSlots], unsigned g0, int t_max, unsigned stride, const Rays &rays,
                                         u64 *__restrict__ traj_black, u64 *__restrict__ traj_white,
                                         uint8_t *__restrict__ traj_move)
{
    u64 own[kSlots], opp[kSlots], legal[kSlots];
#pragma unroll
    for (int k = 0; k < kSlots; k++) {
        const bool bm = BLACK < 0 ? g[k].black : (BLACK == 1);
        const unsigned off = g0 + (unsigned)g[k].t * stride;
        if (g[k].live && (TRAJ == 2 || (TRAJ == 1 && g[k].t <= t_max))) {
            __stcs(traj_black + off + 32 * k, bm ? g[k].own : g[k].opp);
            __stcs(traj_white + off + 32 * k, bm ? g[k].opp : g[k].own);
        }
        own[k] = g[k].own;
        opp[k] = g[k].opp;
    }
    obf::legal_moves4(own, opp, legal);
    bool any = false;
#pragma unroll
    for (int k = 0; k < kSlots; k++) {
        Game &s = g[k];
        const bool moves = legal[k] != 0;
        // go_for's substitution (game_runner.py:134-150) replaces the engine's move by a uniformly
        // random one; behind a random engine both draw the same k-th move from stream 1, so the
        // budgets n_rand_* do not change any game played by this kernel.  (Without a move the draw
        // picks a square all the same, whose flips are dropped.)
        const u32 r1 = rng_draw_fma(s.key, (u32)s.t, 1u, obf::kOpaqueOne);
        int move = obf::kth_set_bit<kKthLut>(legal[k], (int)rng_below(r1, (u32)__popcll(legal[k])), rays);
        u64 x = rays(obf::kRayDirs, move);
        u64 f = obf::flips_lut(move, s.own, s.opp, rays, obf::kOpaqueOne);
        if (!moves) { move = OTHELLO_PASS; x = 0; f = 0; }
        // is_game_over (board.py:57-58) needs the other colour's moves -- which the NEXT ply computes anyway, with the
        // whole warp instead of the few lanes that are here (that second move generation ran 6 % of the kernel's warp
        // instructions at 7 active lanes, profiles/playout_segments_r02.txt).  So a ply without a move is played as a
        // pass; if the next one finds no move either, the game was over before the pass: it is taken back (rows past a
        // game's end are unspecified, and the rows up to it are what they would have been).
        const bool ends = s.live && !moves && s.passed;
        const bool plays = s.live && !ends;
        if (plays && (TRAJ == 2 || (TRAJ == 1 && s.t < t_max)))
            __stcs(traj_move + (g0 + (unsigned)s.t * stride) + 32 * k, (uint8_t)move);
        if (plays) {
            // put_s: place, flip, nturn += 1, turn toggles (board.py:203-208)
            const u64 moved = s.own | f | x;
            s.own = s.opp & ~f;
            s.opp = moved;
            s.passed = !moves;
            if (BLACK < 0) s.black = !s.black;
        }
        s.t += plays ? 1 : ends ? -1 : 0;
        s.live = plays;
        any |= plays;
    }
    return any;
}

// The first kBookDepth plies of the games from the standard opening with Black to move (book[k]: the whole warp agrees
// on slot k), walked down the opening book instead of played: the same draw as play_ply picks the same move (the k-th
// child is the k-th legal move), and the same rows are written.  No ply of the book is a pass, so the games go on with
// Black to move (kBookDepth is even).  The walks of the slots are independent chains of loads; a slot outside the book
// walks it as well and keeps nothing.
template <int TRAJ>
__device__ __forceinline__ void play_book(Game (&g)[kSlots], const bool (&booked)[kSlots], unsigned g0, int t_max, unsigned stride,
                                          const BookNode *__restrict__ book, u64 *__restrict__ traj_black,
                                          u64 *__restrict__ traj_white, uint8_t *__restrict__ traj_move)
{
    const uint4 *node = reinterpret_cast<const uint4 *>(book);       // two 16-byte halves per node: position, links
    const uint4 root = __ldg(node + 1);
    uint4 links[kSlots];
    u64 black[kSlots], white[kSlots];
    bool take[kSlots];
#pragma unroll
    for (int k = 0; k < kSlots; k++) {
        links[k] = root;
        black[k] = OTHELLO_START_BLACK;
        white[k] = OTHELLO_START_WHITE;
        take[k] = booked[k] && g[k].live;
    }
#pragma unroll
    for (int t = 0; t < kBookDepth; t++) {
        const unsigned off = g0 + (unsigned)t * stride;
#pragma unroll
        for (int k = 0; k < kSlots; k++) {
            if (take[k] && (TRAJ == 2 || (TRAJ == 1 && t <= t_max))) {
                __stcs(traj_black + off + 32 * k, black[k]);
                __stcs(traj_white + off + 32 * k, white[k]);
            }
            const u32 r = rng_draw_fma(g[k].key, (u32)t, 1u, obf::kOpaqueOne);
            const u32 child = links[k].x + rng_below(r, links[k].y & 0xffu);
            links[k] = __ldg(node + 2 * child + 1);
            const uint4 pos = __ldg(node + 2 * child);               // (TRAJ == 0: only the last one is kept)
            black[k] = obf::pack(pos.x, pos.y);
            white[k] = obf::pack(pos.z, pos.w);
            if (take[k] && (TRAJ == 2 || (TRAJ == 1 && t < t_max))) __stcs(traj_move + off + 32 * k, (uint8_t)(links[k].y >> 8));
        }
    }
#pragma unroll
    for (int k = 0; k < kSlots; k++) {
        if (take[k]) {
            g[k].own = black[k];
            g[k].opp = white[k];
            g[k].t = kBookDepth;
        }
    }
}

// per warp: the sums of plies and of n_black - n_white over its games and the number of Black and White wins, added
// to othello_playout_args.totals (every lane of the warp must arrive; one atomic per value per warp)
__device__ __forceinline__ void add_totals_sums(unsigned long long *totals, int plies, int diff, int black_wins,
                                                int white_wins)
{
    if (totals == nullptr) return;                     // uniform over the launch
    constexpr unsigned kAll = 0xffffffffu;
    const int p = __reduce_add_sync(kAll, plies);
    const int d = __reduce_add_sync(kAll, diff);
    const int bw = __reduce_add_sync(kAll, black_wins);
    const int ww = __reduce_add_sync(kAll, white_wins);
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(totals + 0, (unsigned long long)p);
        atomicAdd(totals + 1, (unsigned long long)(long long)d);
        atomicAdd(totals + 2, (unsigned long long)bw);
        atomicAdd(totals + 3, (unsigned long long)ww);
    }
}

// UNIFORM: no per-game turn0 -- every game starts with Black, so the loop is unrolled over the two colours
template <int TRAJ, bool UNIFORM>
#if !defined(OB_PLAYOUT_CTAS)
#define OB_PLAYOUT_CTAS 12
#endif
// book: the opening book on this device, or nullptr
__global__ void __launch_bounds__(kPlayoutThreads, OB_PLAYOUT_CTAS) playout_kernel(const othello_playout_args a,
                                                                                   const BookNode *__restrict__ book)
{
    __shared__ __align__(16) u64 ray_s[obf::kRayTable64];
    ob::fill_tables<kPlayoutThreads>(ray_s);
    __syncthreads();
    const Rays rays = {ray_s};
    const int lane = threadIdx.x & 31;
    const int64_t g0 = ((int64_t)blockIdx.x * kPlayoutThreads + (threadIdx.x - lane)) * kSlots + lane;
    Game g[kSlots];
    bool booked[kSlots];
#pragma unroll
    for (int k = 0; k < kSlots; k++) {
        const int64_t gi = g0 + 32 * k;
        const bool live = gi < a.n_games;              // slots past the batch only take part in the totals
        const u64 b0 = live && a.black0 ? a.black0[gi] : OTHELLO_START_BLACK;
        const u64 w0 = live && a.white0 ? a.white0[gi] : OTHELLO_START_WHITE;
        const bool bm = UNIFORM || !live ? true : (a.turn0[gi] == OTHELLO_BLACK);
        // the whole warp takes the book for slot k or none of it (slots past the batch do not object)
        booked[k] = book != nullptr;
        if (booked[k] && (a.black0 || !UNIFORM))
            booked[k] = __all_sync(0xffffffffu, b0 == OTHELLO_START_BLACK && w0 == OTHELLO_START_WHITE && bm);
        g[k].own = bm ? b0 : w0;
        g[k].opp = bm ? w0 : b0;
        g[k].t = 0;
        g[k].key = rng_key(a.seed, a.gid0 + (u64)gi);
        g[k].live = live;
        g[k].passed = false;
        g[k].black = bm;
    }
    const int t_max = a.t_max;
    const unsigned stride = (unsigned)a.stride, base = (unsigned)g0;
    u64 *const traj_black = (u64 *)a.traj_black, *const traj_white = (u64 *)a.traj_white;
    if (booked[0] || booked[1] || booked[2] || booked[3])
        play_book<TRAJ>(g, booked, base, t_max, stride, book, traj_black, traj_white, a.traj_move);

    if (UNIFORM) {
        while (play_ply<TRAJ, 1>(g, base, t_max, stride, rays, traj_black, traj_white, a.traj_move) &&
               play_ply<TRAJ, 0>(g, base, t_max, stride, rays, traj_black, traj_white, a.traj_move)) {}
    } else {
        while (play_ply<TRAJ, -1>(g, base, t_max, stride, rays, traj_black, traj_white, a.traj_move)) {}
    }
    int plies = 0, diff = 0, black_wins = 0, white_wins = 0;
#pragma unroll
    for (int k = 0; k < kSlots; k++) {
        const int64_t gi = g0 + 32 * k;
        if (gi < a.n_games) {
            // the colour to move when the game was found over: with uniform turns the parity of that ply (plies + 1)
            const bool bm = UNIFORM ? (g[k].t & 1) != 0 : g[k].black;
            const u64 fb = bm ? g[k].own : g[k].opp, fw = bm ? g[k].opp : g[k].own;
            a.nplies[gi] = g[k].t;
            a.final_black[gi] = fb;
            a.final_white[gi] = fw;
            const int n_black = __popcll(fb), n_white = __popcll(fw);
            if (a.summary) a.summary[gi] = game_summary(g[k].t, n_black, n_white);
            plies += g[k].t;
            diff += n_black - n_white;
            black_wins += n_black > n_white;
            white_wins += n_white > n_black;
        }
    }
    __syncwarp();
    add_totals_sums(a.totals, plies, diff, black_wins, white_wins);
}

// The opening book on the current device in *book: the tree is built on the host once per process and uploaded once
// per device, by the first launch that can use it, and kept until the process exits.  The upload is complete before
// any kernel is queued, so launches on every stream see the whole table.  *book stays nullptr while `s` is being
// captured into a graph, whose capture an upload would break: the kernel then plays those plies itself, with the same
// results.
int book_on_device(cudaStream_t s, const BookNode **book)
{
    *book = nullptr;
    cudaStreamCaptureStatus capture;
    OB_CUDA(cudaStreamIsCapturing(s, &capture));
    if (capture != cudaStreamCaptureStatusNone) return 0;
    constexpr int kMaxDevices = 64;
    static std::atomic<const BookNode *> on_device[kMaxDevices];
    static std::mutex upload;
    static std::vector<BookNode> tree;
    int dev;
    OB_CUDA(cudaGetDevice(&dev));
    if (dev >= kMaxDevices) return 0;
    if ((*book = on_device[dev].load(std::memory_order_acquire)) != nullptr) return 0;
    std::lock_guard<std::mutex> lock(upload);
    if ((*book = on_device[dev].load(std::memory_order_relaxed)) != nullptr) return 0;
    if (tree.empty() && !obb::build_book(kBookDepth, tree)) {
        fprintf(stderr, "othello_b200: a position of the opening book has no legal move\n");
        abort();
    }
    const size_t bytes = tree.size() * sizeof(BookNode);
    BookNode *d = nullptr;
    cudaStream_t copy = nullptr;
    cudaError_t e = cudaMalloc((void **)&d, bytes);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&copy, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d, tree.data(), bytes, cudaMemcpyHostToDevice, copy);
    if (e == cudaSuccess) e = cudaStreamSynchronize(copy);
    if (copy) cudaStreamDestroy(copy);
    if (e != cudaSuccess) {
        cudaFree(d);
        return (int)e;
    }
    on_device[dev].store(d, std::memory_order_release);
    *book = d;
    return 0;
}

int launch(const othello_playout_args &a, cudaStream_t s)
{
    const unsigned blocks = ob_blocks(a.n_games, kGamesPerCta);
    if (a.traj_black && (int64_t)(a.t_max + 2) * a.stride >= (1ll << 32)) return OTHELLO_E_INVALID;   // 32-bit trajectory index
    const BookNode *book = nullptr;                                          // (OB_PLAYOUT_BOOK_DEPTH=0: no book)
    if (kBookDepth > 0)
        if (const int rc = book_on_device(s, &book)) return rc;
    if (a.traj_black) {
        const bool fits = a.black0 == nullptr && a.t_max >= 120;             // every game from the standard opening fits
        if (a.turn0) {
            if (fits) playout_kernel<2, false><<<blocks, kPlayoutThreads, 0, s>>>(a, book);
            else playout_kernel<1, false><<<blocks, kPlayoutThreads, 0, s>>>(a, book);
        } else {
            if (fits) playout_kernel<2, true><<<blocks, kPlayoutThreads, 0, s>>>(a, book);
            else playout_kernel<1, true><<<blocks, kPlayoutThreads, 0, s>>>(a, book);
        }
    } else {
        if (a.turn0) playout_kernel<0, false><<<blocks, kPlayoutThreads, 0, s>>>(a, book);
        else playout_kernel<0, true><<<blocks, kPlayoutThreads, 0, s>>>(a, book);
    }
    return ob_launch_status();
}

}  // namespace

extern "C" int othello_playout(const othello_playout_args *args, void *stream)
{
    OB_CHECK_ARGS(args != nullptr);
    const othello_playout_args &a = *args;
    OB_CHECK_ARGS(a.n_games >= 0);
    if (a.n_games == 0) return 0;
    OB_CHECK_ARGS(a.nplies && a.final_black && a.final_white);
    OB_CHECK_ARGS((a.black0 == nullptr) == (a.white0 == nullptr));
    auto known = [](int p) { return p == OTHELLO_POLICY_RANDOM || p == OTHELLO_POLICY_GREEDY || p == OTHELLO_POLICY_SEARCH; };
    OB_CHECK_ARGS(known(a.policy));
    OB_CHECK_ARGS(a.policy_white == -1 || known(a.policy_white));
    const int policy_white = a.policy_white == -1 ? a.policy : a.policy_white;
    OB_CHECK_ARGS(a.policy == OTHELLO_POLICY_RANDOM || a.weights != nullptr);
    OB_CHECK_ARGS(policy_white == OTHELLO_POLICY_RANDOM || a.weights != nullptr || a.weights_white != nullptr);
    OB_CHECK_ARGS(a.n_rand_black >= 0 && a.n_rand_white >= 0 && a.random_plies >= 0);
    if (a.traj_black || a.traj_white || a.traj_move)       // (a capacity of 0 plies records only the start position)
        OB_CHECK_ARGS(a.traj_black && a.traj_white && (a.traj_move || a.t_max == 0) && a.t_max >= 0 && a.stride >= a.n_games);
    cudaStream_t s = (cudaStream_t)stream;
    if (a.policy == OTHELLO_POLICY_SEARCH || policy_white == OTHELLO_POLICY_SEARCH) {
        // the engine of each colour as a search depth: 0 = random, 1 = greedy
        const int depth_white = a.policy_white == -1 || a.search_depth_white == 0 ? a.search_depth : a.search_depth_white;
        auto depth_of = [](int policy, int depth) {
            return policy == OTHELLO_POLICY_SEARCH ? depth : policy == OTHELLO_POLICY_GREEDY ? 1 : 0;
        };
        const int depth_b = depth_of(a.policy, a.search_depth), depth_w = depth_of(policy_white, depth_white);
        OB_CHECK_ARGS(a.policy != OTHELLO_POLICY_SEARCH || (depth_b >= 1 && depth_b <= OTHELLO_SEARCH_MAX_DEPTH));
        OB_CHECK_ARGS(policy_white != OTHELLO_POLICY_SEARCH || (depth_w >= 1 && depth_w <= OTHELLO_SEARCH_MAX_DEPTH));
        if (a.workspace == nullptr || a.workspace_bytes < othello_search_workspace_bytes()) return OTHELLO_E_WORKSPACE;
        return ob_launch_search_playout(a, depth_b, depth_w, s);
    }
    const bool greedy = a.policy == OTHELLO_POLICY_GREEDY || policy_white == OTHELLO_POLICY_GREEDY;
    if (greedy) return ob_launch_greedy(a, s);
    return launch(a, s);
}
