// playout.cu -- GameRunner.play_a_game (game_runner.py:165-201) for millions of games at once.
//
// One thread owns one game from the first ply to the last: the position lives in four 32-bit
// registers (own/opp bitboards), a ply is ~300 integer instructions (fastboard.cuh) and touches memory
// only to append the position and the move to the SoA trajectory [t][game] (a warp writes
// 32 consecutive u64 = 256 B per array per ply).  The warp runs in lock step; games that end
// early idle until the longest game of the warp is over.  A warp whose games all start from the
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

// the random engine (uniform over puttables()); the greedy engine lives in greedy.cu
struct Game {
    u64 own, opp;
    unsigned off;               // element index t * stride + game into the three trajectory arrays
    int t;
    bool passed;                // the previous ply was a pass
};

// One ply.  BLACK: 1 = Black moves, 0 = White moves (known at compile time when every game of the
// launch starts with the same colour: Black and White then alternate strictly, passes included),
// -1 = read `black_moves`.  Returns false when the game is over.
// TRAJ: 0 = no trajectory; 1 = trajectory with capacity checks; 2 = a trajectory that is known to fit, so the two
// checks per ply fall away: from the standard opening the first two plies are moves and a pass can only follow a move,
// so a game has at most 60 moves + 59 passes = 119 plies; with the pass that is taken back at the end of a game (below)
// the kernel writes position rows 0 .. plies + 1 <= 120 and move rows 0 .. plies <= 119, i.e. t_max >= 120 holds them.
// The three trajectory arrays are addressed with ONE 32-bit element index t * stride + game (a 32-bit add per
// ply instead of three 64-bit pointer increments), hence (t_max + 2) * stride < 2^32 (othello_playout checks).
template <int TRAJ, int BLACK>
__device__ __forceinline__ bool play_ply(Game &g, bool black_moves, u32 key, int t_max, int64_t stride, const Rays &rays,
                                         u64 *__restrict__ traj_black = nullptr, u64 *__restrict__ traj_white = nullptr,
                                         uint8_t *__restrict__ traj_move = nullptr)
{
    const bool bm = BLACK < 0 ? black_moves : (BLACK == 1);
    if (TRAJ == 2 || (TRAJ == 1 && g.t <= t_max)) {
        __stcs(traj_black + g.off, bm ? g.own : g.opp);
        __stcs(traj_white + g.off, bm ? g.opp : g.own);
    }
    const u64 legal = obf::legal_moves(g.own, g.opp);
    int move = OTHELLO_PASS;
    u64 f = 0, x = 0;
    if (legal == 0) {
        // is_game_over (board.py:57-58) needs the other colour's moves -- which the NEXT ply computes anyway, with the
        // whole warp instead of the few lanes that are here (that second move generation ran 6 % of the kernel's warp
        // instructions at 7 active lanes, profiles/playout_segments_r02.txt).  So the ply is played as a pass; if the
        // next one finds no move either, the game was over before the pass: it is taken back (rows past a game's
        // end are unspecified, and the rows up to it are what they would have been).
        if (g.passed) { g.t--; return false; }
        g.passed = true;
    } else {
        g.passed = false;
        const int n = __popcll(legal);
        const u32 r1 = rng_draw_fma(key, (u32)g.t, 1u, obf::kOpaqueOne);
        // go_for's substitution (game_runner.py:134-150) replaces the engine's move by a uniformly
        // random one; behind a random engine both draw the same k-th move from stream 1, so the
        // budgets n_rand_* do not change any game played by this kernel.
        move = obf::kth_set_bit<kKthLut>(legal, (int)rng_below(r1, (u32)n), rays);
        x = rays(obf::kRayDirs, move);
        f = obf::flips_lut(move, g.own, g.opp, rays, obf::kOpaqueOne);
    }
    if (TRAJ == 2 || (TRAJ == 1 && g.t < t_max)) __stcs(traj_move + g.off, (uint8_t)move);
    if (TRAJ) g.off += (unsigned)stride;
    // put_s: place, flip, nturn += 1, turn toggles (board.py:203-208)
    const u64 moved = g.own | f | x;
    g.own = g.opp & ~f;
    g.opp = moved;
    g.t++;
    return true;
}

// The first kBookDepth plies of a game from the standard opening with Black to move, walked down the opening book
// instead of played: the same draw as play_ply picks the same move (the k-th child is the k-th legal move), and the
// same rows are written.  No ply of the book is a pass, so the game goes on with Black to move (kBookDepth is even).
template <int TRAJ>
__device__ __forceinline__ void play_book(Game &g, u32 key, int t_max, int64_t stride, const BookNode *__restrict__ book,
                                          u64 *__restrict__ traj_black, u64 *__restrict__ traj_white,
                                          uint8_t *__restrict__ traj_move)
{
    const uint4 *node = reinterpret_cast<const uint4 *>(book);       // two 16-byte halves per node: position, links
    uint4 links = __ldg(node + 1);
    u64 black = OTHELLO_START_BLACK, white = OTHELLO_START_WHITE;
#pragma unroll
    for (int t = 0; t < kBookDepth; t++) {
        if (TRAJ == 2 || (TRAJ == 1 && t <= t_max)) {
            __stcs(traj_black + g.off, black);
            __stcs(traj_white + g.off, white);
        }
        const u32 r = rng_draw_fma(key, (u32)t, 1u, obf::kOpaqueOne);
        const u32 child = links.x + rng_below(r, links.y & 0xffu);
        links = __ldg(node + 2 * child + 1);
        const uint4 pos = __ldg(node + 2 * child);                   // (TRAJ == 0: only the last one is kept)
        black = obf::pack(pos.x, pos.y);
        white = obf::pack(pos.z, pos.w);
        if (TRAJ == 2 || (TRAJ == 1 && t < t_max)) __stcs(traj_move + g.off, (uint8_t)(links.y >> 8));
        if (TRAJ) g.off += (unsigned)stride;
    }
    g.own = black;
    g.opp = white;
    g.t = kBookDepth;
}

// UNIFORM: no per-game turn0 -- every game starts with Black, so the loop is unrolled over the two colours
template <int TRAJ, bool UNIFORM>
// (128 threads x >= 10 CTAs per SM measured best on B200: 64/128/256 threads and 9..12 CTAs are within 2 %)
#if !defined(OB_PLAYOUT_CTAS)
#define OB_PLAYOUT_CTAS 10
#endif
// book: the opening book on this device, or nullptr
__global__ void __launch_bounds__(kThreads, OB_PLAYOUT_CTAS) playout_kernel(const othello_playout_args a,
                                                                            const BookNode *__restrict__ book)
{
    __shared__ __align__(16) u64 ray_s[obf::kRayTable64];
    ob::fill_tables<kThreads>(ray_s);
    __syncthreads();
    const Rays rays = {ray_s};
    const int64_t gi = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    const bool live = gi < a.n_games;                  // lanes past the batch only take part in the totals
    const u64 b0 = live && a.black0 ? a.black0[gi] : OTHELLO_START_BLACK;
    const u64 w0 = live && a.white0 ? a.white0[gi] : OTHELLO_START_WHITE;
    bool black_moves = UNIFORM || !live ? true : (a.turn0[gi] == OTHELLO_BLACK);
    // the whole warp takes the book or none of it (lanes past the batch do not object)
    bool booked = book != nullptr;
    if (booked && (a.black0 || !UNIFORM))
        booked = __all_sync(0xffffffffu, b0 == OTHELLO_START_BLACK && w0 == OTHELLO_START_WHITE && black_moves);
    int plies = 0, n_black = 0, n_white = 0;
    if (live) {
        Game g;
        g.own = black_moves ? b0 : w0; g.opp = black_moves ? w0 : b0;
        g.t = 0;
        g.passed = false;
        g.off = (unsigned)gi;
        const u32 key = rng_key(a.seed, a.gid0 + (u64)gi);
        const int t_max = a.t_max;
        const int64_t stride = a.stride;
        if (booked) play_book<TRAJ>(g, key, t_max, stride, book, (u64 *)a.traj_black, (u64 *)a.traj_white, a.traj_move);

        if (UNIFORM) {
            for (;;) {
                if (!play_ply<TRAJ, 1>(g, true, key, t_max, stride, rays, (u64 *)a.traj_black, (u64 *)a.traj_white, a.traj_move)) { black_moves = true; break; }
                if (!play_ply<TRAJ, 0>(g, false, key, t_max, stride, rays, (u64 *)a.traj_black, (u64 *)a.traj_white, a.traj_move)) { black_moves = false; break; }
            }
        } else {
            while (play_ply<TRAJ, -1>(g, black_moves, key, t_max, stride, rays, (u64 *)a.traj_black, (u64 *)a.traj_white, a.traj_move)) black_moves = !black_moves;
        }
        const u64 fb = black_moves ? g.own : g.opp, fw = black_moves ? g.opp : g.own;
        a.nplies[gi] = g.t;
        a.final_black[gi] = fb;
        a.final_white[gi] = fw;
        plies = g.t; n_black = __popcll(fb); n_white = __popcll(fw);
        if (a.summary) a.summary[gi] = game_summary(plies, n_black, n_white);
    }
    __syncwarp();
    add_totals(a.totals, live, plies, n_black, n_white);
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
    const unsigned blocks = ob_blocks(a.n_games, kThreads);
    if (a.traj_black && (int64_t)(a.t_max + 2) * a.stride >= (1ll << 32)) return OTHELLO_E_INVALID;   // 32-bit trajectory index
    const BookNode *book = nullptr;                                          // (OB_PLAYOUT_BOOK_DEPTH=0: no book)
    if (kBookDepth > 0)
        if (const int rc = book_on_device(s, &book)) return rc;
    if (a.traj_black) {
        const bool fits = a.black0 == nullptr && a.t_max >= 120;             // every game from the standard opening fits
        if (a.turn0) {
            if (fits) playout_kernel<2, false><<<blocks, kThreads, 0, s>>>(a, book);
            else playout_kernel<1, false><<<blocks, kThreads, 0, s>>>(a, book);
        } else {
            if (fits) playout_kernel<2, true><<<blocks, kThreads, 0, s>>>(a, book);
            else playout_kernel<1, true><<<blocks, kThreads, 0, s>>>(a, book);
        }
    } else {
        if (a.turn0) playout_kernel<0, false><<<blocks, kThreads, 0, s>>>(a, book);
        else playout_kernel<0, true><<<blocks, kThreads, 0, s>>>(a, book);
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
