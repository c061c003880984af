// solve.cu -- exact endgame solver (othello_solve): perfect-play value and best move of a batch of positions.
//
// One lane solves one position with the search of endgame.cuh.  Solve times at the same number of empties differ
// by orders of magnitude, so the grid is persistent and a lane that finishes takes the next position from a counter
// in the caller's workspace (reset by the call itself): no warp waits for a statically assigned slow lane of
// another warp, only for the slowest of the positions its own lanes hold at the time.
#include "common.cuh"
#include "endgame.cuh"

using namespace ob;

static_assert(obe::kMaxEmpties == OTHELLO_SOLVE_MAX_EMPTIES && obe::kRefused == OTHELLO_SOLVE_REFUSED &&
              obe::kNoMove == OTHELLO_NO_MOVE && obe::kPass == OTHELLO_PASS, "endgame.cuh constants vs the C ABI");

namespace {

constexpr int kThreads = 128;
constexpr int64_t kWorkspaceBytes = 256;

__global__ void __launch_bounds__(kThreads) endgame_kernel(const u64 *__restrict__ black, const u64 *__restrict__ white,
                                                           const uint8_t *__restrict__ turn, int32_t *__restrict__ value,
                                                           uint8_t *__restrict__ move, unsigned long long *__restrict__ nodes,
                                                           int64_t n, unsigned long long *next)
{
    __shared__ u64 ray_s[obf::kRayBasic64];
    fill_rays(ray_s);
    __syncthreads();
    const Rays rays = {ray_s};
    // The stack of the upper levels: per lane, indexed by a run-time depth, so it lives in local memory (L1-cached).
    // It is touched once per node above the register-resident levels, where most nodes are not.
    obe::Frame st[obe::kFrames];
    for (;;) {
        const unsigned long long i = atomicAdd(next, 1ull);
        if (i >= (unsigned long long)n) break;
        const bool black_moves = turn ? turn[i] == OTHELLO_BLACK : true;
        const u64 b = black[i], w = white[i];
        int mv;
        u64 cnt;
        const int v = obe::solve(black_moves ? b : w, black_moves ? w : b, rays, mv, cnt, st);
        value[i] = v;
        move[i] = (uint8_t)mv;
        if (nodes) nodes[i] = cnt;
    }
}

}  // namespace

extern "C" int64_t othello_solve_workspace_bytes(void) { return kWorkspaceBytes; }

extern "C" int othello_solve(const uint64_t *black, const uint64_t *white, const uint8_t *turn, int32_t *value,
                             uint8_t *move, uint64_t *nodes, int64_t n, void *workspace, int64_t workspace_bytes,
                             void *stream)
{
    OB_CHECK_ARGS(n >= 0);
    if (n == 0) return 0;
    OB_CHECK_ARGS(black && white && value && move && workspace);
    if (workspace_bytes < kWorkspaceBytes) return OTHELLO_E_WORKSPACE;
    cudaStream_t s = (cudaStream_t)stream;
    unsigned long long *next = (unsigned long long *)workspace;
    OB_CUDA(cudaMemsetAsync(next, 0, sizeof *next, s));
    unsigned blocks;
    if (const int e = ob_persistent_blocks(endgame_kernel, kThreads, n, blocks)) return e;
    endgame_kernel<<<blocks, kThreads, 0, s>>>((const u64 *)black, (const u64 *)white, turn, value, move,
                                               (unsigned long long *)nodes, n, next);
    return ob_launch_status();
}
