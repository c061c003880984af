// search.cu -- midgame search (othello_search): depth-limited minimax value and best move of a batch of positions on
// the linear evaluation.
//
// One lane searches one position with the search of midgame.cuh.  Node counts at the same depth differ by an order of
// magnitude between positions, so the grid is persistent and a lane that finishes takes the next position from a
// counter in the caller's workspace (reset by the call itself), as in solve.cu.  The 160-byte weight table and the
// ray masks of put() are staged in shared memory.
#include "common.cuh"
#include "midgame.cuh"

using namespace ob;

static_assert(obm::kMaxDepth == OTHELLO_SEARCH_MAX_DEPTH && obm::kNoMove == OTHELLO_NO_MOVE &&
              obm::kPass == OTHELLO_PASS, "midgame.cuh constants vs the C ABI");

namespace {

constexpr int kThreads = 128;
constexpr int kWeights = OTHELLO_PHASES * OTHELLO_WEIGHTS;
constexpr int64_t kWorkspaceBytes = 256;
static_assert(kWeights == 40 && kWeights <= kThreads, "weight table");

__global__ void __launch_bounds__(kThreads) search_kernel(const u64 *__restrict__ black, const u64 *__restrict__ white,
                                                          const uint8_t *__restrict__ turn,
                                                          const float *__restrict__ weights, int depth,
                                                          float *__restrict__ value, uint8_t *__restrict__ move,
                                                          unsigned long long *__restrict__ nodes, int64_t n,
                                                          unsigned long long *next)
{
    __shared__ u64 ray_s[obf::kRayBasic64];
    __shared__ float w_s[kWeights];
    fill_rays(ray_s);
    if (threadIdx.x < kWeights) w_s[threadIdx.x] = weights[threadIdx.x];
    __syncthreads();
    const Rays rays = {ray_s};
    // The root's move order and the stack of the upper levels: per lane, indexed by a run-time level, so they live in
    // local memory (L1-cached).  A frame is touched once per node above the register-resident levels.
    obm::Frame st[obm::kFrames];
    for (;;) {
        const unsigned long long i = atomicAdd(next, 1ull);
        if (i >= (unsigned long long)n) break;
        const bool black_moves = turn ? turn[i] == OTHELLO_BLACK : true;
        const u64 b = black[i], w = white[i];
        int mv;
        u64 cnt;
        value[i] = obm::search_root(black_moves ? b : w, black_moves ? w : b, depth, w_s, rays, mv, cnt, st);
        move[i] = (uint8_t)mv;
        if (nodes) nodes[i] = cnt;
    }
}

}  // namespace

extern "C" int64_t othello_search_workspace_bytes(void) { return kWorkspaceBytes; }

extern "C" int othello_search(const uint64_t *black, const uint64_t *white, const uint8_t *turn, const float *weights,
                              int32_t depth, float *value, uint8_t *move, uint64_t *nodes, int64_t n, void *workspace,
                              int64_t workspace_bytes, void *stream)
{
    OB_CHECK_ARGS(n >= 0 && depth >= 1 && depth <= OTHELLO_SEARCH_MAX_DEPTH);
    if (n == 0) return 0;
    OB_CHECK_ARGS(black && white && weights && value && move && workspace);
    if (workspace_bytes < kWorkspaceBytes) return OTHELLO_E_WORKSPACE;
    cudaStream_t s = (cudaStream_t)stream;
    unsigned long long *next = (unsigned long long *)workspace;
    OB_CUDA(cudaMemsetAsync(next, 0, sizeof *next, s));
    unsigned blocks;
    if (const int e = ob_persistent_blocks(search_kernel, kThreads, n, blocks)) return e;
    search_kernel<<<blocks, kThreads, 0, s>>>((const u64 *)black, (const u64 *)white, turn, weights, depth, value, move,
                                              (unsigned long long *)nodes, n, next);
    return ob_launch_status();
}
