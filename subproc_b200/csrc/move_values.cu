// move_values.cu -- the value of every move of a batch of positions (othello_search_moves, othello_solve_moves).
//
// The work items are (position, slot) pairs, 65 per position: item k is slot k % 65 of position k / 65.  One lane
// computes one item with move_values.cuh and writes one entry of the [n][65] rows.  The grid is the persistent grid of
// search.cu / solve.cu: a lane that finishes takes the next item from a counter in the caller's workspace (reset by
// the call itself).  Most slots are not moves (a midgame position has about 10 of 65), so one item in six or so does
// a search: the lanes of a warp draw their items together, through one atomicAdd per group of converged lanes.
#include "common.cuh"
#include "move_values.cuh"

using namespace ob;

static_assert(obv::kSlots == OTHELLO_PASS + 1 && obe::kPass == OTHELLO_PASS && obe::kRefused == OTHELLO_SOLVE_REFUSED &&
              obe::kMaxEmpties == OTHELLO_SOLVE_MAX_EMPTIES && obm::kMaxDepth == OTHELLO_SEARCH_MAX_DEPTH,
              "move_values.cuh constants vs the C ABI");

namespace {

constexpr int kThreads = 128;
constexpr int kWeights = OTHELLO_PHASES * OTHELLO_WEIGHTS;
static_assert(kWeights <= kThreads, "weight table");

// The next item of this lane.  The lanes of the warp that arrive here together take consecutive items: their leader
// adds the group's size to the counter, and every lane's item is the old value plus its rank in the group.  One
// atomic per group instead of one per lane (with ~55 of 65 items empty, lanes come back for work at a high rate).
__device__ __forceinline__ unsigned long long claim(unsigned long long *next)
{
    const unsigned group = __activemask();
    const unsigned lane = threadIdx.x & 31;
    const int leader = __ffs(group) - 1;
    unsigned long long base = 0;
    if ((int)lane == leader) base = atomicAdd(next, (unsigned long long)__popc(group));
    base = __shfl_sync(group, base, leader);
    return base + (unsigned)__popc(group & ((1u << lane) - 1u));
}

__global__ void __launch_bounds__(kThreads) search_moves_kernel(const u64 *__restrict__ black,
                                                                const u64 *__restrict__ white,
                                                                const uint8_t *__restrict__ turn,
                                                                const float *__restrict__ weights, int depth,
                                                                float *__restrict__ values,
                                                                unsigned long long *__restrict__ nodes,
                                                                unsigned long long items, unsigned long long *next)
{
    __shared__ u64 ray_s[obf::kRayBasic64];
    __shared__ float w_s[kWeights];
    fill_rays(ray_s);
    if (threadIdx.x < kWeights) w_s[threadIdx.x] = weights[threadIdx.x];
    __syncthreads();
    const Rays rays = {ray_s};
    obm::Frame st[obm::kFrames];                       // local memory, as in search.cu (frame 0 is not used here)
    for (;;) {
        const unsigned long long k = claim(next);
        if (k >= items) break;
        const unsigned long long i = k / obv::kSlots;
        const int slot = (int)(k - i * obv::kSlots);
        const bool black_moves = turn ? turn[i] == OTHELLO_BLACK : true;
        const u64 b = black[i], w = white[i];
        u64 cnt;
        values[k] = obv::search_slot(black_moves ? b : w, black_moves ? w : b, slot, depth, w_s, rays, cnt, st);
        if (nodes) nodes[k] = cnt;
    }
}

__global__ void __launch_bounds__(kThreads) solve_moves_kernel(const u64 *__restrict__ black,
                                                               const u64 *__restrict__ white,
                                                               const uint8_t *__restrict__ turn,
                                                               int32_t *__restrict__ values,
                                                               unsigned long long *__restrict__ nodes,
                                                               unsigned long long items, unsigned long long *next)
{
    __shared__ u64 ray_s[obf::kRayBasic64];
    fill_rays(ray_s);
    __syncthreads();
    const Rays rays = {ray_s};
    obe::Frame st[obe::kFrames];                       // local memory, as in solve.cu
    for (;;) {
        const unsigned long long k = claim(next);
        if (k >= items) break;
        const unsigned long long i = k / obv::kSlots;
        const int slot = (int)(k - i * obv::kSlots);
        const bool black_moves = turn ? turn[i] == OTHELLO_BLACK : true;
        const u64 b = black[i], w = white[i];
        u64 cnt;
        values[k] = obv::solve_slot(black_moves ? b : w, black_moves ? w : b, slot, rays, cnt, st);
        if (nodes) nodes[k] = cnt;
    }
}

// the launch both entry points share once their arguments are checked
template <typename Kernel, typename... Args>
int launch(Kernel kernel, int64_t n, void *workspace, void *stream, Args... args)
{
    cudaStream_t s = (cudaStream_t)stream;
    unsigned long long *next = (unsigned long long *)workspace;
    OB_CUDA(cudaMemsetAsync(next, 0, sizeof *next, s));
    const int64_t items = n * obv::kSlots;
    unsigned blocks;
    if (const int e = ob_persistent_blocks(kernel, kThreads, items, blocks)) return e;
    kernel<<<blocks, kThreads, 0, s>>>(args..., (unsigned long long)items, next);
    return ob_launch_status();
}

}  // namespace

extern "C" int othello_search_moves(const uint64_t *black, const uint64_t *white, const uint8_t *turn,
                                    const float *weights, int32_t depth, float *values, uint64_t *nodes, int64_t n,
                                    void *workspace, int64_t workspace_bytes, void *stream)
{
    OB_CHECK_ARGS(n >= 0 && n <= INT64_MAX / obv::kSlots && depth >= 1 && depth <= OTHELLO_SEARCH_MAX_DEPTH);
    if (n == 0) return 0;
    OB_CHECK_ARGS(black && white && weights && values && workspace);
    if (workspace_bytes < othello_search_workspace_bytes()) return OTHELLO_E_WORKSPACE;
    return launch(search_moves_kernel, n, workspace, stream, (const u64 *)black, (const u64 *)white, turn, weights,
                  (int)depth, values, (unsigned long long *)nodes);
}

extern "C" int othello_solve_moves(const uint64_t *black, const uint64_t *white, const uint8_t *turn, int32_t *values,
                                   uint64_t *nodes, int64_t n, void *workspace, int64_t workspace_bytes, void *stream)
{
    OB_CHECK_ARGS(n >= 0 && n <= INT64_MAX / obv::kSlots);
    if (n == 0) return 0;
    OB_CHECK_ARGS(black && white && values && workspace);
    if (workspace_bytes < othello_solve_workspace_bytes()) return OTHELLO_E_WORKSPACE;
    return launch(solve_moves_kernel, n, workspace, stream, (const u64 *)black, (const u64 *)white, turn, values,
                  (unsigned long long *)nodes);
}
