// host_api.cu -- the host-buffer front end of the C ABI: what a caller without torch (the
// ctypes / cgo style binding of INTEGRATION.md) uses.  A context owns its streams and grow-only
// device workspaces; every call copies its inputs in, launches the same kernels as the
// device-pointer entry points and copies results out.
//
// Playouts are the throughput path, so they exist in an asynchronous form
// (othello_playout_host_async -> ticket, othello_ctx_wait): the context keeps kSlots independent
// workspaces and a batch is cut into chunks whose copy-in, kernel and copy-out rotate over
// kPipeStreams streams.  Nothing in that pipeline waits for the host, so the copy-in of batch i+1
// and the copy-out of batch i-1 run under the kernels of batch i: in steady state a caller that
// keeps two batches in flight sees the kernel time, not kernel + PCIe.
#include <new>
#include "common.cuh"
#include "fastboard.cuh"

constexpr int kPipeStreams = 3;     // chunks of a playout rotate over these streams
constexpr int kSlots = 2;           // batches that may be in flight at once
constexpr int kMaxChunks = 8;       // default; OTHELLO_OPT_MAX_CHUNKS changes it per context
constexpr int64_t kMinChunk = 65536;

struct othello_slot {
    char *ws;
    size_t ws_bytes;
    cudaStream_t ctl;               // prologue (weights, totals reset) and epilogue (join, totals copy-out) of the
                                    // slot's batches: its own stream, so that the prologue of batch i+1 does
                                    // not queue behind the epilogue of batch i
    cudaEvent_t ready, tail[3];     // prologue done / last operation of the batch on each pipe stream
    cudaEvent_t done;               // recorded on ctl after the last copy-out of the batch
    bool pending;                   // issued, not yet waited for
    int64_t ticket;
    // trajectory of the batch (views into ws)
    uint64_t *traj_black, *traj_white;
    uint8_t *traj_move;
    int64_t traj_stride;
    int32_t traj_t_max;
    unsigned long long *d_totals;   // [4] device, inside ws
};

struct othello_ctx {
    int device;
    cudaStream_t stream;            // the synchronous small-batch calls
    cudaStream_t pipe[kPipeStreams];
    othello_slot slot[kSlots];
    int64_t next_ticket;
    int64_t chunk_seq;              // rotates the pipe streams across calls
    int last_slot;                  // slot of the most recently issued playout, -1 = none
    int max_chunks;
    // single-position front end (othello_board_apply_host): results land in pinned host memory that
    // the kernel writes directly (mapped), so a call is one launch + one stream synchronise
    othello_position_info *info_h, *info_d;
};

namespace {

size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

// drain everything the context has in flight (error paths, workspace growth, destroy)
void drain(othello_ctx *c)
{
    for (int i = 0; i < kPipeStreams; i++)
        if (c->pipe[i]) cudaStreamSynchronize(c->pipe[i]);
    for (int i = 0; i < kSlots; i++) {
        if (c->slot[i].ctl) cudaStreamSynchronize(c->slot[i].ctl);
        c->slot[i].pending = false;
    }
    if (c->stream) cudaStreamSynchronize(c->stream);
}

int reserve(othello_ctx *c, othello_slot *sl, size_t bytes)
{
    if (bytes <= sl->ws_bytes) return 0;
    drain(c);                                   // nothing may still read or write the old block
    if (sl->ws) { cudaError_t e = cudaFree(sl->ws); sl->ws = nullptr; sl->ws_bytes = 0; if (e != cudaSuccess) return (int)e; }
    sl->traj_black = sl->traj_white = nullptr; sl->traj_move = nullptr; sl->d_totals = nullptr;
    OB_CUDA(cudaMalloc((void **)&sl->ws, bytes));
    sl->ws_bytes = bytes;
    return 0;
}

// the synchronous small-batch calls run on slot 0 and ctx->stream: wait until the slot is idle
int idle_slot0(othello_ctx *c)
{
    othello_slot *sl = &c->slot[0];
    if (sl->pending) { OB_CUDA(cudaEventSynchronize(sl->done)); sl->pending = false; }
    return 0;
}

// bump allocator over a workspace
struct Carver {
    char *base; size_t off;
    template <typename T> T *take(size_t count) { T *p = (T *)(base + off); off += align256(count * sizeof(T)); return p; }
};

// after a failure in the middle of a call: make sure no copy into caller memory is still running
int fail(othello_ctx *c, int rc) { drain(c); return rc; }
#define OBH_TRY(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return fail(c, (int)e_); } while (0)

// Board.put(piece, x, y) (board.py:161-174) on ONE position, then everything the reference's callers ask
// about the resulting position before the next move (game_runner.py:137,162,194-196; game_recorder.py:112;
// counts(), parameter_progress_position_moves_learn.py:5-17): legal moves and features of both colours,
// disc counts.  One warp; lane 0 does the rules, the result goes straight to mapped host memory.
__global__ void __launch_bounds__(32) board_kernel(ob::u64 black, ob::u64 white, int color, int move,
                                                   othello_position_info *out)
{
    __shared__ ob::u64 ray_s[obf::kRayBasic64];
    ob::fill_rays(ray_s);
    __syncwarp();
    if (threadIdx.x != 0) return;
    const ob::Rays rays = {ray_s};
    ob::u64 flips = 0;
    if (move >= 0 && move < 64) {
        const ob::u64 x = 1ull << move;
        const bool is_black = color == OTHELLO_BLACK;          // hostile(piece) is Black for anything but Black (board.py:155-159)
        const ob::u64 own = is_black ? black : white, opp = is_black ? white : black;
        if (!((black | white) & x)) flips = ob::put_flips(move, own, opp, rays);
        if (flips) {
            const ob::u64 no = own | flips | x, np = opp & ~flips;
            black = is_black ? no : np; white = is_black ? np : no;
        }
    }
    out->black = black; out->white = white; out->flips = flips;
    out->ret = __popcll(flips);
    out->legal_black = obf::legal_moves(black, white);
    out->legal_white = obf::legal_moves(white, black);
    out->n_black = __popcll(black); out->n_white = __popcll(white); out->n_empty = 64 - __popcll(black | white);
    int fb[10], fw[10];
    ob::features10(black, white, fb);
    ob::features10(white, black, fw);
    for (int k = 0; k < 10; k++) { out->features_black[k] = fb[k]; out->features_white[k] = fw[k]; }
    __threadfence_system();
}

}  // namespace

extern "C" {

int othello_abi_version(void) { return OTHELLO_ABI_VERSION; }

const char *othello_error_string(int code)
{
    switch (code) {
    case 0: return "ok";
    case OTHELLO_E_INVALID: return "invalid argument";
    case OTHELLO_E_WORKSPACE: return "workspace too small";
    case OTHELLO_E_NO_DEVICE: return "no CUDA device";
    default: return code > 0 ? cudaGetErrorString((cudaError_t)code) : "unknown error";
    }
}

void othello_ctx_destroy(othello_ctx *c)
{
    if (!c) return;
    cudaSetDevice(c->device);
    drain(c);
    for (int i = 0; i < kSlots; i++) {
        othello_slot *sl = &c->slot[i];
        if (sl->ws) cudaFree(sl->ws);
        if (sl->done) cudaEventDestroy(sl->done);
        if (sl->ready) cudaEventDestroy(sl->ready);
        for (int j = 0; j < kPipeStreams; j++)
            if (sl->tail[j]) cudaEventDestroy(sl->tail[j]);
        if (sl->ctl) cudaStreamDestroy(sl->ctl);
    }
    for (int i = 0; i < kPipeStreams; i++)
        if (c->pipe[i]) cudaStreamDestroy(c->pipe[i]);
    if (c->stream) cudaStreamDestroy(c->stream);
    if (c->info_h) cudaFreeHost(c->info_h);
    delete c;
}

int othello_ctx_create(int device, othello_ctx **out)
{
    OB_CHECK_ARGS(out != nullptr);
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) return OTHELLO_E_NO_DEVICE;
    OB_CHECK_ARGS(device >= 0 && device < count);
    OB_CUDA(cudaSetDevice(device));
    othello_ctx *c = new (std::nothrow) othello_ctx();      // value-initialised: every handle starts null
    if (!c) return OTHELLO_E_INVALID;
    c->device = device; c->next_ticket = 1; c->chunk_seq = 0; c->last_slot = -1; c->max_chunks = kMaxChunks;
    static_assert(kPipeStreams == 3, "othello_slot::tail has kPipeStreams entries");
    cudaError_t e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    for (int i = 0; i < kPipeStreams && e == cudaSuccess; i++)
        e = cudaStreamCreateWithFlags(&c->pipe[i], cudaStreamNonBlocking);
    for (int i = 0; i < kSlots && e == cudaSuccess; i++) {
        othello_slot *sl = &c->slot[i];
        e = cudaStreamCreateWithFlags(&sl->ctl, cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&sl->ready, cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&sl->done, cudaEventDisableTiming);
        for (int j = 0; j < kPipeStreams && e == cudaSuccess; j++)
            e = cudaEventCreateWithFlags(&sl->tail[j], cudaEventDisableTiming);
    }
    if (e == cudaSuccess) e = cudaHostAlloc((void **)&c->info_h, sizeof(othello_position_info), cudaHostAllocMapped);
    if (e == cudaSuccess) e = cudaHostGetDevicePointer((void **)&c->info_d, c->info_h, 0);
    if (e != cudaSuccess) { othello_ctx_destroy(c); return (int)e; }   // destroys exactly what was created
    *out = c;
    return 0;
}

int othello_ctx_set_option(othello_ctx *c, int32_t option, int64_t value)
{
    OB_CHECK_ARGS(c != nullptr);
    switch (option) {
    case OTHELLO_OPT_MAX_CHUNKS:
        OB_CHECK_ARGS(value >= 1 && value <= 64);
        c->max_chunks = (int)value;
        return 0;
    default:
        return OTHELLO_E_INVALID;
    }
}

int othello_board_apply_host(othello_ctx *c, uint64_t black, uint64_t white, int32_t color, int32_t move,
                             othello_position_info *info)
{
    OB_CHECK_ARGS(c && info);
    OB_CUDA(cudaSetDevice(c->device));
    board_kernel<<<1, 32, 0, c->stream>>>(black, white, color, move, c->info_d);
    OB_CUDA(cudaGetLastError());
    OB_CUDA(cudaStreamSynchronize(c->stream));
    *info = *c->info_h;
    return 0;
}

int othello_legal_host(othello_ctx *c, const uint64_t *own, const uint64_t *opp, uint64_t *legal, int64_t n)
{
    OB_CHECK_ARGS(c && n >= 0 && (n == 0 || (own && opp && legal)));
    if (n == 0) return 0;
    OB_CUDA(cudaSetDevice(c->device));
    int rc = idle_slot0(c);
    if (rc) return rc;
    rc = reserve(c, &c->slot[0], 3 * align256((size_t)n * 8));
    if (rc) return rc;
    c->slot[0].traj_black = nullptr;                     // the slot's trajectory is overwritten
    Carver k = {c->slot[0].ws, 0};
    uint64_t *d_own = k.take<uint64_t>(n), *d_opp = k.take<uint64_t>(n), *d_legal = k.take<uint64_t>(n);
    OBH_TRY(cudaMemcpyAsync(d_own, own, n * 8, cudaMemcpyHostToDevice, c->stream));
    OBH_TRY(cudaMemcpyAsync(d_opp, opp, n * 8, cudaMemcpyHostToDevice, c->stream));
    rc = othello_legal(d_own, d_opp, d_legal, n, c->stream);
    if (rc) return fail(c, rc);
    OBH_TRY(cudaMemcpyAsync(legal, d_legal, n * 8, cudaMemcpyDeviceToHost, c->stream));
    OBH_TRY(cudaStreamSynchronize(c->stream));
    return 0;
}

int othello_step_host(othello_ctx *c, uint64_t *black, uint64_t *white, uint8_t *turn, int32_t *nturn,
                      const uint8_t *move, uint64_t *flips_out, int32_t *ret, uint8_t *flags, int64_t n)
{
    OB_CHECK_ARGS(c && n >= 0 && (n == 0 || (black && white && turn && nturn && move)));
    if (n == 0) return 0;
    OB_CUDA(cudaSetDevice(c->device));
    int rc = idle_slot0(c);
    if (rc) return rc;
    rc = reserve(c, &c->slot[0], 3 * align256((size_t)n * 8) + 2 * align256((size_t)n * 4) + 3 * align256((size_t)n));
    if (rc) return rc;
    c->slot[0].traj_black = nullptr;
    Carver k = {c->slot[0].ws, 0};
    uint64_t *d_b = k.take<uint64_t>(n), *d_w = k.take<uint64_t>(n), *d_f = k.take<uint64_t>(n);
    int32_t *d_nt = k.take<int32_t>(n), *d_ret = k.take<int32_t>(n);
    uint8_t *d_t = k.take<uint8_t>(n), *d_mv = k.take<uint8_t>(n), *d_fl = k.take<uint8_t>(n);
    cudaStream_t s = c->stream;
    OBH_TRY(cudaMemcpyAsync(d_b, black, n * 8, cudaMemcpyHostToDevice, s));
    OBH_TRY(cudaMemcpyAsync(d_w, white, n * 8, cudaMemcpyHostToDevice, s));
    OBH_TRY(cudaMemcpyAsync(d_t, turn, n, cudaMemcpyHostToDevice, s));
    OBH_TRY(cudaMemcpyAsync(d_nt, nturn, n * 4, cudaMemcpyHostToDevice, s));
    OBH_TRY(cudaMemcpyAsync(d_mv, move, n, cudaMemcpyHostToDevice, s));
    rc = othello_step(d_b, d_w, d_t, d_nt, d_mv, d_f, d_ret, d_fl, n, s);
    if (rc) return fail(c, rc);
    OBH_TRY(cudaMemcpyAsync(black, d_b, n * 8, cudaMemcpyDeviceToHost, s));
    OBH_TRY(cudaMemcpyAsync(white, d_w, n * 8, cudaMemcpyDeviceToHost, s));
    OBH_TRY(cudaMemcpyAsync(turn, d_t, n, cudaMemcpyDeviceToHost, s));
    OBH_TRY(cudaMemcpyAsync(nturn, d_nt, n * 4, cudaMemcpyDeviceToHost, s));
    if (flips_out) OBH_TRY(cudaMemcpyAsync(flips_out, d_f, n * 8, cudaMemcpyDeviceToHost, s));
    if (ret) OBH_TRY(cudaMemcpyAsync(ret, d_ret, n * 4, cudaMemcpyDeviceToHost, s));
    if (flags) OBH_TRY(cudaMemcpyAsync(flags, d_fl, n, cudaMemcpyDeviceToHost, s));
    OBH_TRY(cudaStreamSynchronize(s));
    return 0;
}

int othello_playout_host_async(othello_ctx *c, uint64_t seed, uint64_t gid0, int64_t n, const uint64_t *black0,
                               const uint64_t *white0, const uint8_t *turn0, int32_t policy, int32_t random_plies,
                               int32_t n_rand_black, int32_t n_rand_white, const float *weights, int32_t policy_white,
                               const float *weights_white, int32_t t_max, uint64_t *traj_black, uint64_t *traj_white,
                               uint8_t *traj_move, int32_t *nplies, uint64_t *final_black, uint64_t *final_white,
                               uint16_t *summary, int64_t *totals, int64_t *ticket)
{
    OB_CHECK_ARGS(c && n >= 0 && t_max >= 0 && ticket);
    *ticket = 0;                                         // ticket 0 = nothing to wait for
    if (n == 0) { if (totals) totals[0] = totals[1] = totals[2] = totals[3] = 0; return 0; }
    OB_CHECK_ARGS((black0 == nullptr) == (white0 == nullptr));
    OB_CHECK_ARGS((final_black == nullptr) == (final_white == nullptr));
    OB_CHECK_ARGS((traj_black == nullptr) == (traj_white == nullptr) && (traj_black == nullptr) == (traj_move == nullptr));
    OB_CUDA(cudaSetDevice(c->device));
    const int si_slot = (int)(c->next_ticket % kSlots);
    othello_slot *sl = &c->slot[si_slot];
    const size_t row8 = align256((size_t)n * 8), row1 = align256((size_t)n);
    const size_t tb_bytes = align256((size_t)(t_max + 1) * n * 8), tm_bytes = align256((size_t)t_max * n + 1);
    int rc = reserve(c, sl, 4 * row8 + row1 + align256((size_t)n * 4) + align256((size_t)n * 2) + 3 * 256 + 2 * tb_bytes + tm_bytes);
    if (rc) return rc;
    Carver k = {sl->ws, 0};
    uint64_t *d_b0 = k.take<uint64_t>(n), *d_w0 = k.take<uint64_t>(n), *d_fb = k.take<uint64_t>(n), *d_fw = k.take<uint64_t>(n);
    uint8_t *d_t0 = k.take<uint8_t>(n);
    int32_t *d_np = k.take<int32_t>(n);
    uint16_t *d_sum = k.take<uint16_t>(n);
    float *d_wt = k.take<float>(OTHELLO_PHASES * OTHELLO_WEIGHTS), *d_wt2 = k.take<float>(OTHELLO_PHASES * OTHELLO_WEIGHTS);
    unsigned long long *d_tot = k.take<unsigned long long>(4);
    uint64_t *d_tb = k.take<uint64_t>((size_t)(t_max + 1) * n), *d_tw = k.take<uint64_t>((size_t)(t_max + 1) * n);
    uint8_t *d_tm = k.take<uint8_t>((size_t)t_max * n + 1);
    // The slot's previous batch (two tickets ago) ended on this very stream, so stream order already
    // protects the device buffers.  If the caller never waited for that batch, wait for it now: once its
    // slot has been reused, an old ticket must mean "complete" to othello_ctx_wait.
    cudaStream_t s = sl->ctl;
    if (sl->pending) { OBH_TRY(cudaEventSynchronize(sl->done)); sl->pending = false; }
    if (weights) OBH_TRY(cudaMemcpyAsync(d_wt, weights, sizeof(float) * OTHELLO_PHASES * OTHELLO_WEIGHTS, cudaMemcpyHostToDevice, s));
    if (weights_white) OBH_TRY(cudaMemcpyAsync(d_wt2, weights_white, sizeof(float) * OTHELLO_PHASES * OTHELLO_WEIGHTS, cudaMemcpyHostToDevice, s));
    if (totals) OBH_TRY(cudaMemsetAsync(d_tot, 0, 4 * sizeof(unsigned long long), s));
    OBH_TRY(cudaEventRecord(sl->ready, s));

    // Games are independent, so the batch is cut into chunks whose copy-in, kernel and copy-out run
    // on rotating streams: the PCIe traffic of one chunk hides behind the integer work of the others
    // (with pinned host buffers; pageable buffers simply serialise).  Kernels of different chunks run
    // concurrently, so a chunk smaller than one wave of the playout kernel costs no occupancy.
    int64_t chunk = (n + c->max_chunks - 1) / c->max_chunks;
    if (chunk < kMinChunk) chunk = kMinChunk;
    chunk = (chunk + 127) & ~(int64_t)127;
    bool used[kPipeStreams] = {false, false, false};
    for (int64_t c0 = 0; c0 < n; c0 += chunk) {
        const int64_t m = (n - c0 < chunk) ? n - c0 : chunk;
        const int si = (int)(c->chunk_seq++ % kPipeStreams);
        cudaStream_t st = c->pipe[si];
        if (!used[si]) { OBH_TRY(cudaStreamWaitEvent(st, sl->ready, 0)); used[si] = true; }
        if (black0) {
            OBH_TRY(cudaMemcpyAsync(d_b0 + c0, black0 + c0, m * 8, cudaMemcpyHostToDevice, st));
            OBH_TRY(cudaMemcpyAsync(d_w0 + c0, white0 + c0, m * 8, cudaMemcpyHostToDevice, st));
        }
        if (turn0) OBH_TRY(cudaMemcpyAsync(d_t0 + c0, turn0 + c0, m, cudaMemcpyHostToDevice, st));
        othello_playout_args a;
        a.seed = seed; a.gid0 = gid0 + (uint64_t)c0; a.n_games = m;
        a.black0 = black0 ? d_b0 + c0 : nullptr; a.white0 = black0 ? d_w0 + c0 : nullptr; a.turn0 = turn0 ? d_t0 + c0 : nullptr;
        a.policy = policy; a.random_plies = random_plies; a.n_rand_black = n_rand_black; a.n_rand_white = n_rand_white;
        a.weights = weights ? d_wt : nullptr;
        a.policy_white = policy_white; a.games_per_warp = 0; a.weights_white = weights_white ? d_wt2 : nullptr;
        a.t_max = t_max; a.stride = n;
        a.traj_black = d_tb + c0; a.traj_white = d_tw + c0; a.traj_move = d_tm + c0;
        a.nplies = d_np + c0; a.final_black = d_fb + c0; a.final_white = d_fw + c0;
        a.totals = totals ? d_tot : nullptr;
        a.summary = summary ? d_sum + c0 : nullptr;
        a.search_depth = 0; a.search_depth_white = 0; a.workspace = nullptr; a.workspace_bytes = 0;   // (no search engine)
        rc = othello_playout(&a, st);
        if (rc) return fail(c, rc);
        if (summary) OBH_TRY(cudaMemcpyAsync(summary + c0, d_sum + c0, m * 2, cudaMemcpyDeviceToHost, st));
        if (nplies) OBH_TRY(cudaMemcpyAsync(nplies + c0, d_np + c0, m * 4, cudaMemcpyDeviceToHost, st));
        if (final_black) {
            OBH_TRY(cudaMemcpyAsync(final_black + c0, d_fb + c0, m * 8, cudaMemcpyDeviceToHost, st));
            OBH_TRY(cudaMemcpyAsync(final_white + c0, d_fw + c0, m * 8, cudaMemcpyDeviceToHost, st));
        }
        if (traj_black) {
            // host and device trajectories are both [t][n]: a chunk is a column block
            OBH_TRY(cudaMemcpy2DAsync(traj_black + c0, (size_t)n * 8, d_tb + c0, (size_t)n * 8, (size_t)m * 8, t_max + 1, cudaMemcpyDeviceToHost, st));
            OBH_TRY(cudaMemcpy2DAsync(traj_white + c0, (size_t)n * 8, d_tw + c0, (size_t)n * 8, (size_t)m * 8, t_max + 1, cudaMemcpyDeviceToHost, st));
            if (t_max > 0)
                OBH_TRY(cudaMemcpy2DAsync(traj_move + c0, (size_t)n, d_tm + c0, (size_t)n, (size_t)m, t_max, cudaMemcpyDeviceToHost, st));
        }
    }
    sl->traj_black = d_tb; sl->traj_white = d_tw; sl->traj_move = d_tm; sl->traj_stride = n; sl->traj_t_max = t_max;
    sl->d_totals = d_tot;
    for (int i = 0; i < kPipeStreams; i++) {
        if (!used[i]) continue;
        OBH_TRY(cudaEventRecord(sl->tail[i], c->pipe[i]));
        OBH_TRY(cudaStreamWaitEvent(s, sl->tail[i], 0));
    }
    if (totals) OBH_TRY(cudaMemcpyAsync(totals, d_tot, 4 * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    OBH_TRY(cudaEventRecord(sl->done, s));
    sl->pending = true;
    sl->ticket = c->next_ticket;
    c->last_slot = si_slot;
    *ticket = c->next_ticket++;
    return 0;
}

int othello_ctx_wait(othello_ctx *c, int64_t ticket)
{
    OB_CHECK_ARGS(c && ticket >= 0 && ticket < c->next_ticket);
    if (ticket == 0) return 0;
    othello_slot *sl = &c->slot[ticket % kSlots];
    // an older ticket of this slot was completed (waited for) when the slot was reused
    if (sl->pending && sl->ticket == ticket) {
        OB_CUDA(cudaSetDevice(c->device));
        OB_CUDA(cudaEventSynchronize(sl->done));
        sl->pending = false;
    }
    return 0;
}

int othello_playout_host(othello_ctx *c, uint64_t seed, uint64_t gid0, int64_t n, const uint64_t *black0,
                         const uint64_t *white0, const uint8_t *turn0, int32_t policy, int32_t random_plies,
                         int32_t n_rand_black, int32_t n_rand_white, const float *weights, int32_t policy_white,
                         const float *weights_white, int32_t t_max, uint64_t *traj_black, uint64_t *traj_white, uint8_t *traj_move, int32_t *nplies,
                         uint64_t *final_black, uint64_t *final_white)
{
    OB_CHECK_ARGS(c && n >= 0);
    if (n == 0) return 0;
    OB_CHECK_ARGS(nplies && final_black && final_white);
    int64_t ticket = 0;
    int rc = othello_playout_host_async(c, seed, gid0, n, black0, white0, turn0, policy, random_plies, n_rand_black,
                                        n_rand_white, weights, policy_white, weights_white, t_max, traj_black, traj_white,
                                        traj_move, nplies, final_black, final_white, nullptr, nullptr, &ticket);
    if (rc) return rc;
    return othello_ctx_wait(c, ticket);
}

int othello_ctx_trajectory(othello_ctx *c, uint64_t **traj_black, uint64_t **traj_white, uint8_t **traj_move,
                           int64_t *stride, int32_t *t_max)
{
    OB_CHECK_ARGS(c && c->last_slot >= 0 && c->slot[c->last_slot].traj_black);
    const othello_slot *sl = &c->slot[c->last_slot];
    if (traj_black) *traj_black = sl->traj_black;
    if (traj_white) *traj_white = sl->traj_white;
    if (traj_move) *traj_move = sl->traj_move;
    if (stride) *stride = sl->traj_stride;
    if (t_max) *t_max = sl->traj_t_max;
    return 0;
}

}  // extern "C"
