// common.cuh -- launch helpers shared by the translation units of libothello_b200.so
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/othello_b200.h"
#include "bitboard.cuh"

#define OB_CHECK_ARGS(cond) do { if (!(cond)) return OTHELLO_E_INVALID; } while (0)

// Surface the launch error (if any) of the kernel just enqueued, as the C ABI's return code.
static inline int ob_launch_status()
{
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : (int)e;
}

#define OB_CUDA(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return (int)e_; } while (0)

static inline unsigned ob_blocks(int64_t n, int threads) { return (unsigned)((n + threads - 1) / threads); }

// The grid of a persistent kernel whose lanes take their work from a counter: as many CTAs as fit on the device at
// once (a CTA beyond that would only start once the work had run out), fewer for a small n.
template <typename Kernel>
static inline int ob_persistent_blocks(Kernel kernel, int threads, int64_t n, unsigned &blocks)
{
    int dev = 0, sms = 0, per_sm = 0;
    OB_CUDA(cudaGetDevice(&dev));
    OB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    OB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, 0));
    const int64_t want = (n + threads - 1) / threads, fit = (int64_t)sms * (per_sm > 0 ? per_sm : 1);
    blocks = (unsigned)(want < fit ? want : fit);
    return 0;
}
