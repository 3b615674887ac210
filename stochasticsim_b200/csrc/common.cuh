// common.cuh -- context object and error plumbing shared by every translation unit of libssb200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include "../../include/ssb200.h"

struct ssb_ctx {
    int          device;
    cudaStream_t stream;       // compute stream (all kernels + the timer)
    cudaStream_t copy_stream;  // second stream for double-buffered host<->device copies
    cudaEvent_t  t0, t1;
    cudaEvent_t  ev[4];        // scratch events for stream hand-offs
    int          sm_count;
    size_t       total_mem;
    char         name[128];
    char         err[512];
    uint64_t     launches;
    // lazily grown device scratch, reused across calls
    void        *scratch;
    size_t       scratch_bytes;
    void        *pinned;
    size_t       pinned_bytes;
    // optional per-kernel device timing (ssb_profile_*): CUDA events around individual launches
    int          prof_on;
    struct ssb_prof *prof;
};

// kernel slots for ssb_profile_read()
enum { SSB_K_TNC_SCAN = 0, SSB_K_TNC_FIXUP = 1, SSB_K_SPIKE_PARSE = 2, SSB_K_SPIKE_EMIT = 3, SSB_K_SPIKE_CHAIN = 4,
       SSB_K_SPIKE_OTHER = 5, SSB_K_SPIKE_TALLY = 6, SSB_K_TNC_INTERVALS = 7, SSB_K_SLOTS = 8 };
void ssb_prof_begin(ssb_ctx *ctx, int slot, cudaStream_t s);
void ssb_prof_end(ssb_ctx *ctx, int slot, cudaStream_t s);

#define SSB_CUDA(ctx, call)                                                                  \
    do {                                                                                     \
        cudaError_t e_ = (call);                                                             \
        if (e_ != cudaSuccess) {                                                             \
            snprintf((ctx)->err, sizeof((ctx)->err), "%s:%d: %s: %s", __FILE__, __LINE__,    \
                     #call, cudaGetErrorString(e_));                                         \
            return SSB_E_CUDA;                                                               \
        }                                                                                    \
    } while (0)

// Every kernel launch goes through this so ssb_kernel_launches() is an honest count.
#define SSB_LAUNCH(ctx, kernel, grid, block, smem, stream, ...)                              \
    do {                                                                                     \
        kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__);                          \
        (ctx)->launches++;                                                                   \
        SSB_CUDA(ctx, cudaGetLastError());                                                   \
    } while (0)

// Same, with the launch bracketed by profiling events when ssb_profile_enable() is on.
#define SSB_LAUNCH_P(ctx, slot, kernel, grid, block, smem, stream, ...)                      \
    do {                                                                                     \
        if ((ctx)->prof_on) ssb_prof_begin((ctx), (slot), (stream));                         \
        kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__);                          \
        (ctx)->launches++;                                                                   \
        if ((ctx)->prof_on) ssb_prof_end((ctx), (slot), (stream));                           \
        SSB_CUDA(ctx, cudaGetLastError());                                                   \
    } while (0)

int ssb_scratch_reserve(ssb_ctx *ctx, size_t bytes);   // ctx->scratch has at least `bytes`
int ssb_pinned_reserve(ssb_ctx *ctx, size_t bytes);    // ctx->pinned  has at least `bytes`
