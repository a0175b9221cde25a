// ctx.hpp — the context behind the C ABI (internal; shared by api.cu and comm.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdio.h>
#include <string.h>

#include <vector>

#include "program.hpp"

namespace mdim {

constexpr int kErrSlots = 64;

struct Pending {
    Plan* plan;  // heap copy, only for collects that can fail on the device
    void* out;
    int slot;
    uint64_t pos_base;  // added to the reported position (chunks of a host collect)
};

struct HostPipe {  // staging for mdim_collect_host
    cudaStream_t h2d = nullptr, d2h = nullptr;
    cudaEvent_t up[2] = {nullptr, nullptr}, done[2] = {nullptr, nullptr}, down[2] = {nullptr, nullptr};
    char* arena = nullptr;  // grow-only device staging arena
    size_t arena_bytes = 0;
};

struct Comm;  // comm.cu: NCCL communicator + peer tables (one process per GPU)

}  // namespace mdim

struct mdim_ctx {
    int device = 0;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    mdim::ErrWord* d_err = nullptr;  // kErrSlots device error words
    mdim::ErrWord* h_err = nullptr;  // pinned mirror
    int next_slot = 0;
    std::vector<mdim::Pending> pending;
    uint64_t launches = 0;
    int sm_count = 0, cc_major = 0, cc_minor = 0;
    size_t hbm = 0;
    mdim_error_info last;
    mdim::HostPipe pipe;
    uint64_t pos_base = 0;  // applied to collects issued while a host collect is chunking
    // Dependency-aware launches (launch.cuh): byte ranges touched by the kernels launched on own_stream since the last one
    // that waited for its predecessor.  A launch that conflicts with none of them skips the wait.
    struct Touched { uint64_t lo, hi; bool write; };
    std::vector<Touched> inflight;
    bool dep_tracking = true;  // MDIM_DEP_TRACK=0: every kernel waits (round-1 behaviour)
    size_t host_chunk_bytes = 128u << 20;  // measured: 8 MB 60.7, 32 MB 73.1, 128 MB 75.8, 512 MB 76.3 GB/s end to end
    mdim::Comm* comm = nullptr;  // mdim_comm_init (comm.cu)
    char last_kernel[96] = {0};  // mdim_last_kernel: what the last collect actually launched
    // k_fold_split's scratch: kSplitMaxOuts tickets (zeroed once here; every launch leaves them at 0), then the chunks' partials.
    // Grown on first use, freed by mdim_shutdown.  Every split fold writes it, so may_skip_wait never lets two overlap.
    char* split_scratch = nullptr;
    size_t split_scratch_bytes = 0;
};

namespace mdim {

inline int cuda_fail(mdim_ctx* ctx, cudaError_t e, const char* what) {
    if (ctx) {
        memset(&ctx->last, 0, sizeof ctx->last);
        ctx->last.status = MDIM_ERR_CUDA;
        ctx->last.node = -1;
        snprintf(ctx->last.message, sizeof ctx->last.message, "%s: %s", what, cudaGetErrorString(e));
    }
    return e == cudaErrorMemoryAllocation ? MDIM_ERR_NOMEM : MDIM_ERR_CUDA;
}

#define CU(ctx, call)                                     \
    do {                                                  \
        cudaError_t e_ = (call);                          \
        if (e_ != cudaSuccess) return mdim::cuda_fail(ctx, e_, #call); \
    } while (0)

inline int set_error(mdim_ctx* ctx, int status, const char* msg) {
    memset(&ctx->last, 0, sizeof ctx->last);
    ctx->last.status = status;
    ctx->last.node = -1;
    snprintf(ctx->last.message, sizeof ctx->last.message, "%s", msg);
    return status;
}

// A kernel that is not one of ours (NCCL) ran on the stream: the next collect must wait for its predecessor.
inline void poison_inflight(mdim_ctx* ctx) {
    ctx->inflight.clear();
    ctx->inflight.push_back({0, ~0ull, true});
}

void comm_destroy(mdim_ctx* ctx);  // comm.cu (called by mdim_shutdown)

}  // namespace mdim
