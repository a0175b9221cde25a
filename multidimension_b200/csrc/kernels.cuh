// kernels.cuh — __global__ entry points (sm_100a) and their host-side launch table.
#pragma once
#include <cuda_runtime.h>

#include "exec.cuh"
#include "launch.cuh"
#include "program.hpp"

namespace mdim {

constexpr int kEvalThreads = 256;

// ------------------------------------------------------------------------------------------------
// K1 / K3 / K5: the rank-N fused evaluator.  One thread = one output vector per loop trip; the
// grid has one thread per vector (more trips only past 2^31 - 1 CTAs).
// All operands are read-only and never alias `out` (C-ABI contract), so loads use the
// non-coherent path; stores are streaming (evict-first) because nothing re-reads the output.
// ------------------------------------------------------------------------------------------------
template <class Sig, class S, int V, int MAXD, bool WIDE, int MAXR>
__global__ void __launch_bounds__(kEvalThreads)
k_eval(const __grid_constant__ Program P, void* __restrict__ out, ErrWord* __restrict__ err, uint64_t g_begin, uint64_t g_end) {
    pdl_entry((P.flags & PF_NOWAIT) != 0);
    const uint64_t step = (uint64_t)gridDim.x * kEvalThreads;
    for (uint64_t g = g_begin + (uint64_t)blockIdx.x * kEvalThreads + threadIdx.x; g < g_end; g += step)
        eval_vector<Sig, S, V, MAXD, WIDE, MAXR>(P, out, err, g);
}

using EvalKernel = void (*)(const Program, void*, ErrWord*, uint64_t, uint64_t);

// The kernels of the variants_*.inc lists, in list order, defined in k_eval_{s32,s64}_{interp,static}.cu (four translation units:
// the build parallelises over them).  Concatenated s32 static, s64 static, s32 interp, s64 interp they follow kEvalVariants.
const EvalKernel* eval_kernels_s32_interp(int* n);
const EvalKernel* eval_kernels_s32_static(int* n);
const EvalKernel* eval_kernels_s64_interp(int* n);
const EvalKernel* eval_kernels_s64_static(int* n);

// The launchers of the dedicated kernels (KK_TRANSPOSE, KK_FOLD_ROWS, KK_FOLD_COLS, KK_FOLD_SPLIT) share one shape: each launches its
// plan's kernel on `stream`, without griddepcontrol.wait if `nowait` (launch.cuh), and returns the name of the kernel launched,
// nullptr on a launch error.

// ------------------------------------------------------------------------------------------------
// K2: tiled transpose of one leaf (see k_transpose.cu)
// ------------------------------------------------------------------------------------------------
constexpr int kTrThreads = 256;
const char* launch_transpose(const Plan& p, void* out, bool nowait, cudaStream_t stream, int sm_count);

// ------------------------------------------------------------------------------------------------
// K4: sequential-order last-axis fold, optionally fused with a broadcast epilogue (k_fold.cu)
// ------------------------------------------------------------------------------------------------
constexpr int kFoldThreads = 256;
const char* launch_fold_rows(const Plan& p, void* out, bool nowait, cudaStream_t stream, int sm_count);

// ------------------------------------------------------------------------------------------------
// Fold over the SHARDED axis, bit-exact, pipelined through the ranks over NVLink (k_fold_ring.cu)
// ------------------------------------------------------------------------------------------------
int launch_fold_ring(const FoldRingArgs& A, const void* rows, int sm_count, cudaStream_t stream);

// Fold over the SHARDED axis, blocked by rank + in-kernel all-reduce in rank order over NVLink (k_fold_xchg.cu)
int launch_fold_xchg(const FoldXchgArgs& A, int dtype, int op, int sm_count, cudaStream_t stream);
// ... and the same column walk on one GPU, no exchange (KK_FOLD_COLS)
const char* launch_fold_cols(const Plan& p, void* out, bool nowait, cudaStream_t stream, int sm_count);

// ------------------------------------------------------------------------------------------------
// Integer fold with few outputs and a long reduction, the reduction cut into chunks over the whole GPU (k_fold_split.cu)
// ------------------------------------------------------------------------------------------------
// Its scratch holds kSplitMaxOuts tickets, zeroed before first use and left at zero by every launch, then the chunks' partials.
size_t fold_split_scratch_bytes(const FoldSplitPlan& F, int sm_count);
const char* launch_fold_split(const Plan& p, void* out, bool nowait, cudaStream_t stream, int sm_count, char* scratch);

}  // namespace mdim
