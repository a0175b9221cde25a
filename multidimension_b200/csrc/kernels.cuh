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

struct EvalVariant {
    const char* name;
    int slot_bytes, vec, max_depth, wide, maxr;  // maxr: iteration axes walked (1 = contiguous stream)
    const SigInstr* sig;  // nullptr = interpreter
    int sig_n;
    EvalKernel fn;
};

// defined in k_eval_{s32,s64}_{interp,static}.cu (four translation units: the build parallelises over them)
const EvalVariant* eval_variants_s32_interp(int* n);
const EvalVariant* eval_variants_s32_static(int* n);
const EvalVariant* eval_variants_s64_interp(int* n);
const EvalVariant* eval_variants_s64_static(int* n);

// ------------------------------------------------------------------------------------------------
// K2: tiled transpose of one leaf (see k_transpose.cu)
// ------------------------------------------------------------------------------------------------
constexpr int kTrThreads = 256;
const char* launch_transpose(const TransposePlan& T, void* out, int grid, cudaStream_t stream);  // -> name of the kernel launched

// ------------------------------------------------------------------------------------------------
// K4: sequential-order last-axis fold, optionally fused with a broadcast epilogue (k_fold.cu)
// ------------------------------------------------------------------------------------------------
constexpr int kFoldThreads = 256;
const char* launch_fold_rows(const FoldRowsPlan& R, void* out, int sm_count, cudaStream_t stream);  // -> name of the kernel launched

// ------------------------------------------------------------------------------------------------
// Fold over the SHARDED axis, bit-exact, pipelined through the ranks over NVLink (k_fold_ring.cu)
// ------------------------------------------------------------------------------------------------
int launch_fold_ring(const FoldRingArgs& A, const void* rows, int sm_count, cudaStream_t stream);

// Fold over the SHARDED axis, blocked by rank + in-kernel all-reduce in rank order over NVLink (k_fold_xchg.cu)
int launch_fold_xchg(const FoldXchgArgs& A, int dtype, int op, int sm_count, cudaStream_t stream);
// ... and the same column walk on one GPU, no exchange (KK_FOLD_COLS): -> name of the kernel launched, nullptr on a launch error
const char* launch_fold_cols(const FoldColsPlan& C, void* out, cudaStream_t stream);

// ------------------------------------------------------------------------------------------------
// Integer fold with few outputs and a long reduction, the reduction cut into chunks over the whole GPU (k_fold_split.cu)
// ------------------------------------------------------------------------------------------------
struct SplitGeometry {
    uint64_t units;     // RUNS: outputs; COLS: batches.  Each has one ticket.
    uint64_t n_chunks;  // chunks per unit: the grid is units x n_chunks CTAs
    uint64_t chunk;     // RUNS: elements per chunk; COLS: rows per chunk
    uint64_t partials;  // slots of scratch the launch writes (each slot_bytes wide)
};
SplitGeometry fold_split_geometry(const FoldSplitPlan& F, int sm_count);
// tickets: units zeroed words; partials: G.partials slots.  -> name of the instantiation launched, nullptr on a launch error
const char* launch_fold_split(const FoldSplitPlan& F, const SplitGeometry& G, void* out, unsigned int* tickets, void* partials,
                              cudaStream_t stream, char* name, size_t name_len);

}  // namespace mdim
