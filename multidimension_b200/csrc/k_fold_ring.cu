// k_fold_ring.cu — fold over the SHARDED (outermost) axis, bit-identical to the reference's sequential add chain,
// as ONE fused compute + exchange kernel per GPU over NVLink peer memory (no NCCL call on the data path).
//
// The reference sums  s = init; for i in 0..I { s = s (op) x[i][c] }  strictly in index order (src/view.rs:250-252,
// 617-622).  With the I axis cut over N GPUs (rank r owns rows [r I/N, (r+1) I/N)) that chain runs THROUGH the ranks:
// rank 0 folds its rows from `init`, hands the running values to rank 1, which continues with its rows, ... rank N-1
// ends with the result — the same sequence of roundings as one GPU folding all the rows, so the result is bit-exact
// (an all-reduce reassociates the sum: 1e-6 relative, SURVEY.md §8e).  The chain is pipelined over column slices:
//
//   CTA (persistent, one per SM) loops over slices of 256 columns; per slice
//     producer thread : TMA (cp.async.bulk.tensor.2d, UTMALDG) streams the rank's rows of that slice through a ring of
//                       32 KB shared-memory stages (full / empty mbarriers), far ahead of the adds;
//     consumers       : 64 threads, 4 columns each: poll THIS GPU's inbox for the previous rank's running values of this
//                       slice, fold the staged rows in order, then store the running values into the NEXT rank's inbox.
//                       The hand-off is flag-in-data: 16-byte lines {word, epoch, word, epoch} written with one volatile
//                       vector store into peer-mapped HBM; the receiver trusts a line once both epochs match (8-byte store
//                       atomicity suffices — NCCL's LL argument), so a hop costs one NVLink store latency: no fence, no
//                       separate flag, no publisher thread.
//   The last rank writes the finished slice as the same kind of lines into every rank's result area; every CTA copies
//   its slices from the local result area to `out` as their lines arrive, so stream order still means "the kernel has
//   completed => out is complete on this GPU".  One set of areas suffices: a rank cannot start launch e+1 before it has
//   all of launch e's results, which exist only after every rank has consumed its launch-e inbox.
//
// Rank r starts slice s as soon as rank r-1 has finished it, so with S slices per CTA the whole fold takes about
// T_local (1 + (N-1)/S) + (N-1) hops instead of N T_local; measured on 8 GPUs: see profiles/r2_scale_ops.md.
// Spins are bounded (~2 s): a rank that never arrives turns into MDIM_ERR_NCCL on the others, not a hung GPU.
#include <cuda.h>
#include <stdlib.h>
#include <string.h>

#include "exec.cuh"
#include "kernels.cuh"

namespace mdim {

namespace {

constexpr int kRingThreads = 96;        // warp 0: producer (one lane); warps 1-2: consumers
constexpr int kRingCons = 64;
constexpr int kRingStageBytes = 32 * 1024;
constexpr int kRingStages = 6;
constexpr unsigned long long kSpinLimit = 3ull * 1000 * 1000;  // polls of a local line (one L2 round trip each, ~0.7 us): ~2 s

__device__ __forceinline__ uint32_t rsm(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void st_line(char* p, uint32_t a, uint32_t b, uint32_t flag) {
    asm volatile("st.volatile.global.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(a), "r"(flag), "r"(b), "r"(flag) : "memory");
}
__device__ __forceinline__ uint4 ld_line(const char* p) {
    uint4 v;
    asm volatile("ld.volatile.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
    return v;
}
// -> false when `*give_up` is raised before the phase completes (a peer never arrived: the producer has stopped)
__device__ __forceinline__ bool mbar_wait_parity_or(uint32_t bar, uint32_t parity, const volatile int* give_up) {
    for (;;) {
        uint32_t done;
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n" : "=r"(done) : "r"(bar), "r"(parity) : "memory");
        if (done) return true;
        if (*give_up) return false;
    }
}
// polls one line until both epochs match; -> false on timeout
__device__ __forceinline__ bool wait_line(const char* p, uint32_t epoch, uint4& v) {
    for (unsigned long long spins = 0; spins < kSpinLimit; ++spins) {
        v = ld_line(p);
        if (v.y == epoch && v.w == epoch) return true;
        if (spins > 8) __nanosleep(32);
    }
    return false;
}

// One staged tile folded into the running values, strictly in row order: this IS the reference's add chain.  The element type
// and operator are compile-time here (bin_op's switches fold away): dispatched once per tile, not once per element.
template <class S, int DT, int OP>
__device__ __forceinline__ void fold_tile(S (&acc)[4], uint32_t p, uint32_t rows) {
    constexpr int ES = (int)sizeof(S), SC = kRingCons * 4;
#pragma unroll 8
    for (uint32_t r = 0; r < rows; ++r) {
        S x[4];
        if constexpr (ES == 4) asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(x[0]), "=r"(x[1]), "=r"(x[2]), "=r"(x[3]) : "r"(p + r * SC * ES));
        else {
            asm volatile("ld.shared.v2.u64 {%0,%1}, [%2];" : "=l"(x[0]), "=l"(x[1]) : "r"(p + r * SC * ES));
            asm volatile("ld.shared.v2.u64 {%0,%1}, [%2];" : "=l"(x[2]), "=l"(x[3]) : "r"(p + r * SC * ES + 16));
        }
#pragma unroll
        for (int e = 0; e < 4; ++e) { bool arith = false; acc[e] = bin_op<S, false>(DT, OP, DT, acc[e], x[e], arith); }
    }
}
template <class S, int DT>
__device__ __forceinline__ void fold_tile_op(int op, S (&acc)[4], uint32_t p, uint32_t rows) {
    switch (op) {
        case MDIM_ADD: fold_tile<S, DT, MDIM_ADD>(acc, p, rows); break;
        case MDIM_SUB: fold_tile<S, DT, MDIM_SUB>(acc, p, rows); break;
        case MDIM_MUL: fold_tile<S, DT, MDIM_MUL>(acc, p, rows); break;
        case MDIM_AND: fold_tile<S, DT, MDIM_AND>(acc, p, rows); break;
        case MDIM_OR: fold_tile<S, DT, MDIM_OR>(acc, p, rows); break;
        default: fold_tile<S, DT, MDIM_XOR>(acc, p, rows); break;
    }
}
template <class S>
__device__ __forceinline__ void fold_tile_dispatch(int dtype, int op, S (&acc)[4], uint32_t p, uint32_t rows) {
    if constexpr (sizeof(S) == 4) {
        if (dtype == MDIM_F32) fold_tile_op<S, MDIM_F32>(op, acc, p, rows);
        else if (dtype == MDIM_I32) fold_tile_op<S, MDIM_I32>(op, acc, p, rows);
        else fold_tile_op<S, MDIM_U32>(op, acc, p, rows);
    } else {
        if (dtype == MDIM_F64) fold_tile_op<S, MDIM_F64>(op, acc, p, rows);
        else if (dtype == MDIM_I64) fold_tile_op<S, MDIM_I64>(op, acc, p, rows);
        else fold_tile_op<S, MDIM_U64>(op, acc, p, rows);
    }
}

template <class S>  // S = uint32_t (4-byte elements) or uint64_t (8-byte)
__global__ void __launch_bounds__(kRingThreads) k_fold_ring(const __grid_constant__ CUtensorMap rows_map, const __grid_constant__ FoldRingArgs A) {
    constexpr int ES = (int)sizeof(S), EPT = 4;            // elements per consumer thread
    constexpr int SC = kRingCons * EPT;                     // columns per slice (256)
    constexpr int ROWS = kRingStageBytes / (SC * ES);       // rows per stage (32 or 16)
    constexpr int LPT = EPT * ES / 8;                       // 16-byte lines per consumer thread and slice (2 or 4): 8 data bytes each
    extern __shared__ uint8_t ring_raw[];
    const uint32_t base = (rsm(ring_raw) + 127u) & ~127u;
    const uint32_t bars = base + kRingStages * kRingStageBytes;  // full[s] at bars + 16 s, empty[s] at bars + 16 s + 8
    __shared__ int timed_out;
    const int tid = threadIdx.x, warp = tid >> 5;
    pdl_entry(false);  // reads the caller's rows: always waits for its predecessor in the stream
    if (tid == 0) {
        timed_out = 0;
        for (int s = 0; s < kRingStages; ++s) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bars + 16 * s) : "memory");
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bars + 16 * s + 8), "r"(kRingCons) : "memory");
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const uint64_t n_slices = (A.n_cols + SC - 1) / SC;
    const uint32_t n_row_tiles = (uint32_t)((A.n_rows + ROWS - 1) / ROWS);
    const volatile int* give_up = &timed_out;
    uint32_t fill = 0, drain = 0;  // stage counters (producer / consumers): stage = k % kRingStages, parity = (k / kRingStages) & 1
    if (warp == 0) {
        if (tid == 0) {  // ---- producer: every row tile of every slice of this CTA, in order ------------------------------
            for (uint64_t s = blockIdx.x; s < n_slices; s += gridDim.x) {
                for (uint32_t t = 0; t < n_row_tiles; ++t, ++fill) {
                    const uint32_t st = fill % kRingStages;
                    // the consumers have left this stage (or given up: a peer never arrived)
                    if (fill >= kRingStages && !mbar_wait_parity_or(bars + 16 * st + 8, ((fill / kRingStages) - 1) & 1, give_up)) goto producer_done;
                    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bars + 16 * st), "r"((uint32_t)kRingStageBytes) : "memory");
                    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(base + st * kRingStageBytes),
                                 "l"(&rows_map), "r"((int)(s * SC)), "r"((int)(t * ROWS)), "r"(bars + 16 * st)
                                 : "memory");
                }
            }
        producer_done:
            if (*give_up) __nanosleep(200000);  // let the loads still in flight land before the CTA gives its shared memory back
        }
    } else {  // ---- consumers: 64 threads, EPT consecutive columns each -----------------------------------------------------
        const int ct = tid - 32;
        const bool first = A.rank == 0, last = A.rank == A.world - 1;
        for (uint64_t s = blockIdx.x; s < n_slices && !*give_up; s += gridDim.x) {
            const uint64_t col = s * SC + (uint64_t)ct * EPT;
            const bool live = col < A.n_cols;   // n_cols * ES is a multiple of 16 and EPT * ES of 16: a thread's columns are all in or all out
            S acc[EPT];
            if (first || !live) {
#pragma unroll
                for (int e = 0; e < EPT; ++e) acc[e] = (S)A.init;
            } else {  // the previous rank's running values of these columns: lines in THIS GPU's inbox
                uint32_t w[2 * LPT];
                bool ok = true;
#pragma unroll
                for (int l = 0; l < LPT; ++l) {
                    uint4 v;
                    ok = ok && wait_line((const char*)A.inbox + s * (2 * SC * ES) + (l * kRingCons + ct) * 16, A.epoch, v);
                    w[2 * l] = v.x; w[2 * l + 1] = v.z;
                }
                if (!ok) { timed_out = 1; break; }
#pragma unroll
                for (int e = 0; e < EPT; ++e) {
                    if constexpr (ES == 4) acc[e] = w[e];
                    else acc[e] = (uint64_t)w[2 * e] | ((uint64_t)w[2 * e + 1] << 32);
                }
            }
            bool staged = true;
            for (uint32_t t = 0; t < n_row_tiles; ++t, ++drain) {
                const uint32_t st = drain % kRingStages;
                if (!mbar_wait_parity_or(bars + 16 * st, (drain / kRingStages) & 1, give_up)) { staged = false; break; }
                const uint32_t rows = min((uint64_t)ROWS, A.n_rows - (uint64_t)t * ROWS);
                const uint32_t p = base + st * kRingStageBytes + (uint32_t)ct * EPT * ES;
                fold_tile_dispatch<S>(A.dtype, A.op, acc, p, rows);
                asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bars + 16 * st + 8) : "memory");
            }
            if (!staged) break;
            if (!live) continue;
            // hand the running values on (or, on the last rank, publish the result to everyone): flag-in-data lines
            uint32_t w[2 * LPT];
#pragma unroll
            for (int e = 0; e < EPT; ++e) {
                if constexpr (ES == 4) w[e] = acc[e];
                else { w[2 * e] = (uint32_t)acc[e]; w[2 * e + 1] = (uint32_t)(acc[e] >> 32); }
            }
            const int n_dst = last ? A.world : 1;
            for (int k = 0; k < n_dst; ++k) {
                int d = A.rank + 1 + k;  // the last rank serves the others first, itself last
                if (d >= A.world) d -= A.world;
                // a slice's lines: [line 0..LPT-1][consumer], so every warp store instruction writes 512 contiguous bytes
                char* dst = (char*)(last ? A.result[d] : A.next_inbox) + s * (2 * SC * ES) + ct * 16;
#pragma unroll
                for (int l = 0; l < LPT; ++l) st_line(dst + l * (kRingCons * 16), w[2 * l], w[2 * l + 1], A.epoch);
            }
        }
    }
    __syncthreads();
    // ---- every slice of this CTA: copy the finished values from the local result area to `out` as their lines arrive (all threads;
    //      one line = 8 bytes of `out`) -------------------------------------------------------------------------------------------
    const uint32_t my_slices = blockIdx.x < n_slices ? (uint32_t)((n_slices - blockIdx.x + gridDim.x - 1) / gridDim.x) : 0;
    constexpr uint32_t LPS = SC * ES / 8;  // lines per slice
    for (uint32_t k = tid; k < my_slices * LPS && !*give_up; k += kRingThreads) {
        const uint64_t s = blockIdx.x + (uint64_t)(k / LPS) * gridDim.x;
        const uint32_t j = k % LPS, l = j / kRingCons, ct = j % kRingCons;                        // line j of the slice = line l of consumer ct
        const uint64_t byte = s * (uint64_t)(SC * ES) + (uint64_t)ct * (EPT * ES) + l * 8;      // where its 8 data bytes live in `out`
        if (byte >= A.n_cols * ES) continue;
        uint4 v;
        if (!wait_line((const char*)A.result[A.rank] + s * (2 * SC * ES) + j * 16, A.epoch, v)) { timed_out = 1; break; }
        *(uint2*)((char*)A.out + byte) = make_uint2(v.x, v.z);
    }
    __syncthreads();
    if (timed_out && tid == 0) atomicExch(A.error, 1u);
}

typedef CUresult (*EncodeTiledFn2)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                   CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

}  // namespace

// -> 0 ok; cudaError / -1 when the rows cannot be described by a tensor map (misaligned pointer or row pitch)
int launch_fold_ring(const FoldRingArgs& A, const void* rows, int sm_count, cudaStream_t stream) {
    static const EncodeTiledFn2 encode = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) p = nullptr;
        return (EncodeTiledFn2)p;
    }();
    const int es = A.esize;
    if (!encode || ((uintptr_t)rows & 15) || ((uintptr_t)A.out & 7) || (A.n_cols * (uint64_t)es) % 16 != 0 || A.n_rows == 0 || A.n_cols == 0) return -1;
    const uint32_t words = (uint32_t)(es / 4);
    CUtensorMap map;
    cuuint64_t dims[2] = {A.n_cols * words, A.n_rows}, strides[1] = {A.n_cols * (uint64_t)es};
    cuuint32_t box[2] = {(cuuint32_t)(kRingCons * 4 * words), (cuuint32_t)(kRingStageBytes / (kRingCons * 4 * es))}, estr[2] = {1, 1};
    if (box[0] > 256) {  // 8-byte elements: 512 words per row exceed the 256-element box limit -> describe pairs of words as one 8-byte element
        dims[0] = A.n_cols; box[0] = kRingCons * 4;
        if (encode(&map, CU_TENSOR_MAP_DATA_TYPE_UINT64, 2, const_cast<void*>(rows), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS) return -1;
    } else if (encode(&map, CU_TENSOR_MAP_DATA_TYPE_UINT32, 2, const_cast<void*>(rows), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                      CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS) return -1;
    const size_t smem = (size_t)kRingStages * kRingStageBytes + 16 * kRingStages + 256;
    const uint64_t n_slices = (A.n_cols + kRingCons * 4 - 1) / (kRingCons * 4);
    const int grid = (int)std::min<uint64_t>(n_slices, (uint64_t)sm_count);  // one CTA per SM: every CTA is resident, so waiting on peers cannot starve anyone
    cudaError_t e;
    if (es == 4) {
        static const bool ok = cudaFuncSetAttribute(k_fold_ring<uint32_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) == cudaSuccess;
        if (!ok) return -1;
        e = launch_pdl(k_fold_ring<uint32_t>, dim3(grid), dim3(kRingThreads), smem, stream, map, A);
    } else {
        static const bool ok = cudaFuncSetAttribute(k_fold_ring<uint64_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) == cudaSuccess;
        if (!ok) return -1;
        e = launch_pdl(k_fold_ring<uint64_t>, dim3(grid), dim3(kRingThreads), smem, stream, map, A);
    }
    return e == cudaSuccess ? 0 : (int)e;
}

}  // namespace mdim
