// k_fold_split.cu — an integer fold with few outputs and a long reduction, spread over the whole GPU (sm_100a).
//
// Wrapping +, *, &, | and ^ are associative and commutative, and a Sub fold equals init - (x0 + x1 + ...) under wrapping, so
// for these operators any order of combination gives exactly the bits of the reference's left-to-right fold (the same fact
// k_fold_xchg relies on at rank boundaries).  Each output's reduction is therefore cut into chunks, one CTA per (output unit,
// chunk):
//   walk     : threads stream the chunk — 256-bit loads of a run (RUNS), or 128-bit column groups row after row (COLS) — and
//              fold each element into a 32- or 64-bit slot.  An element is first sign- or zero-extended from its source width, or
//              truncated to the slot: truncation mod 2^k commutes with all five operations, so this is exact;
//   combine  : warp shuffle, then across the CTA through shared memory; the CTA stores one partial per output into the scratch
//              the context owns and takes the unit's ticket;
//   finish   : the CTA that takes the last ticket of a unit combines the unit's partials in chunk order, writes init (op) P (for
//              Sub, init - P with P a sum) as one scalar per output, and resets the ticket to 0 for the next launch.
// One launch per collect: the tickets are zeroed once when the scratch is allocated and left at 0 by every launch.  None of the
// operations can fail, so there is no error channel.  Offsets are 64-bit throughout.
#include <stdio.h>

#include <algorithm>

#include "kernels.cuh"

namespace mdim {

namespace {

enum SplitOp { SOP_ADD = 0, SOP_MUL, SOP_AND, SOP_OR, SOP_XOR };  // Sub folds with SOP_ADD
constexpr int kSplitThreads = 256, kSplitWarps = kSplitThreads / 32;
constexpr int kSplitCtasPerSm = 3;  // resident CTAs per SM (the register bound below keeps every instantiation free of spills)
constexpr uint64_t kSplitMinChunkBytes = 32 * 1024;  // 128 bytes per thread: four 256-bit loads in flight
constexpr uint64_t kSplitMaxCombine = 32 * 1024;     // COLS: partials one finishing CTA may combine (chunks x columns)

__device__ __forceinline__ uint64_t umin64(uint64_t a, uint64_t b) { return a < b ? a : b; }

template <class S, int OP> __device__ __forceinline__ constexpr S identity() {
    return OP == SOP_MUL ? (S)1 : OP == SOP_AND ? (S)~(S)0 : (S)0;
}
template <int OP, class S> __device__ __forceinline__ S combine(S a, S b) {
    if constexpr (OP == SOP_ADD) return a + b;
    else if constexpr (OP == SOP_MUL) return a * b;
    else if constexpr (OP == SOP_AND) return a & b;
    else if constexpr (OP == SOP_OR) return a | b;
    else return a ^ b;
}
// one source element (its ES bytes in the low bits of x) into a slot
template <class S, int ES> __device__ __forceinline__ S extend(uint64_t x, bool sgn) {
    if constexpr (ES == 1) return (S)(x & 0xffu);  // U8 is the only 1-byte integer: unsigned
    else if constexpr (ES == 4) {
        if constexpr (sizeof(S) == 8) return sgn ? (S)(int64_t)(int32_t)(uint32_t)x : (S)(uint32_t)x;
        else return (S)(uint32_t)x;
    } else return (S)x;  // 8 bytes: all of it, or its low 32 bits
}

__device__ __forceinline__ void ld256(const void* p, uint32_t (&r)[8]) {
    asm volatile("ld.global.nc.L1::no_allocate.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]) : "l"(p));
}
__device__ __forceinline__ void ld128(const void* p, uint32_t (&r)[4]) {
    asm volatile("ld.global.nc.L1::no_allocate.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "l"(p));
}
template <int ES> __device__ __forceinline__ uint64_t ld_elem(const char* p) {
    if constexpr (ES == 1) return *(const uint8_t*)p;
    else if constexpr (ES == 4) return __ldg((const unsigned int*)p);
    else return __ldg((const unsigned long long*)p);
}
// element k of a vector of N 32-bit words
template <int ES, int N> __device__ __forceinline__ uint64_t elem_of(const uint32_t (&r)[N], int k) {
    if constexpr (ES == 1) return (r[k >> 2] >> ((k & 3) * 8)) & 0xffu;
    else if constexpr (ES == 4) return r[k];
    else return (uint64_t)r[2 * k] | ((uint64_t)r[2 * k + 1] << 32);
}

// Fold a whole 32-byte vector into acc.  Bytes: Add sums the vector in 32 bits first (at most 32 x 255); the bit operations
// combine whole words into `wacc`, each byte lane apart, and fold its four lanes into acc once at the end (bytes_into); Mul goes
// element by element.
template <int ES, int OP> constexpr bool kByteLanes = ES == 1 && (OP == SOP_AND || OP == SOP_OR || OP == SOP_XOR);
template <class S, int ES, int OP> __device__ __forceinline__ void fold_vec(S& acc, uint32_t& wacc, const uint32_t (&r)[8], bool sgn) {
    if constexpr (ES == 1 && OP == SOP_ADD) {
        uint32_t t = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) t = __dp4a(r[w], 0x01010101u, t);
        acc += (S)t;
    } else if constexpr (kByteLanes<ES, OP>) {
#pragma unroll
        for (int w = 0; w < 8; ++w) wacc = combine<OP>(wacc, r[w]);
    } else {
#pragma unroll
        for (int k = 0; k < 32 / ES; ++k) acc = combine<OP>(acc, extend<S, ES>(elem_of<ES, 8>(r, k), sgn));
    }
}
template <class S, int OP> __device__ __forceinline__ S bytes_into(S acc, uint32_t t) {
    t = combine<OP>(t, t >> 16);
    t = combine<OP>(t, t >> 8);
    return combine<OP>(acc, (S)(t & 0xffu));
}

template <int OP, class S> __device__ __forceinline__ S warp_combine(S v) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v = combine<OP>(v, (S)__shfl_xor_sync(0xffffffffu, v, d));
    return v;
}

// the whole CTA's values -> thread 0 (the others get garbage)
template <int OP, class S> __device__ __forceinline__ S cta_combine(S v, S* red) {
    v = warp_combine<OP>(v);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    __syncthreads();  // red[] may still be read by a previous call
    if (lane == 0) red[warp] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        v = red[0];
#pragma unroll
        for (int w = 1; w < kSplitWarps; ++w) v = combine<OP>(v, red[w]);
    }
    return v;
}

template <class S> __device__ __forceinline__ void store_out(void* out, uint64_t o, int es, S v) {
    if (es == 1) ((uint8_t*)out)[o] = (uint8_t)v;
    else if (es == 4) ((uint32_t*)out)[o] = (uint32_t)v;
    else ((uint64_t*)out)[o] = (uint64_t)v;
}
template <int OP, class S> __device__ __forceinline__ S finish(const FoldSplitPlan& F, S p) {
    const S init = (S)F.init;
    return F.op == MDIM_SUB ? (S)(init - p) : combine<OP>(init, p);
}

// Store this CTA's partial(s), then take the unit's ticket: true in the CTA that finishes the unit (all its partials visible).
__device__ __forceinline__ bool take_ticket(unsigned int* ticket, uint32_t n_chunks, bool* last) {
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) *last = atomicAdd(ticket, 1u) == n_chunks - 1;
    __syncthreads();
    if (*last) __threadfence();
    return *last;
}

// S: slot type; ES: source bytes; OP: SplitOp; LAYOUT: SPLIT_RUNS / SPLIT_COLS.  grid = units x n_chunks, unit-major.
template <class S, int ES, int OP, int LAYOUT>
__global__ void __launch_bounds__(kSplitThreads, kSplitCtasPerSm)
k_fold_split(const __grid_constant__ FoldSplitPlan F, void* __restrict__ out, unsigned int* __restrict__ tickets, void* __restrict__ partials_v,
             uint64_t chunk, uint32_t n_chunks) {
    pdl_entry(F.nowait != 0);
    S* __restrict__ partials = (S*)partials_v;
    __shared__ S red[kSplitWarps];
    __shared__ bool last;
    const bool sgn = F.src_dtype == MDIM_I32 || F.src_dtype == MDIM_I64;
    const uint64_t unit = blockIdx.x / n_chunks;
    const uint32_t j = blockIdx.x % n_chunks;
    const int tid = threadIdx.x;
    const int out_es = F.dtype == MDIM_U8 ? 1 : (F.dtype == MDIM_I32 || F.dtype == MDIM_U32) ? 4 : 8;
    if constexpr (LAYOUT == SPLIT_RUNS) {
        // ---- one run: elements [k0, k1) of output `unit` -------------------------------------------------------------------
        const uint64_t i0 = unit / F.out_len[1], i1 = unit % F.out_len[1];
        const char* run = (const char*)F.src + (int64_t)(i0 * (uint64_t)F.out_stride[0] + i1 * (uint64_t)F.out_stride[1]) * ES;
        const uint64_t k0 = (uint64_t)j * chunk, k1 = min(F.red, k0 + chunk);
        const char* p = run + k0 * ES;
        const uint64_t n = k1 - k0;
        constexpr int VE = 32 / ES;  // elements per 256-bit vector
        const uint64_t head = min(n, (uint64_t)(((32 - ((uintptr_t)p & 31)) & 31) / ES));  // up to the first 32-byte boundary
        const uint64_t nv = (n - head) / VE;
        const uint64_t tail0 = head + nv * VE;
        S acc = identity<S, OP>();
        uint32_t wacc = identity<uint32_t, OP>();
        if ((uint64_t)tid < head) acc = combine<OP>(acc, extend<S, ES>(ld_elem<ES>(p + (uint64_t)tid * ES), sgn));
        if ((uint64_t)tid < n - tail0) acc = combine<OP>(acc, extend<S, ES>(ld_elem<ES>(p + (tail0 + tid) * ES), sgn));
        const char* body = p + head * ES;
        uint64_t v = tid;
        for (; v + 3 * kSplitThreads < nv; v += 4 * kSplitThreads) {  // four 256-bit loads in flight
            uint32_t r[4][8];
#pragma unroll
            for (int u = 0; u < 4; ++u) ld256(body + (v + (uint64_t)u * kSplitThreads) * 32, r[u]);
#pragma unroll
            for (int u = 0; u < 4; ++u) fold_vec<S, ES, OP>(acc, wacc, r[u], sgn);
        }
        for (; v < nv; v += kSplitThreads) {
            uint32_t r[8];
            ld256(body + v * 32, r);
            fold_vec<S, ES, OP>(acc, wacc, r, sgn);
        }
        if constexpr (kByteLanes<ES, OP>)
            if ((uint64_t)tid < nv) acc = bytes_into<S, OP>(acc, wacc);  // (only lanes that saw a byte: for And, (S)0xff is no identity)
        acc = cta_combine<OP>(acc, red);
        if (tid == 0) partials[unit * n_chunks + j] = acc;
        if (!take_ticket(&tickets[unit], n_chunks, &last)) return;
        S t = identity<S, OP>();
        for (uint32_t c = tid; c < n_chunks; c += kSplitThreads) t = combine<OP>(t, __ldcg(&partials[unit * n_chunks + c]));
        t = cta_combine<OP>(t, red);
        if (tid == 0) {
            store_out(out, unit, out_es, finish<OP>(F, t));
            tickets[unit] = 0;
        }
    } else {
        // ---- rows [r0, r1) of batch `unit`, every column: thread t walks column group g = t % gp, rows r0 + t / gp, step rl --------
        constexpr int W = 16 / ES;  // columns per 128-bit group
        __shared__ S part[kSplitThreads * W];
        const uint64_t cols = F.cols;
        const uint64_t n_groups = (cols + W - 1) / W;
        const int gp = (int)umin64(n_groups, (uint64_t)kSplitThreads);
        const int rl = kSplitThreads / gp;
        const uint64_t r0 = (uint64_t)j * chunk, r1 = min(F.red, r0 + chunk);
        const char* base = (const char*)F.src + unit * (uint64_t)F.batch_stride * ES;
        const uint64_t pitch = (uint64_t)F.pitch * ES;
        const bool vec = (((uintptr_t)base | pitch) & 15) == 0;
        const int gi = tid % gp, ri = tid / gp;
        const bool live = ri < rl;
        for (uint64_t g0 = 0; g0 < n_groups; g0 += (uint64_t)gp) {
            const uint64_t g = g0 + gi;
            S acc[W];
#pragma unroll
            for (int w = 0; w < W; ++w) acc[w] = identity<S, OP>();
            if (live && g < n_groups) {
                const uint64_t c0 = g * W;
                const char* colp = base + c0 * ES;
                if (vec && c0 + W <= cols) {
#pragma unroll 4
                    for (uint64_t r = r0 + ri; r < r1; r += (uint64_t)rl) {
                        uint32_t q[4];
                        ld128(colp + r * pitch, q);
#pragma unroll
                        for (int w = 0; w < W; ++w) acc[w] = combine<OP>(acc[w], extend<S, ES>(elem_of<ES, 4>(q, w), sgn));
                    }
                } else {
                    const int nw = (int)umin64((uint64_t)W, cols - c0);
                    for (uint64_t r = r0 + ri; r < r1; r += (uint64_t)rl)
#pragma unroll
                        for (int w = 0; w < W; ++w)
                            if (w < nw) acc[w] = combine<OP>(acc[w], extend<S, ES>(ld_elem<ES>(colp + r * pitch + (uint64_t)w * ES), sgn));
                }
            }
            __syncthreads();  // part[] is free again
#pragma unroll
            for (int w = 0; w < W; ++w) part[tid * W + w] = acc[w];
            __syncthreads();
            for (int u = tid; u < gp * W; u += kSplitThreads) {  // one column of this pass: combine its row lanes
                const uint64_t c = (g0 + (uint64_t)(u / W)) * W + (uint64_t)(u % W);
                S t = identity<S, OP>();
                for (int k = 0; k < rl; ++k) t = combine<OP>(t, part[(k * gp + u / W) * W + u % W]);
                if (c < cols) partials[(unit * n_chunks + j) * cols + c] = t;
            }
        }
        if (!take_ticket(&tickets[unit], n_chunks, &last)) return;
        for (uint64_t c = tid; c < cols; c += kSplitThreads) {
            S t = identity<S, OP>();
            for (uint32_t k = 0; k < n_chunks; ++k) t = combine<OP>(t, __ldcg(&partials[(unit * n_chunks + k) * cols + c]));
            store_out(out, unit * cols + c, out_es, finish<OP>(F, t));
        }
        if (tid == 0) tickets[unit] = 0;
    }
}

using SplitKernel = void (*)(const FoldSplitPlan, void*, unsigned int*, void*, uint64_t, uint32_t);

template <class S, int ES, int OP>
SplitKernel pick_layout(int layout) {
    return layout == SPLIT_RUNS ? k_fold_split<S, ES, OP, SPLIT_RUNS> : k_fold_split<S, ES, OP, SPLIT_COLS>;
}
template <class S, int ES>
SplitKernel pick_op(int op, int layout) {
    switch (op) {
        case SOP_MUL: return pick_layout<S, ES, SOP_MUL>(layout);
        case SOP_AND: return pick_layout<S, ES, SOP_AND>(layout);
        case SOP_OR: return pick_layout<S, ES, SOP_OR>(layout);
        case SOP_XOR: return pick_layout<S, ES, SOP_XOR>(layout);
        default: return pick_layout<S, ES, SOP_ADD>(layout);
    }
}
template <class S>
SplitKernel pick_src(int es, int op, int layout) {
    return es == 1 ? pick_op<S, 1>(op, layout) : es == 4 ? pick_op<S, 4>(op, layout) : pick_op<S, 8>(op, layout);
}

}  // namespace

struct SplitGeometry {
    uint64_t units;     // RUNS: outputs; COLS: batches.  Each has one ticket.
    uint64_t n_chunks;  // chunks per unit: the grid is units x n_chunks CTAs
    uint64_t chunk;     // RUNS: elements per chunk; COLS: rows per chunk
    uint64_t partials;  // slots of scratch the launch writes (each slot_bytes wide)
};

static SplitGeometry fold_split_geometry(const FoldSplitPlan& F, int sm_count) {
    SplitGeometry G;
    const uint64_t target = (uint64_t)std::max(sm_count, 1) * kSplitCtasPerSm;
    const int es = dtype_size(F.src_dtype);
    if (F.layout == SPLIT_RUNS) {
        G.units = F.n_out;
        uint64_t n = std::min((target + G.units - 1) / G.units, std::max<uint64_t>(1, F.red * es / kSplitMinChunkBytes));
        n = std::max<uint64_t>(n, 1);
        G.chunk = (F.red + n - 1) / n;
        G.chunk = (G.chunk + 31) / 32 * 32;  // chunks start at the same alignment as the run
        G.n_chunks = (F.red + G.chunk - 1) / G.chunk;
        G.partials = G.units * G.n_chunks;
    } else {
        G.units = F.n_batch;
        uint64_t n = std::min((target + G.units - 1) / G.units, std::max<uint64_t>(1, F.red * F.cols * es / kSplitMinChunkBytes));
        n = std::min(n, std::max<uint64_t>(1, kSplitMaxCombine / F.cols));
        n = std::max<uint64_t>(n, 1);
        G.chunk = (F.red + n - 1) / n;
        G.n_chunks = (F.red + G.chunk - 1) / G.chunk;
        G.partials = G.units * G.n_chunks * F.cols;
    }
    return G;
}

size_t fold_split_scratch_bytes(const FoldSplitPlan& F, int sm_count) {
    return kSplitMaxOuts * sizeof(unsigned int) + fold_split_geometry(F, sm_count).partials * 8;
}

static const char* const kOpName[] = {"add", "mul", "and", "or", "xor"};

const char* launch_fold_split(const Plan& p, void* out, bool nowait, cudaStream_t stream, int sm_count, char* scratch) {
    FoldSplitPlan F = p.fs;
    F.nowait = nowait;
    const SplitGeometry G = fold_split_geometry(F, sm_count);
    const int op = F.op == MDIM_MUL ? SOP_MUL : F.op == MDIM_AND ? SOP_AND : F.op == MDIM_OR ? SOP_OR : F.op == MDIM_XOR ? SOP_XOR : SOP_ADD;
    const int es = dtype_size(F.src_dtype);
    const SplitKernel k = F.slot_bytes == 8 ? pick_src<unsigned long long>(es, op, F.layout) : pick_src<unsigned int>(es, op, F.layout);
    const cudaError_t e = launch_pdl(k, dim3((unsigned)(G.units * G.n_chunks)), dim3(kSplitThreads), 0, stream, F, out, (unsigned int*)scratch,
                                     (void*)(scratch + kSplitMaxOuts * sizeof(unsigned int)), (uint64_t)G.chunk, (uint32_t)G.n_chunks);
    if (e != cudaSuccess) return nullptr;
    static thread_local char name[48];
    snprintf(name, sizeof name, "k_fold_split<u%d,src=u%d,%s,%s>", F.slot_bytes * 8, es * 8, kOpName[op], F.layout == SPLIT_RUNS ? "runs" : "cols");
    return name;
}

}  // namespace mdim
