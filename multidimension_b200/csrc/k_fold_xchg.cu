// k_fold_xchg.cu — fold over the SHARDED (outermost) axis as per-rank partial folds combined in RANK ORDER, the all-reduce
// route of SURVEY.md §8(e), as ONE fused compute + exchange kernel per GPU (no NCCL call, no fence, no separate flag).
//
//   P_r[c]  = (((start_r (op) x[r0][c]) (op) x[r0+1][c]) ... )   rank r's own rows, strictly in index order (the reference's add
//             chain, src/view.rs:250-252, 617-622); start_0 = init, start_r = the operator's identity for r > 0
//   out[c]  = ((P_0[c] (op) P_1[c]) (op) P_2[c]) ... (op) P_{N-1}[c]          on EVERY rank, the same order everywhere
//
// Integer and bitwise folds are bit-identical to the reference (the operators are associative); a float sum is reassociated
// once per rank boundary (1e-6 relative, SURVEY.md §8e) but DETERMINISTIC: the blocked order above is what the parity test's
// oracle restates, bit for bit.  An NCCL all-reduce of 1 MiB costs ~60 us at 8 GPUs, most of it launch and protocol latency.
//
// One thread owns 32 bytes of columns and walks down the rank's rows with ROWS independent 256-bit loads in flight (the
// column fold needs no shared memory: every address is known up front).  When its partial values are final it sends them to
// every rank as flag-in-data packets: 16-byte lines {word, epoch, word, epoch} written with ONE volatile vector store into the
// destination's packet area over NVLink (the receiver trusts a line only when both epochs match, so 8-byte store atomicity is
// enough — the same argument NCCL's LL protocol makes).  Two ranks: everybody sends to everybody, polls its own area for both
// ranks' packets of its columns, combines them in rank order and stores 32 bytes of `out` (one hop).  More ranks: every warp's
// columns have an OWNER rank (round robin) that collects the partial values, combines them in rank order and sends the result
// to everybody (two hops, but only 2 (N-1)/N rows per GPU over NVLink instead of N-1).  Areas alternate with the launch parity: a rank can be at most one launch ahead of the slowest
// (it cannot finish launch e+1 without everybody's e+1 packets, which are sent after their launch e has completed).
// Every CTA of the grid is co-resident (grid <= occupancy x SMs), so waiting on peers cannot starve a CTA that has not run.
// Spins are bounded (~2 s): a rank that never arrives becomes MDIM_ERR_NCCL on the others, not a hung GPU.
#include <cuda.h>
#include <string.h>

#include <algorithm>
#include <type_traits>

#include "exec.cuh"
#include "kernels.cuh"

namespace mdim {

namespace {

constexpr int kXThreads = 64;
constexpr unsigned long long kXSpinLimit = 4ull * 1000 * 1000;  // polling rounds (~0.5 us each): ~2 s

__device__ __forceinline__ void st_line(char* p, uint32_t a, uint32_t b, uint32_t flag) {
    asm volatile("st.volatile.global.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(a), "r"(flag), "r"(b), "r"(flag) : "memory");
}
__device__ __forceinline__ uint4 ld_line(const char* p) {
    uint4 v;
    asm volatile("ld.volatile.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
    return v;
}

template <class S> __device__ __forceinline__ void unpack(const uint32_t (&w)[8], S (&v)[32 / sizeof(S)]) {
    if constexpr (sizeof(S) == 4) {
#pragma unroll
        for (int e = 0; e < 8; ++e) v[e] = w[e];
    } else {
#pragma unroll
        for (int e = 0; e < 4; ++e) v[e] = (uint64_t)w[2 * e] | ((uint64_t)w[2 * e + 1] << 32);
    }
}
template <class S> __device__ __forceinline__ void pack(const S (&v)[32 / sizeof(S)], uint32_t (&w)[8]) {
    if constexpr (sizeof(S) == 4) {
#pragma unroll
        for (int e = 0; e < 8; ++e) w[e] = v[e];
    } else {
#pragma unroll
        for (int e = 0; e < 4; ++e) { w[2 * e] = (uint32_t)v[e]; w[2 * e + 1] = (uint32_t)(v[e] >> 32); }
    }
}

// S = slot type (raw bits), DT / OP compile-time (bin_op's switches fold away), ROWS = rows in flight per thread
// EXCHANGE = false: the column walk alone (one GPU, KK_FOLD_COLS): the chain's values ARE the result.
template <class S, int DT, int OP, int ROWS, bool EXCHANGE>
// min blocks per SM = ptxas's register budget (168 / 255): left to itself it settles at ~56 registers with 2-3 loads in flight (4.1 TB/s)
__global__ void __launch_bounds__(kXThreads, EXCHANGE ? 4 : 6) k_fold_xchg(const __grid_constant__ FoldXchgArgs A) {
    constexpr int EPT = 32 / (int)sizeof(S);
    pdl_entry(!EXCHANGE && A.nowait != 0);  // the exchange form always waits for its predecessor in the stream
    const uint64_t gpr = (A.row_bytes + 31) / 32;  // 32-byte column groups per row (the last one may be half: row_bytes % 16 == 0)
    const uint64_t n_groups = EXCHANGE ? gpr : gpr * A.n_batch;  // one-GPU form: n_batch independent (rows x columns) blocks, results back to back
    const uint64_t n_slices = (n_groups + kXThreads - 1) / kXThreads;
    for (uint64_t slice = blockIdx.x; slice < n_slices; slice += gridDim.x) {
        const uint64_t g = slice * kXThreads + threadIdx.x;
        if (g >= n_groups) continue;
        uint64_t gc = g, bi = 0;  // column group within the row, batch index
        if constexpr (!EXCHANGE) {
            if (A.n_batch > 1) { bi = g / gpr; gc = g - bi * gpr; }
        }
        const uint64_t b0 = gc * 32;
        const uint64_t o0 = bi * A.row_bytes + b0;  // byte offset of this thread's results in `out`
        const bool full = b0 + 32 <= A.row_bytes;  // else only the first 16 bytes exist
        const int n_lines = full ? 4 : 2;
        S acc[EPT];
#pragma unroll
        for (int e = 0; e < EPT; ++e) acc[e] = (S)A.start;
        // ---- this rank's rows, in order ------------------------------------------------------------------------------------
        const char* p = (const char*)A.rows + bi * A.batch_pitch_bytes + b0;
        uint64_t r = 0;
        // A rolling window of ROWS loads in flight per thread: row r is folded, then its registers are refilled with row r + ROWS
        // (ROWS = 12 measured best: profiles/r2_fold_cols_rows_in_flight.log).  The alignment test is hoisted out of the loop.
        auto walk = [&](auto wide_tag) {
            constexpr bool WIDE = decltype(wide_tag)::value;
            if (A.n_rows < (uint64_t)ROWS) return;  // short blocks: the row-at-a-time loop below
            uint32_t x[ROWS][8];
#define MDIM_LOAD_ROW(u, row)                                                                                  \
    do {                                                                                                       \
        if constexpr (WIDE) ld256_stream(p + (row) * A.pitch_bytes, x[u]);                                     \
        else { /* rows only 16-byte aligned: two 128-bit loads */                                              \
            ld128_stream(p + (row) * A.pitch_bytes, x[u][0], x[u][1], x[u][2], x[u][3]);                       \
            ld128_stream(p + (row) * A.pitch_bytes + 16, x[u][4], x[u][5], x[u][6], x[u][7]);                  \
        }                                                                                                      \
    } while (0)
#define MDIM_FOLD_ROW(u)                                                                                       \
    do {                                                                                                       \
        S v[EPT];                                                                                              \
        unpack<S>(x[u], v);                                                                                    \
        _Pragma("unroll") for (int e = 0; e < EPT; ++e) { bool arith = false; acc[e] = bin_op<S, false>(DT, OP, DT, acc[e], v[e], arith); } \
    } while (0)
#pragma unroll
            for (int u = 0; u < ROWS; ++u) MDIM_LOAD_ROW(u, (uint64_t)u);
            for (; r + 2 * ROWS <= A.n_rows; r += ROWS) {
#pragma unroll
                for (int u = 0; u < ROWS; ++u) {
                    MDIM_FOLD_ROW(u);
                    MDIM_LOAD_ROW(u, r + ROWS + u);
                }
            }
#pragma unroll
            for (int u = 0; u < ROWS; ++u) MDIM_FOLD_ROW(u);  // the window's last rows
            r += ROWS;
#undef MDIM_LOAD_ROW
#undef MDIM_FOLD_ROW
        };
        if (full) {
            if (A.wide) walk(std::true_type{}); else walk(std::false_type{});
        }
        for (; r < A.n_rows; ++r) {
            uint32_t x[8] = {0, 0, 0, 0, 0, 0, 0, 0};
            ld128_stream(p + r * A.pitch_bytes, x[0], x[1], x[2], x[3]);
            if (full) ld128_stream(p + r * A.pitch_bytes + 16, x[4], x[5], x[6], x[7]);
            S v[EPT];
            unpack<S>(x, v);
#pragma unroll
            for (int e = 0; e < EPT; ++e) { bool arith = false; acc[e] = bin_op<S, false>(DT, OP, DT, acc[e], v[e], arith); }
        }
        // ---- exchange.  Two ranks: everybody sends to everybody and combines (one hop).  More: the columns have an OWNER (warp-
        //      granular, round robin) that collects the partial values, combines them in rank order and sends the result to
        //      everybody: two hops, but 2 (N-1)/N of a row per GPU over NVLink instead of N-1 rows ---------------------------------
        if constexpr (!EXCHANGE) {
            uint32_t ow[8];
            pack<S>(acc, ow);
            st128((char*)A.out + o0, ow[0], ow[1], ow[2], ow[3], false);
            if (full) st128((char*)A.out + o0 + 16, ow[4], ow[5], ow[6], ow[7], false);
            continue;
        }
        uint32_t w[8];
        pack<S>(acc, w);
        const bool one_shot = A.one_shot != 0;
        const int owner = one_shot ? A.rank : (int)((g >> 5) % (uint64_t)A.world);
        const uint64_t slot_base = (uint64_t)A.slot * (A.world + 1) * A.cap_words * 8;   // [slot][source rank 0..N-1, then the results][cap_words x 8 B]
        {
            const uint64_t line_off = slot_base + (uint64_t)A.rank * A.cap_words * 8 + (g >> 5) * 2048 + (g & 31) * 16;  // a warp's lines: [line 0..3][lane], so every store instruction writes 512 contiguous bytes
            for (int k = 0; k < (one_shot ? A.world : 1); ++k) {  // nearest neighbour first, own area last (one code path)
                int d = one_shot ? A.rank + 1 + k : owner;
                if (d >= A.world) d -= A.world;
                char* dst = A.area[d] + line_off;
#pragma unroll
                for (int l = 0; l < 4; ++l)
                    if (l < n_lines) st_line(dst + 512 * l, w[2 * l], w[2 * l + 1], A.epoch);
            }
        }
        const char* mine = A.area[A.rank] + slot_base + (g >> 5) * 2048 + (g & 31) * 16;  // a warp's lines: [line 0..3][lane], so every store instruction writes 512 contiguous bytes
        S tot[EPT];
        bool lost = false;
        if (owner == A.rank) {
            // every rank's partial values of these columns.  Each round re-reads ALL the lines that are not there yet with independent
            // loads (one memory latency per round; polling line after line costs one latency PER LINE: 32 lines at 8 ranks = 20+ us)
            uint4 L[MDIM_MAX_PEERS][4];
#pragma unroll
            for (int q = 0; q < MDIM_MAX_PEERS; ++q) {
#pragma unroll
                for (int l = 0; l < 4; ++l) L[q][l] = make_uint4(0, ~A.epoch, 0, ~A.epoch);
            }
            for (unsigned long long spins = 0;; ++spins) {
#pragma unroll
                for (int q = 0; q < MDIM_MAX_PEERS; ++q)
                    if (q < A.world) {
#pragma unroll
                        for (int l = 0; l < 4; ++l)
                            if (l < n_lines && (L[q][l].y != A.epoch || L[q][l].w != A.epoch)) L[q][l] = ld_line(mine + (uint64_t)q * A.cap_words * 8 + 512 * l);
                    }
                bool pending = false;
#pragma unroll
                for (int q = 0; q < MDIM_MAX_PEERS; ++q)
                    if (q < A.world) {
#pragma unroll
                        for (int l = 0; l < 4; ++l)
                            if (l < n_lines && (L[q][l].y != A.epoch || L[q][l].w != A.epoch)) pending = true;
                    }
                if (!pending) break;
                if (spins > kXSpinLimit) { lost = true; break; }
                if (spins > 4) __nanosleep(64);
            }
            if (lost) { atomicExch(A.error, 1u); continue; }
            // combine in rank order
#pragma unroll
            for (int q = 0; q < MDIM_MAX_PEERS; ++q)
                if (q < A.world) {
                    uint32_t pw[8] = {L[q][0].x, L[q][0].z, L[q][1].x, L[q][1].z, 0, 0, 0, 0};
                    if (full) { pw[4] = L[q][2].x; pw[5] = L[q][2].z; pw[6] = L[q][3].x; pw[7] = L[q][3].z; }
                    S v[EPT];
                    unpack<S>(pw, v);
#pragma unroll
                    for (int e = 0; e < EPT; ++e) {
                        bool arith = false;
                        tot[e] = q == 0 ? v[e] : bin_op<S, false>(DT, OP, DT, tot[e], v[e], arith);
                    }
                }
            if (!one_shot) {  // the result goes to everybody else's result area
                uint32_t rw[8];
                pack<S>(tot, rw);
                const uint64_t res_off = slot_base + (uint64_t)A.world * A.cap_words * 8 + (g >> 5) * 2048 + (g & 31) * 16;  // a warp's lines: [line 0..3][lane], so every store instruction writes 512 contiguous bytes
                for (int k = 0; k + 1 < A.world; ++k) {
                    int d = A.rank + 1 + k;
                    if (d >= A.world) d -= A.world;
                    char* dst = A.area[d] + res_off;
#pragma unroll
                    for (int l = 0; l < 4; ++l)
                        if (l < n_lines) st_line(dst + 512 * l, rw[2 * l], rw[2 * l + 1], A.epoch);
                }
            }
        } else {  // the owner's result
            uint32_t pw[8] = {0, 0, 0, 0, 0, 0, 0, 0};
            uint4 R[4];
#pragma unroll
            for (int l = 0; l < 4; ++l) R[l] = make_uint4(0, ~A.epoch, 0, ~A.epoch);
            for (unsigned long long spins = 0;; ++spins) {
#pragma unroll
                for (int l = 0; l < 4; ++l)
                    if (l < n_lines && (R[l].y != A.epoch || R[l].w != A.epoch)) R[l] = ld_line(mine + (uint64_t)A.world * A.cap_words * 8 + 512 * l);
                bool pending = false;
#pragma unroll
                for (int l = 0; l < 4; ++l)
                    if (l < n_lines && (R[l].y != A.epoch || R[l].w != A.epoch)) pending = true;
                if (!pending) break;
                if (spins > kXSpinLimit) { lost = true; break; }
                if (spins > 4) __nanosleep(64);
            }
#pragma unroll
            for (int l = 0; l < 4; ++l)
                if (l < n_lines) { pw[2 * l] = R[l].x; pw[2 * l + 1] = R[l].z; }
            if (lost) { atomicExch(A.error, 1u); continue; }
            unpack<S>(pw, tot);
        }
        uint32_t ow[8];
        pack<S>(tot, ow);
        st128((char*)A.out + b0, ow[0], ow[1], ow[2], ow[3], false);
        if (full) st128((char*)A.out + b0 + 16, ow[4], ow[5], ow[6], ow[7], false);
    }
}

using XchgKernel = void (*)(const FoldXchgArgs);

template <class S, int DT, int kXRows, bool EXCHANGE> XchgKernel pick_op(int op) {
    constexpr bool is_float = DT == MDIM_F32 || DT == MDIM_F64;
    switch (op) {
        case MDIM_ADD: return k_fold_xchg<S, DT, MDIM_ADD, kXRows, EXCHANGE>;
        case MDIM_MUL: return k_fold_xchg<S, DT, MDIM_MUL, kXRows, EXCHANGE>;
        default: break;
    }
    if constexpr (!EXCHANGE) {  // no identity: a chain, but nothing to combine partial results with
        if (op == MDIM_SUB) return k_fold_xchg<S, DT, MDIM_SUB, kXRows, EXCHANGE>;
    }
    if constexpr (!is_float) {
        switch (op) {
            case MDIM_AND: return k_fold_xchg<S, DT, MDIM_AND, kXRows, EXCHANGE>;
            case MDIM_OR: return k_fold_xchg<S, DT, MDIM_OR, kXRows, EXCHANGE>;
            case MDIM_XOR: return k_fold_xchg<S, DT, MDIM_XOR, kXRows, EXCHANGE>;
            default: break;
        }
    }
    return nullptr;
}

template <bool EXCHANGE> XchgKernel pick_kernel(int dtype, int op) {
    switch (dtype) {  // wrapping integer + - * and the bitwise operators do not care about the sign: one instantiation per width
        case MDIM_F32: return pick_op<uint32_t, MDIM_F32, 12, EXCHANGE>(op);  // 12 rows in flight per thread: 3 / 4 / 6 / 8 / 12 / 16 -> 4.5 / 5.4 / 6.5 / 7.0 / 7.25 / 6.0 TB/s (profiles/)
        case MDIM_I32: case MDIM_U32: return pick_op<uint32_t, MDIM_U32, 12, EXCHANGE>(op);
        case MDIM_F64: return pick_op<uint64_t, MDIM_F64, 12, EXCHANGE>(op);
        case MDIM_I64: case MDIM_U64: return pick_op<uint64_t, MDIM_U64, 12, EXCHANGE>(op);
        default: return nullptr;
    }
}

}  // namespace

// -> 0 ok; -1 when the rows are not 16-byte aligned or the operator has no identity; else a cudaError
int launch_fold_xchg(const FoldXchgArgs& A, int dtype, int op, int sm_count, cudaStream_t stream) {
    if (((uintptr_t)A.rows & 15) || (A.pitch_bytes & 15) || (A.row_bytes & 15) || ((uintptr_t)A.out & 15) || !A.n_rows || !A.row_bytes) return -1;
    FoldXchgArgs B = A;
    // two ranks: one hop; more: owners (two hops, 2 (N-1)/N rows per GPU over NVLink instead of N-1)
    B.one_shot = A.world <= 2;
    B.wide = !(((uintptr_t)A.rows & 31) || (A.pitch_bytes & 31));
    XchgKernel fn = pick_kernel<true>(dtype, op);
    if (!fn) return -1;
    static XchgKernel known_fn[32];
    static int known_per_sm[32], n_known = 0;  // the context is single-threaded (mdim.h)
    int per_sm = 0;
    cudaError_t e = cudaSuccess;
    for (int i = 0; i < n_known; ++i)
        if (known_fn[i] == fn) per_sm = known_per_sm[i];
    if (!per_sm) {
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, kXThreads, 0);
        if (e != cudaSuccess) return (int)e;
        if (per_sm < 1) return -1;
        if (n_known < 32) { known_fn[n_known] = fn; known_per_sm[n_known++] = per_sm; }
    }
    const uint64_t n_groups = (A.row_bytes + 31) / 32, n_slices = (n_groups + kXThreads - 1) / kXThreads;
    const int grid = (int)std::min<uint64_t>(n_slices, (uint64_t)per_sm * (uint64_t)sm_count);
    e = launch_pdl(fn, dim3(grid), dim3(kXThreads), 0, stream, B);
    return e == cudaSuccess ? 0 : (int)e;
}

// The column walk on one GPU (KK_FOLD_COLS, planned in plan.cpp): no packets, no co-residency requirement.
const char* launch_fold_cols(const Plan& p, void* out, bool nowait, cudaStream_t stream, int) {
    const FoldColsPlan& C = p.fc;
    XchgKernel fn = pick_kernel<false>(C.dtype, C.op);
    if (!fn) return nullptr;
    FoldXchgArgs A;
    memset(&A, 0, sizeof A);
    A.n_rows = C.n_rows; A.row_bytes = C.row_bytes; A.pitch_bytes = C.pitch_bytes;
    A.world = 1; A.start = C.init; A.rows = C.src; A.out = out; A.nowait = nowait;
    A.n_batch = C.n_batch ? C.n_batch : 1; A.batch_pitch_bytes = C.batch_pitch_bytes;
    A.wide = !(((uintptr_t)C.src & 31) || (C.pitch_bytes & 31) || (A.n_batch > 1 && (C.batch_pitch_bytes & 31)));
    const uint64_t n_groups = (C.row_bytes + 31) / 32 * A.n_batch, n_slices = (n_groups + kXThreads - 1) / kXThreads;
    const int grid = (int)std::min<uint64_t>(n_slices, 1u << 30);
    return launch_pdl(fn, dim3(grid), dim3(kXThreads), 0, stream, A) == cudaSuccess ? "k_fold_cols" : nullptr;
}

}  // namespace mdim
