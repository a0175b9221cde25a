// k_fold.cu — K4: last-axis fold in the reference's SEQUENTIAL order, optionally fused with a
// broadcast epilogue, one HBM pass (sm_100a; TMA bulk copies + mbarrier pipeline).
//
// The reference has no reduce API; a fold over an axis is spelled
//     a.rows::<I,J>().map(|row| { let mut s = init; row.each(|x| s = s (op) x); s })
// (src/view.rs:617-622 rows, :1341 Rows::at, :250-252 each → src/int.rs:23-25), i.e. a strictly
// left-to-right accumulation in index order.  For f32 that order IS the parity contract
// (SURVEY.md fact 3 / §7 hard part 6), so this kernel never uses a shuffle tree: it parallelises
// ACROSS rows and keeps each row's add chain serial, which is bit-exact with the reference.
//
// Layout / schedule.  Rows are contiguous (n_rows x row_len 4-byte elements).  Each WARP owns a
// ring of STAGES shared-memory tiles of 32 rows (pitch = row_len + pad words, pitch/4 odd).  Lane 0
// issues one `cp.async.bulk` (TMA, 1-D) per row into the tile and arms the tile's mbarrier with
// the byte count; while that lands, the warp works on the previous tile:
//   sum      : lane l walks row l with 16-byte shared loads (conflict-free because pitch/4 is odd)
//              and a dependent chain of row_len adds — 32 independent chains per warp;
//   epilogue : (fused form, BASELINE config 4) the whole warp re-reads the tile row by row,
//              applies  x (eop) g(fold[row])  with the row's fold broadcast by shuffle, and writes
//              coalesced 16-byte streaming stores; or (fold-only form) lane l stores fold[l].
// The input is read from HBM exactly once for fold + broadcast-subtract: algorithmic bytes
// = 2 x n_rows x row_len x 4 (SURVEY.md §8d C4c).  No block-level barrier anywhere: warps only use
// their own mbarriers and __syncwarp.
#include "kernels.cuh"

namespace mdim {

namespace {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t"
        "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// 1-D TMA: global -> this CTA's shared memory, completion counted in bytes on `bar`
__device__ __forceinline__ void tma_load_1d(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

__device__ __forceinline__ float apply_f32(int op, float a, float b) {
    switch (op) {
        case MDIM_ADD: return __fadd_rn(a, b);
        case MDIM_SUB: return __fsub_rn(a, b);
        case MDIM_MUL: return __fmul_rn(a, b);
        case MDIM_DIV: return __fdiv_rn(a, b);
        case MDIM_REM: return fmodf(a, b);
    }
    return a;
}

// generic element op through the shared value semantics (ints wrap; errors cannot be reported from
// here, so the planner only routes float ops and non-trapping integer ops to this kernel)
__device__ __forceinline__ uint32_t apply_any(int dtype, int op, uint32_t a, uint32_t b) {
    if (dtype == MDIM_F32) return __float_as_uint(apply_f32(op, __uint_as_float(a), __uint_as_float(b)));
    bool arith = false;
    return bin_op<uint32_t>(dtype, op, dtype, a, b, arith);
}

constexpr int kRowsPerTile = 32;  // one row per lane
constexpr int kBarBytes = 512;     // mbarriers ahead of the tiles: 8 warps x up to 8 stages x 8 B

// Work is cut into ITEMS: (block of 32 rows) x (chunk of `ch` columns), column chunks of one row block
// consecutive, so a lane's accumulator simply carries over from chunk to chunk.  Each warp owns a ring
// of `stages` shared-memory tiles [32][ch] (dense, no padding) and walks its items in order:
//   fill   : when ch == row_len the 32 rows are one contiguous run of global memory — ONE
//            cp.async.bulk (TMA) of up to 64 KB issued by lane 0; otherwise each lane issues the bulk copy
//            of its own row piece (32 copies in flight at once).  Completion is counted in bytes on
//            the tile's mbarrier.
//   fold   : lane l walks row l with 16-byte shared loads and a dependent chain of adds — strictly left
//            to right.  Lanes start `skew * (l & 7)` steps late, which makes the 8 lanes of each
//            quarter-warp hit 8 different 16-byte bank groups of the dense tile (no padding needed).
//   finish : after the last chunk, either lane l stores fold[l] (fold only), or (ch == row_len) the warp
//            re-reads the tile row by row and writes  x (eop) g(fold[row])  with coalesced 16-byte
//            streaming stores (BASELINE config 4: the input is read from HBM exactly once).
// FAST = f32 with fold op ADD and epilogue op SUB (or none): the shape of BASELINE config 4.
template <bool FAST>
__global__ void __launch_bounds__(kFoldThreads)
k_fold_rows(const __grid_constant__ FoldRowsPlan R, void* __restrict__ out_v, int n_warps, int stages, int ch, int skew, uint32_t q4_mul,
            uint32_t q4_shr) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    pdl_entry(R.nowait != 0);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp >= n_warps) return;
    const uint32_t tile_words = (uint32_t)kRowsPerTile * (uint32_t)ch;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw);  // [n_warps][stages], 8 B each (<= kBarBytes)
    uint32_t* tiles = reinterpret_cast<uint32_t*>(smem_raw + kBarBytes) + (size_t)warp * stages * tile_words;
    uint64_t* my_bars = bars + warp * stages;

    const uint32_t row_len = R.row_len, row_bytes = row_len * 4u;
    const uint32_t n_chunks = (row_len + (uint32_t)ch - 1) / (uint32_t)ch;
    const bool dense = n_chunks == 1;
    const char* __restrict__ src = (const char*)R.src + R.src_offset * 4;
    const uint64_t n_blocks = (R.n_rows + kRowsPerTile - 1) / kRowsPerTile;
    const uint64_t total_warps = (uint64_t)gridDim.x * n_warps;
    const uint64_t gw = (uint64_t)blockIdx.x * n_warps + warp;
    // this warp's row blocks: gw, gw + total_warps, ...; its items: those blocks x n_chunks, in order
    const uint64_t my_blocks = gw < n_blocks ? (n_blocks - gw + total_warps - 1) / total_warps : 0;
    const uint64_t my_items = my_blocks * n_chunks;

    auto fill = [&](uint64_t item) {  // whole warp
        const int s = (int)(item % (uint64_t)stages);
        const uint64_t blk = gw + (item / n_chunks) * total_warps;
        const uint32_t c = (uint32_t)(item % n_chunks);
        const uint64_t row0 = blk * kRowsPerTile;
        const uint32_t nrows = (uint32_t)min((uint64_t)kRowsPerTile, R.n_rows - row0);
        const uint32_t cols = min((uint32_t)ch, row_len - c * (uint32_t)ch);
        uint32_t* dst = tiles + (size_t)s * tile_words;
        if (lane == 0) mbar_expect_tx(&my_bars[s], nrows * cols * 4u);
        __syncwarp();
        if (dense) {
            if (lane == 0) tma_load_1d(dst, src + row0 * (uint64_t)row_bytes, nrows * row_bytes, &my_bars[s]);
        } else if ((uint32_t)lane < nrows) {
            tma_load_1d(dst + lane * ch, src + (row0 + lane) * (uint64_t)row_bytes + (uint64_t)c * ch * 4u, cols * 4u, &my_bars[s]);
        }
    };

    if (lane == 0) {
        for (int s = 0; s < stages; ++s) mbar_init(&my_bars[s], 1);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // make the inits visible to the TMA unit
    }
    __syncwarp();
    for (uint64_t it = 0; it < (uint64_t)stages && it < my_items; ++it) fill(it);

    const int my_skew = skew * (lane & 7);
    uint32_t fold = (uint32_t)R.init;
    for (uint64_t it = 0; it < my_items; ++it) {
        const int s = (int)(it % (uint64_t)stages);
        const uint32_t parity = (uint32_t)((it / (uint64_t)stages) & 1u);
        const uint64_t blk = gw + (it / n_chunks) * total_warps;
        const uint32_t c = (uint32_t)(it % n_chunks);
        const uint64_t row0 = blk * kRowsPerTile;
        const uint32_t nrows = (uint32_t)min((uint64_t)kRowsPerTile, R.n_rows - row0);
        const uint32_t cols = min((uint32_t)ch, row_len - c * (uint32_t)ch);
        const int q4 = (int)(cols >> 2);
        uint32_t* tile_s = tiles + (size_t)s * tile_words;
        if (c == 0) fold = (uint32_t)R.init;
        mbar_wait(&my_bars[s], parity);

        // ---- fold: lane l folds row l, strictly left to right ------------------------------------------
        {
            const uint4* rowp = reinterpret_cast<const uint4*>(tile_s + lane * ch);
            const bool live = (uint32_t)lane < nrows;
            const int steps = q4 + 7 * skew;
            if constexpr (FAST) {
                float acc = __uint_as_float(fold);
                for (int t0 = 0; t0 < steps; t0 += 4) {  // 4 shared loads in flight ahead of the dependent add chain
                    uint4 v[4];
                    bool ok[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int k = t0 + j - my_skew;
                        ok[j] = live && k >= 0 && k < q4;
                        if (ok[j]) v[j] = rowp[k];
                    }
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        if (ok[j]) {  // never add a padding zero: -0.0 + 0.0 would flip the sign
                            acc = __fadd_rn(acc, __uint_as_float(v[j].x));
                            acc = __fadd_rn(acc, __uint_as_float(v[j].y));
                            acc = __fadd_rn(acc, __uint_as_float(v[j].z));
                            acc = __fadd_rn(acc, __uint_as_float(v[j].w));
                        }
                    }
                }
                fold = __float_as_uint(acc);
            } else {
                for (int t = 0; t < steps; ++t) {
                    const int k = t - my_skew;
                    if (live && k >= 0 && k < q4) {
                        const uint4 v = rowp[k];
                        fold = apply_any(R.dtype, R.op, fold, v.x);
                        fold = apply_any(R.dtype, R.op, fold, v.y);
                        fold = apply_any(R.dtype, R.op, fold, v.z);
                        fold = apply_any(R.dtype, R.op, fold, v.w);
                    }
                }
            }
        }

        // ---- finish ---------------------------------------------------------------------------------------
        if (c + 1 == n_chunks) {
            if (R.epilogue == 0) {
                // fold only: one value per row, coalesced 128 B per warp
                if ((uint32_t)lane < nrows) reinterpret_cast<uint32_t*>(out_v)[row0 + lane] = fold;
            } else {
                // out[row][k] = src[row][k] (eop) g[row]; Zip over (I, J) x (I, ()) — the () axis of the
                // fold is expanded by Broadcast (src/broadcast.rs:54-60), i.e. g is constant along k
                uint32_t g = fold;
                if (R.has_post) g = apply_any(R.dtype, R.post_op, g, (uint32_t)R.post_imm);
                // The dense tile [nrows][row_len] is also ONE contiguous run of the output: walk it flat, 512
                // bytes per warp instruction, each lane fetching its row's g by shuffle.
                char* __restrict__ obase = (char*)out_v + row0 * (uint64_t)row_bytes;
                const uint4* tp = reinterpret_cast<const uint4*>(tile_s);
                const uint32_t n16 = nrows * (uint32_t)q4;
#pragma unroll 4
                for (uint32_t i0 = 0; i0 < n16; i0 += 32) {
                    const uint32_t i = i0 + lane;
                    const bool in = i < n16;
                    const uint32_t row = __umulhi(in ? i : 0u, q4_mul) >> q4_shr;  // i / q4
                    const uint32_t gr = __shfl_sync(0xffffffffu, g, (int)row);
                    if (in) {
                        uint4 v = tp[i];
                        if constexpr (FAST) {
                            const float m = __uint_as_float(gr);
                            v.x = __float_as_uint(__fsub_rn(__uint_as_float(v.x), m));
                            v.y = __float_as_uint(__fsub_rn(__uint_as_float(v.y), m));
                            v.z = __float_as_uint(__fsub_rn(__uint_as_float(v.z), m));
                            v.w = __float_as_uint(__fsub_rn(__uint_as_float(v.w), m));
                        } else {
                            v.x = apply_any(R.dtype, R.eop, v.x, gr);
                            v.y = apply_any(R.dtype, R.eop, v.y, gr);
                            v.z = apply_any(R.dtype, R.eop, v.z, gr);
                            v.w = apply_any(R.dtype, R.eop, v.w, gr);
                        }
                        asm volatile("st.global.cs.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(obase + (size_t)i * 16u), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
                    }
                }
            }
        }
        __syncwarp();  // every lane is done reading this stage before it is refilled
        if (it + (uint64_t)stages < my_items) fill(it + (uint64_t)stages);
    }
}


// ---- register-resident form (row_len = 32 * L elements, L a power of two <= 32) ------------------------
// No shared memory, no TMA, no barrier: the massively threaded, one-trip-per-warp shape that the plain
// streaming kernels use.  L lanes share a row; lane j holds the 16-byte chunks j, L + j, 2L + j, ... (so every
// load and store instruction of the warp covers whole 16L-byte runs of 32/L adjacent rows), and the fold is
// passed around the L lanes in INDEX ORDER — chunk c is added by lane c % L, then the running value is
// broadcast to the group by shuffle — so the add chain is exactly the reference's sequential one.
// The row stays in registers for the fused epilogue: the input is read from HBM once.
template <int L, bool FAST>
__global__ void __launch_bounds__(256) k_fold_regs(const __grid_constant__ FoldRowsPlan R, void* __restrict__ out_v) {
    constexpr int M = 8;         // 16-byte chunks per lane
    constexpr int RPW = 32 / L;  // rows per warp
    pdl_entry(R.nowait != 0);
    const int lane = threadIdx.x & 31, j = lane % L, grp = lane / L;
    const uint64_t warp = (uint64_t)blockIdx.x * (256 / 32) + (threadIdx.x >> 5);
    const uint64_t row = warp * RPW + grp;
    const bool live = row < R.n_rows;
    const uint64_t row_bytes = (uint64_t)R.row_len * 4u;
    const char* __restrict__ src = (const char*)R.src + R.src_offset * 4 + row * row_bytes;
    uint4 v[M];
#pragma unroll
    for (int m = 0; m < M; ++m) {
        v[m] = make_uint4(0, 0, 0, 0);
        if (live)
            asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                         : "=r"(v[m].x), "=r"(v[m].y), "=r"(v[m].z), "=r"(v[m].w) : "l"(src + (size_t)(m * L + j) * 16u));
    }
    uint32_t acc = (uint32_t)R.init;
#pragma unroll
    for (int m = 0; m < M; ++m) {
#pragma unroll
        for (int jj = 0; jj < L; ++jj) {
            if (j == jj) {  // chunk m * L + jj: strictly after chunk m * L + jj - 1
                if constexpr (FAST) {
                    float a = __uint_as_float(acc);
                    a = __fadd_rn(a, __uint_as_float(v[m].x));
                    a = __fadd_rn(a, __uint_as_float(v[m].y));
                    a = __fadd_rn(a, __uint_as_float(v[m].z));
                    a = __fadd_rn(a, __uint_as_float(v[m].w));
                    acc = __float_as_uint(a);
                } else {
                    acc = apply_any(R.dtype, R.op, acc, v[m].x);
                    acc = apply_any(R.dtype, R.op, acc, v[m].y);
                    acc = apply_any(R.dtype, R.op, acc, v[m].z);
                    acc = apply_any(R.dtype, R.op, acc, v[m].w);
                }
            }
            if constexpr (L > 1) acc = __shfl_sync(0xffffffffu, acc, grp * L + jj);
        }
    }
    // every lane of the group now holds the row's fold
    if (R.epilogue == 0) {
        if (live && j == 0) reinterpret_cast<uint32_t*>(out_v)[row] = acc;
        return;
    }
    uint32_t g = acc;
    if (R.has_post) g = apply_any(R.dtype, R.post_op, g, (uint32_t)R.post_imm);
    char* __restrict__ orow = (char*)out_v + row * row_bytes;
#pragma unroll
    for (int m = 0; m < M; ++m) {
        uint4 x = v[m];
        if constexpr (FAST) {
            const float mm = __uint_as_float(g);
            x.x = __float_as_uint(__fsub_rn(__uint_as_float(x.x), mm));
            x.y = __float_as_uint(__fsub_rn(__uint_as_float(x.y), mm));
            x.z = __float_as_uint(__fsub_rn(__uint_as_float(x.z), mm));
            x.w = __float_as_uint(__fsub_rn(__uint_as_float(x.w), mm));
        } else {
            x.x = apply_any(R.dtype, R.eop, x.x, g);
            x.y = apply_any(R.dtype, R.eop, x.y, g);
            x.z = apply_any(R.dtype, R.eop, x.z, g);
            x.w = apply_any(R.dtype, R.eop, x.w, g);
        }
        if (live) asm volatile("st.global.cs.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(orow + (size_t)(m * L + j) * 16u), "r"(x.x), "r"(x.y), "r"(x.z), "r"(x.w) : "memory");
    }
}

// -> false: the register form does not take this row length or row count (*e: the launch's result otherwise)
template <bool FAST> static bool launch_regs(const FoldRowsPlan& R, void* out, cudaStream_t stream, cudaError_t* e) {
    const uint32_t L = R.row_len / 32;  // row_len = 4 elements x 8 chunks x L lanes
    if (R.row_len % 32 != 0 || L < 1 || L > 32 || (L & (L - 1)) != 0) return false;
    const uint64_t warps = (R.n_rows + (32 / L) - 1) / (32 / L);
    const uint64_t ctas = (warps + 7) / 8;
    if (ctas > 0x7fffffffull) return false;
    const dim3 grid((unsigned)ctas), block(256);
    switch (L) {
        case 1: *e = launch_pdl(k_fold_regs<1, FAST>, grid, block, 0, stream, R, out); break;
        case 2: *e = launch_pdl(k_fold_regs<2, FAST>, grid, block, 0, stream, R, out); break;
        case 4: *e = launch_pdl(k_fold_regs<4, FAST>, grid, block, 0, stream, R, out); break;
        case 8: *e = launch_pdl(k_fold_regs<8, FAST>, grid, block, 0, stream, R, out); break;
        case 16: *e = launch_pdl(k_fold_regs<16, FAST>, grid, block, 0, stream, R, out); break;
        default: *e = launch_pdl(k_fold_regs<32, FAST>, grid, block, 0, stream, R, out); break;
    }
    return true;
}

}  // namespace

const char* launch_fold_rows(const Plan& p, void* out, bool nowait, cudaStream_t stream, int sm_count) {
    FoldRowsPlan R = p.fr;
    R.nowait = nowait;
    // column chunk: the whole row when a 32-row tile of it fits 64 KB (and always for the fused form,
    // which needs the whole row resident); else 256 columns per item
    int ch = (int)R.row_len;
    if (R.epilogue == 0 && R.row_len > 512) ch = 256;
    const size_t tile_bytes = (size_t)kRowsPerTile * ch * 4;
    const size_t budget = 227 * 1024 - kBarBytes;  // the whole opt-in shared memory of an SM: 7 tiles of 32 KB
    int max_tiles = (int)(budget / tile_bytes);
    if (max_tiles < 1) max_tiles = 1;
    // Measured on B200 (profiles/): warps hide each other's latency better than stages do — six warps with
    // one tile each beat three warps with two — so fill the warps first, then deepen the rings.
    const int n_warps = std::min(kFoldThreads / 32, max_tiles);
    const int stages = std::min(4, max_tiles / n_warps);
    const size_t smem = kBarBytes + (size_t)n_warps * stages * tile_bytes;
    const uint64_t n_blocks = (R.n_rows + kRowsPerTile - 1) / kRowsPerTile;
    // Not one resident CTA per SM but up to 16 queued per SM (each warp then folds ~2 tiles): the hardware scheduler
    // evens out the tail.  Measured on B200, config 4a: 6 724 GB/s (x1) -> 6 892 (x4) -> 7 047 (x16) -> 6 983 (x64);
    // a pure read stream reaches 7 570 (scripts/probe/read_bw.cu).
    int grid = (int)std::min<uint64_t>((n_blocks + n_warps - 1) / n_warps, (uint64_t)sm_count * 16);
    if (grid < 1) grid = 1;
    // bank-conflict-free skew needs the dense row pitch to be a multiple of 8 sixteen-byte chunks
    const int skew = ((ch / 4) % 8 == 0) ? 1 : 0;
    const bool fast = R.dtype == MDIM_F32 && R.op == MDIM_ADD && (R.epilogue == 0 || (R.eop == MDIM_SUB));
    // Measured on B200 (profiles/): the register form wins for the fused epilogue (config 4c: 6.27 vs 5.74 TB/s),
    // the TMA / shared-memory form for the fold alone (config 4a: 6.28 vs 5.66 TB/s).
    static const int mode = [] { const char* e = getenv("MDIM_FOLD_MODE"); return e ? atoi(e) : 0; }();  // 1 = always smem, 2 = always registers
    const bool want_regs = mode == 2 || (mode == 0 && R.epilogue != 0);
    cudaError_t e = cudaSuccess;
    if (want_regs && (fast ? launch_regs<true>(R, out, stream, &e) : launch_regs<false>(R, out, stream, &e))) return e == cudaSuccess ? "k_fold_regs" : nullptr;
    // i / q4 for the flat epilogue walk: umulhi(i, mul) >> shr, exact for i < 2^31 (q4 >= 2 here)
    uint32_t q4 = (uint32_t)ch / 4, lg = 0;
    while ((1u << lg) < q4) ++lg;
    const uint32_t q4_shr = lg - 1 + (q4 == 1 ? 1 : 0);
    const uint32_t q4_mul = (uint32_t)(((1ull << (31 + lg)) + q4 - 1) / q4);
    auto go = [&](auto kern) {
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        return launch_pdl(kern, dim3(grid), dim3(kFoldThreads), smem, stream, R, out, n_warps, stages, ch, skew, q4_mul, q4_shr);
    };
    e = fast ? go(k_fold_rows<true>) : go(k_fold_rows<false>);
    return e == cudaSuccess ? "k_fold_rows" : nullptr;
}

}  // namespace mdim
