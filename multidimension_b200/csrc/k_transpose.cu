// k_transpose.cu — K2: batched tiled transpose of one leaf through swizzled shared memory (sm_100a).
//
// Serves `Transpose<V,I,X,Y,J>` (reference src/view.rs:586-592, 1266-1294) — and any other pure
// index permutation of a single Array — whenever the axis that is contiguous in the SOURCE
// (call it A) is not the output's innermost axis (call it B).  Everything else is batch.
//
//   out[batch, a, b]  (b has out stride 1)   =   src[batch', b, a]  (a has src stride 1)
//
// One CTA moves one tile of TB = 64 B-rows x TAC = 16 chunks (16 bytes each) of A, i.e. 64x64 4-byte or 64x32 8-byte
// elements, 16 KB of shared memory, both global directions 128-bit and coalesced:
//   load : each thread reads 16 B along A (a warp covers 2 source rows x 256 B) and writes them
//          with ONE 16-byte shared store at row b, chunk (a_chunk ^ swz(b));
//   store: each thread assembles 16 B along B from CH scalar shared loads (one per source row) and
//          writes one 16-byte global store; a warp covers 4 output rows x 128 B.
// Swizzle swz(b) = (b / CH) & 7 makes both shared phases bank-conflict-free: a quarter warp's
// 16-byte stores hit 8 distinct chunks, and in the read phase the 32 lanes (8 b-groups x 4 a's)
// hit 8 distinct chunks x 4 distinct words.
// The grid is NOT persistent (up to 128 CTAs per SM are launched, each takes 1-4 tiles): the hardware scheduler
// then balances the tail, worth +11 % at 16384^2 and +8 % at 4096^2 over one resident set of CTAs.
// Bit-exact by construction (pure data movement).  HBM-bound: algorithmic bytes = 2 x elements.
#include <cuda.h>  // CUtensorMap and the cuTensorMapEncodeTiled prototype only: the entry point is fetched through the runtime
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "kernels.cuh"

namespace mdim {

// Resident CTAs per SM the register allocation aims for.  6 (40 registers) lets all four loads of a thread issue before
// the first shared store; with 8 (32 registers) they go out two at a time.  Measured at 4096^2 on rotating buffers:
// 8 -> 5 675 GB/s, 7 -> same code as 8, 6 -> 5 750, 5 -> 5 646.
constexpr int kTrMinCtas = 6;

// Address of element `e` of the source.  PEER: the Array is cut into equal blocks of peer_block elements, block p in
// the HBM of GPU p (mapped into this process with CUDA IPC); the owner is e / peer_block, estimated in f32 and
// corrected exactly (e < 2^31 on this path, at most 8 peers, so the estimate is off by at most one).
template <bool PEER, int ES>
__device__ __forceinline__ const char* tr_src(const TransposePlan& T, int64_t e) {
    if constexpr (!PEER) return (const char*)T.src + e * ES;
    else {
        int p = (int)((float)e * T.peer_inv);
        p = p >= T.n_peers ? T.n_peers - 1 : p;
        if ((int64_t)((uint64_t)p * T.peer_block) > e) --p;
        else if ((int64_t)((uint64_t)(p + 1) * T.peer_block) <= e) ++p;
        return (const char*)T.peer[p] + (e - (int64_t)((uint64_t)p * T.peer_block)) * ES;
    }
}

template <int ES, bool VEC, bool PEER>
__global__ void __launch_bounds__(kTrThreads, kTrMinCtas) k_transpose(const __grid_constant__ TransposePlan T, void* __restrict__ out_v) {
    constexpr int TAC = kTrTileChunks, TB = kTrTileRows;
    constexpr int CH = 16 / ES;            // elements per 16-byte chunk
    constexpr int EW = ES / 4;             // 32-bit words per element
    constexpr int TA = TAC * CH;           // tile extent along A (elements); TAC chunks = TAC*16 bytes per source run
    constexpr int RW = TAC * 4;            // shared row pitch in words
    constexpr int RPP = kTrThreads / TAC;  // source rows per load pass
    constexpr int NP = TB / RPP;           // passes per tile (load and store phases alike)
    constexpr int LB = NP > 8 ? 8 : NP;    // loads kept in registers at once
    constexpr int PA = TA / 32;            // store-phase groups along A
    constexpr int NBG = TB / (8 * CH);     // store-phase groups of 8 output chunks along B
    static_assert(NP * RPP == TB && PA * NBG == NP && TAC % 8 == 0, "tile shape");
    extern __shared__ __align__(16) uint32_t smem[];  // TB x RW words
    pdl_entry(T.nowait != 0);

    char* __restrict__ out = (char*)out_v;
    const int tid = threadIdx.x;
    // load-phase coordinates
    const int aq = tid % TAC, br = tid / TAC;
    // store-phase coordinates
    const int lane = tid & 31, w = tid >> 5;
    const int bq_lo = lane & 7, a_lo = lane >> 3;

    for (uint64_t tile = blockIdx.x; tile < T.n_tiles; tile += gridDim.x) {
        // neighbouring CTAs write neighbouring pieces of the same output rows
        const uint64_t tb = tile % T.tiles_b;
        const uint64_t r = tile / T.tiles_b;
        const uint64_t ta = r % T.tiles_a;
        uint64_t batch = r / T.tiles_a;
        int64_t src_base = T.src_offset, out_base = 0;
#pragma unroll
        for (int k = kMaxRank - 1; k >= 0; --k) {
            if (k < T.n_batch) {
                const uint64_t c = batch % T.batch_len[k];
                batch /= T.batch_len[k];
                src_base += (int64_t)c * T.batch_src_stride[k];
                out_base += (int64_t)c * T.batch_out_stride[k];
            }
        }
        const uint64_t a0 = ta * TA, b0 = tb * TB;
        const bool full = a0 + TA <= T.len_a && b0 + TB <= T.len_b;  // interior tile: no per-access bounds tests

        // ---- load: global (contiguous along A) -> swizzled shared --------------------------------
#pragma unroll
        for (int h = 0; h < NP; h += LB) {
            uint4 v[LB];
#pragma unroll
            for (int q = 0; q < LB; ++q) {
                const int b_l = (h + q) * RPP + br;
                const uint64_t b = b0 + b_l, a = a0 + (uint64_t)aq * CH;
                const int64_t e = src_base + (int64_t)b * T.src_stride_b + (int64_t)a;
                v[q] = make_uint4(0, 0, 0, 0);
                if constexpr (VEC) {
                    if (full || (b < T.len_b && a < T.len_a))
                        asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                                     : "=r"(v[q].x), "=r"(v[q].y), "=r"(v[q].z), "=r"(v[q].w) : "l"(tr_src<PEER, ES>(T, e)));
                } else {
                    uint32_t wds[4] = {0, 0, 0, 0};
#pragma unroll
                    for (int i = 0; i < CH; ++i) {
                        if (b < T.len_b && a + i < T.len_a) {
                            if constexpr (ES == 4) wds[i] = __ldg((const uint32_t*)tr_src<PEER, ES>(T, e + i));
                            else { const uint2 t = __ldg((const uint2*)tr_src<PEER, ES>(T, e + i)); wds[2 * i] = t.x; wds[2 * i + 1] = t.y; }
                        }
                    }
                    v[q] = make_uint4(wds[0], wds[1], wds[2], wds[3]);
                }
            }
#pragma unroll
            for (int q = 0; q < LB; ++q) {
                const int b_l = (h + q) * RPP + br;
                const int chunk = aq ^ ((b_l / CH) & 7);
                *reinterpret_cast<uint4*>(&smem[b_l * RW + chunk * 4]) = v[q];
            }
        }
        __syncthreads();

        // ---- store: shared (gathered along B) -> global (contiguous along B) ---------------------
        // Passes walk the B groups first, so one warp finishes a whole TB*ES-byte output run per A row
        // in NBG consecutive instructions.
#pragma unroll
        for (int p = 0; p < NP; ++p) {
            const int a_l = 4 * (w + 8 * (p / NBG)) + a_lo;
            const int bq = bq_lo + 8 * (p % NBG);
            uint32_t wds[4];
#pragma unroll
            for (int i = 0; i < CH; ++i) {
                const int b_l = bq * CH + i;
                const int word = b_l * RW + (((a_l / CH) ^ (bq & 7)) * 4) + (a_l % CH) * EW;
                if constexpr (ES == 4) wds[i] = smem[word];
                else { const uint2 t = *reinterpret_cast<const uint2*>(&smem[word]); wds[2 * i] = t.x; wds[2 * i + 1] = t.y; }
            }
            const uint64_t a = a0 + a_l, b = b0 + (uint64_t)bq * CH;
            const int64_t e = out_base + (int64_t)a * T.out_stride_a + (int64_t)b;
            if constexpr (VEC) {
                if (full || (a < T.len_a && b < T.len_b))
                    asm volatile("st.global.cs.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(out + e * ES), "r"(wds[0]), "r"(wds[1]), "r"(wds[2]), "r"(wds[3]) : "memory");
            } else {
#pragma unroll
                for (int i = 0; i < CH; ++i) {
                    if (a < T.len_a && b + i < T.len_b) {
                        if constexpr (ES == 4) *(uint32_t*)(out + (e + i) * 4) = wds[i];
                        else *(uint2*)(out + (e + i) * 8) = make_uint2(wds[2 * i], wds[2 * i + 1]);
                    }
                }
            }
        }
        __syncthreads();
    }
}

// ---- tensor-map TMA form (round 2) ---------------------------------------------------------------------------------
// One CTA = one tile of 64 x 64 elements.  Thread 0 decodes the tile coordinates and issues
//   load : cp.async.bulk.tensor (UTMALDG) of GA boxes, each 128 bytes along A x (GB * E) source rows, SWIZZLE_128B,
//          completion counted in bytes on one mbarrier;
// every thread then moves blocks of CH rows x 16 bytes shared -> registers -> shared: block (bb, c) of the tile as
// loaded ([b][a], a contiguous) becomes block (c, bb) of the tile as stored ([a][b], b contiguous), the CH x CH
// transposition itself being a renaming of registers.  The 8 lanes of a quarter-warp take the blocks (c, bb) =
// (k, (k + d) & 7): with the 128-byte swizzle (16-byte chunk ^ (row & 7)) both the loads and the stores then hit 8
// distinct bank groups — no conflicts, no padding.  Thread 0 finally issues
//   store: cp.async.bulk.tensor (UTMASTG) of GB boxes, each 128 bytes along B x (GA * E) output rows.
// Edge tiles need no code: TMA zero-fills loads and clips stores at the tensor bounds.  All the address arithmetic of
// the register-staged kernel above (323 IMAD + 75 LDC per thread and tile, SM 44 % busy) is gone: per thread and tile this
// is CH x (LDS.128 + STS.128) per block, one mbarrier wait and one CTA barrier.
// Measured on a B200 (scripts/probe/tr_tma_probe.cu, profiles/r2_tr_tma_probe.md): 16384^2 f32 6 566 GB/s (register-staged:
// 6 320), and together with dependency-aware launches (launch.cuh) 4096^2 f32 20.5 us per launch back to back = 6 560 GB/s
// (5 766).  Persistent forms with 4-12 stage rings were slower at every size (one issuing thread per SM serialises).
struct TmaTrArgs {
    uint32_t tiles_a, tiles_b, n_tiles;
    uint32_t batch_len[3];
    int32_t n_batch, a_fastest, nowait;
    int32_t n_peers;            // > 1: source row block p (tiles_b_per_peer tiles along B each) is read through src.m[p]
    uint32_t tiles_b_per_peer;
};
template <int N> struct TmaSrcMaps { CUtensorMap m[N]; };

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void tma_load_tile(uint32_t dst, const CUtensorMap* m, int rank, int c0, int c1, int c2, int c3, int c4, uint32_t bar) {
    switch (rank) {
        case 2: asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst), "l"(m), "r"(c0), "r"(c1), "r"(bar) : "memory"); break;
        case 3: asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(dst), "l"(m), "r"(c0), "r"(c1), "r"(c2), "r"(bar) : "memory"); break;
        case 4: asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];" ::"r"(dst), "l"(m), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(bar) : "memory"); break;
        default: asm volatile("cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5, %6}], [%7];" ::"r"(dst), "l"(m), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4), "r"(bar) : "memory"); break;
    }
}
__device__ __forceinline__ void tma_store_tile(const CUtensorMap* m, int rank, int c0, int c1, int c2, int c3, int c4, uint32_t src) {
    switch (rank) {
        case 2: asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];" ::"l"(m), "r"(c0), "r"(c1), "r"(src) : "memory"); break;
        case 3: asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%1, %2, %3}], [%4];" ::"l"(m), "r"(c0), "r"(c1), "r"(c2), "r"(src) : "memory"); break;
        case 4: asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%1, %2, %3, %4}], [%5];" ::"l"(m), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(src) : "memory"); break;
        default: asm volatile("cp.async.bulk.tensor.5d.global.shared::cta.bulk_group [%0, {%1, %2, %3, %4, %5}], [%6];" ::"l"(m), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4), "r"(src) : "memory"); break;
    }
}

template <int ES> struct TmaTile {
    static constexpr int E = 128 / ES;       // elements per 128-byte shared row
    static constexpr int G = 64 / E;         // boxes per tile side: the tile is 64 x 64 elements
    static constexpr int NT = ES == 4 ? 128 : 256;
    static constexpr int SUB = E * 128;      // bytes of one E x E sub-tile
    static constexpr int TILE = G * G * SUB; // 16 KB (f32) / 32 KB (f64, usize)
    static constexpr int SMEM = 2 * TILE + 1024 + 16;
};

template <int ES, int NP>
__global__ void __launch_bounds__(TmaTile<ES>::NT) k_transpose_tma(const __grid_constant__ TmaSrcMaps<NP> src_maps, const __grid_constant__ CUtensorMap dst_map,
                                                                   const __grid_constant__ TmaTrArgs A) {
    using TT = TmaTile<ES>;
    constexpr int E = TT::E, CH = 16 / ES, G = TT::G, SUB = TT::SUB, TILE = TT::TILE, NT = TT::NT, NBLK = G * G * 64;
    extern __shared__ uint8_t tma_smem_raw[];
    const uint32_t ib = (smem_u32(tma_smem_raw) + 1023u) & ~1023u;  // SWIZZLE_128B repeats every 1024 bytes: chunk ^ (row & 7) needs 1 KB alignment
    const uint32_t ob = ib + TILE, bar = ob + TILE;
    const int tid = threadIdx.x;
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    int ca = 0, cb = 0, cx[3] = {0, 0, 0};  // cx[j]: coordinate along tensor-map dimension 2 + j = batch axis n_batch - 1 - j
    const int rank = 2 + A.n_batch;
    if (tid == 0) {
        // only this thread touches global memory, so it alone takes part in the stream-order wait (launch.cuh)
        uint32_t t = blockIdx.x, ta, tb;
        if (A.a_fastest) { ta = t % A.tiles_a; t /= A.tiles_a; tb = t % A.tiles_b; t /= A.tiles_b; }
        else { tb = t % A.tiles_b; t /= A.tiles_b; ta = t % A.tiles_a; t /= A.tiles_a; }
#pragma unroll
        for (int j = 0; j < 3; ++j)
            if (j < A.n_batch) { const uint32_t n = A.batch_len[A.n_batch - 1 - j]; cx[j] = (int)(t % n); t /= n; }
        const CUtensorMap* sm = &src_maps.m[0];
        int row0 = (int)tb * 64;
        if constexpr (NP > 1) {
            // spread neighbouring CTAs over the peers, so that every NVLink port is busy from the first wave on
            const uint32_t p = tb % (uint32_t)A.n_peers, i = tb / (uint32_t)A.n_peers;
            tb = p * A.tiles_b_per_peer + i;
            sm = &src_maps.m[p];
            row0 = (int)i * 64;  // row inside peer p's block
        }
        ca = (int)ta * 64; cb = (int)tb * 64;
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        if (!A.nowait || blockIdx.x == gridDim.x - 1) asm volatile("griddepcontrol.wait;" ::: "memory");
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"((uint32_t)TILE) : "memory");
#pragma unroll
        for (int ga = 0; ga < G; ++ga)  // box ga: words [32 (ca / E + ga), +32) of the source rows [row0, row0 + 64)
            tma_load_tile(ib + ga * (G * SUB), sm, rank, (ca / E + ga) * 32, row0, cx[0], cx[1], cx[2], bar);
    }
    __syncthreads();  // the barrier is initialised
    asm volatile(
        "{\n .reg .pred p;\n TR_WAIT_%=:\n mbarrier.try_wait.parity.shared::cta.b64 p, [%0], 0;\n @p bra TR_DONE_%=;\n bra TR_WAIT_%=;\n TR_DONE_%=:\n}\n" ::"r"(bar) : "memory");
#pragma unroll
    for (int w0 = 0; w0 < NBLK; w0 += NT) {
        const int w = w0 + tid;
        const int k = w & 7, q = (w >> 3) & 3, u = w >> 5, st = u & 1, sub = u >> 1;
        const int ga = sub % G, gb = sub / G;
        const int c = k, bb = (k + q + 4 * st) & 7;
        uint32_t v[CH][4];
#pragma unroll
        for (int i = 0; i < CH; ++i) {
            const int r = gb * E + bb * CH + i;
            asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v[i][0]), "=r"(v[i][1]), "=r"(v[i][2]), "=r"(v[i][3]) : "r"(ib + ga * (G * SUB) + r * 128 + ((c ^ (r & 7)) << 4)));
        }
#pragma unroll
        for (int j = 0; j < CH; ++j) {
            const int r = ga * E + c * CH + j;
            const uint32_t addr = ob + gb * (G * SUB) + r * 128 + ((bb ^ (r & 7)) << 4);
            if constexpr (ES == 4)
                asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(v[0][j]), "r"(v[1][j]), "r"(v[2][j]), "r"(v[3][j]) : "memory");
            else
                asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(v[0][2 * j]), "r"(v[0][2 * j + 1]), "r"(v[1][2 * j]), "r"(v[1][2 * j + 1]) : "memory");
        }
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // the generic-proxy stores above become visible to the TMA engine
    __syncthreads();
    if (tid == 0) {
#pragma unroll
        for (int gb = 0; gb < G; ++gb)  // box gb: words [32 (cb / E + gb), +32) of the output rows [ca, ca + 64)
            tma_store_tile(&dst_map, rank, (cb / E + gb) * 32, ca, cx[0], cx[1], cx[2], ob + gb * (G * SUB));
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");  // shared memory must outlive the reads of the store engine
    }
}

static bool transpose_vec_ok(const TransposePlan& T, const void* out) {
    const int ch = 16 / T.esize;
    bool vec = ((uintptr_t)T.src + (uintptr_t)(T.src_offset * T.esize)) % 16 == 0 && ((uintptr_t)out % 16) == 0 && T.src_stride_b % ch == 0 &&
               T.out_stride_a % ch == 0 && T.len_a % ch == 0 && T.len_b % ch == 0;
    for (int k = 0; k < T.n_batch; ++k) vec = vec && T.batch_src_stride[k] % ch == 0 && T.batch_out_stride[k] % ch == 0;
    if (T.n_peers > 1) {  // every 16-byte chunk must lie inside one peer's block, 16-byte aligned there
        vec = vec && T.peer_block % ch == 0 && T.src_offset % ch == 0;
        for (int p = 0; p < T.n_peers; ++p) vec = vec && ((uintptr_t)T.peer[p] % 16) == 0;
    }
    return vec;
}

template <int ES, bool VEC, bool PEER>
static cudaError_t launch_tr1(const TransposePlan& T, void* out, int grid, cudaStream_t stream) {
    constexpr int smem = kTrTileRows * kTrTileChunks * 16;
    static const bool once = [] { return cudaFuncSetAttribute(k_transpose<ES, VEC, PEER>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) == cudaSuccess; }();
    (void)once;
    return launch_pdl(k_transpose<ES, VEC, PEER>, dim3(grid), dim3(kTrThreads), smem, stream, T, out);
}

template <int ES>
static cudaError_t launch_tr(const TransposePlan& T, void* out, int grid, bool vec, cudaStream_t stream) {
    const bool peer = T.n_peers > 1;
    if (vec) return peer ? launch_tr1<ES, true, true>(T, out, grid, stream) : launch_tr1<ES, true, false>(T, out, grid, stream);
    return peer ? launch_tr1<ES, false, true>(T, out, grid, stream) : launch_tr1<ES, false, false>(T, out, grid, stream);
}

// ---- host side of the TMA form ---------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn tma_encode_fn() {  // libcuda is not linked: the driver entry point comes through the runtime
    static const EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) p = nullptr;
        return (EncodeTiledFn)p;
    }();
    return fn;
}

// A tensor of 32-bit words: dimension 0 = the contiguous axis (`inner` elements of `es` bytes), dimension 1 = `rows` rows
// `row_stride` elements apart, then the batch axes innermost first.  Box = 128 bytes x 64 rows.
static bool tma_encode(CUtensorMap* m, const void* base, int es, uint64_t inner, uint64_t rows, int64_t row_stride, int n_batch, const uint64_t* batch_len,
                       const int64_t* batch_stride) {
    const EncodeTiledFn fn = tma_encode_fn();
    if (!fn || ((uintptr_t)base & 15)) return false;
    cuuint64_t dims[5], strides[4];
    cuuint32_t box[5] = {32, 64, 1, 1, 1}, estr[5] = {1, 1, 1, 1, 1};
    auto stride_ok = [&](int64_t s) { return s > 0 && ((uint64_t)s * (uint64_t)es) % 16 == 0 && (uint64_t)s * (uint64_t)es < (1ull << 40); };
    dims[0] = inner * (uint64_t)(es / 4); dims[1] = rows;
    if (!stride_ok(row_stride) || dims[0] > 0xffffffffull || rows > 0xffffffffull) return false;
    strides[0] = (uint64_t)row_stride * (uint64_t)es;
    for (int j = 0; j < n_batch; ++j) {
        const int k = n_batch - 1 - j;
        if (!stride_ok(batch_stride[k]) || batch_len[k] > 0xffffffffull) return false;
        dims[2 + j] = batch_len[k];
        strides[1 + j] = (uint64_t)batch_stride[k] * (uint64_t)es;
    }
    return fn(m, CU_TENSOR_MAP_DATA_TYPE_UINT32, (cuuint32_t)(2 + n_batch), const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
              CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <int ES, int NP>
static bool launch_tma1(const TmaSrcMaps<NP>& sm, const CUtensorMap& dm, const TmaTrArgs& A, cudaStream_t stream) {
    using TT = TmaTile<ES>;
    static const bool ok = cudaFuncSetAttribute(k_transpose_tma<ES, NP>, cudaFuncAttributeMaxDynamicSharedMemorySize, TT::SMEM) == cudaSuccess;
    if (!ok) return false;
    return launch_pdl(k_transpose_tma<ES, NP>, dim3(A.n_tiles), dim3(TT::NT), TT::SMEM, stream, sm, dm, A) == cudaSuccess;
}

// MDIM_TR_TMA=0 keeps the register-staged kernel (benchmarks, and the fallback's own tests)
static bool use_tma() {
    static const bool on = [] { const char* e = getenv("MDIM_TR_TMA"); return !(e && e[0] == '0'); }();
    return on;
}

// -> false: not expressible as tensor maps (misaligned base, negative / unaligned strides, > 3 batch axes, a sharded source
// whose tiles straddle peers ...): the caller falls back to the register-staged kernel.
static bool launch_transpose_tma(const TransposePlan& T, void* out, cudaStream_t stream) {
    if (!use_tma() || (T.esize != 4 && T.esize != 8) || T.n_batch > 3) return false;
    const int es = T.esize;
    TmaTrArgs A;
    memset(&A, 0, sizeof A);
    const uint64_t tiles_a = (T.len_a + 63) / 64, tiles_b = (T.len_b + 63) / 64;
    uint64_t n_tiles = tiles_a * tiles_b;
    for (int k = 0; k < T.n_batch; ++k) { n_tiles *= T.batch_len[k]; A.batch_len[k] = (uint32_t)T.batch_len[k]; }
    if (n_tiles == 0 || n_tiles > 0x7fffffffull) return false;
    A.tiles_a = (uint32_t)tiles_a; A.tiles_b = (uint32_t)tiles_b; A.n_tiles = (uint32_t)n_tiles; A.n_batch = T.n_batch; A.nowait = T.nowait;
    // tile order: A-fastest measured +2.5 % at 4096^2 and -0.5 % at 16384^2 (profiles/r2_tr_tma_probe.md)
    A.a_fastest = 2 * T.len_a * T.len_b * (uint64_t)es <= (512ull << 20) ? 1 : 0;
    CUtensorMap dm;
    if (!tma_encode(&dm, out, es, T.len_b, T.len_a, T.out_stride_a, T.n_batch, T.batch_len, T.batch_out_stride)) return false;
    if (T.n_peers > 1) {
        // row-sharded 2-D source of row pitch S, peer p holding rows [p * rows_pp, (p + 1) * rows_pp); this launch reads the column
        // window [src_offset, src_offset + len_a) of every row (a rank's block of the transposed rows).  One tensor map per peer,
        // and a tile never straddles two of them.
        const int64_t S = T.src_stride_b;
        if (T.n_batch != 0 || S <= 0 || T.src_offset < 0 || T.src_offset + (int64_t)T.len_a > S || T.peer_block % ((uint64_t)S * 64) != 0) return false;
        const uint64_t rows_pp = T.peer_block / (uint64_t)S;
        if (rows_pp * (uint64_t)T.n_peers != T.len_b) return false;
        TmaSrcMaps<MDIM_MAX_PEERS> sm;
        memset(&sm, 0, sizeof sm);
        for (int p = 0; p < T.n_peers; ++p)
            if (!tma_encode(&sm.m[p], (const char*)T.peer[p] + T.src_offset * es, es, T.len_a, rows_pp, S, 0, nullptr, nullptr)) return false;
        A.n_peers = T.n_peers; A.tiles_b_per_peer = (uint32_t)(rows_pp / 64);
        return es == 4 ? launch_tma1<4, MDIM_MAX_PEERS>(sm, dm, A, stream) : launch_tma1<8, MDIM_MAX_PEERS>(sm, dm, A, stream);
    }
    TmaSrcMaps<1> sm;
    if (!tma_encode(&sm.m[0], (const char*)T.src + T.src_offset * es, es, T.len_a, T.len_b, T.src_stride_b, T.n_batch, T.batch_len, T.batch_src_stride)) return false;
    return es == 4 ? launch_tma1<4, 1>(sm, dm, A, stream) : launch_tma1<8, 1>(sm, dm, A, stream);
}

const char* launch_transpose(const Plan& p, void* out, bool nowait, cudaStream_t stream, int sm_count) {
    TransposePlan T = p.tr;
    T.nowait = nowait;
    if (launch_transpose_tma(T, out, stream)) return T.n_peers > 1 ? "k_transpose_tma<peer>" : "k_transpose_tma";
    // Not persistent: far more CTAs than fit at once, so the hardware scheduler balances the tail.
    // Measured (B200, 16384^2 f32): 8/SM (resident set) 5.71 TB/s, 64/SM 6.18, 128/SM 6.32, one CTA per tile 6.35.
    const int grid = (int)std::min<uint64_t>(T.n_tiles, std::max<uint64_t>((uint64_t)sm_count * 128, 1));
    const bool vec = transpose_vec_ok(T, out);
    const cudaError_t e = T.esize == 4 ? launch_tr<4>(T, out, grid, vec, stream) : launch_tr<8>(T, out, grid, vec, stream);
    if (e != cudaSuccess) return nullptr;
    return vec ? "k_transpose<regs,vec>" : "k_transpose<regs,scalar>";
}

}  // namespace mdim
