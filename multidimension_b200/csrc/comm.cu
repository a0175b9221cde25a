// comm.cu — the multi-GPU surface of the C ABI (include/mdim.h, "one process per GPU"): an NCCL communicator
// bound to the context, the two collectives the north star names (all-gather of a sharded compose() source,
// all-reduce of the partial folds over a sharded axis), and the peer table that lets the gather / transpose /
// fold kernels read the other GPUs' blocks directly over NVLink (CUDA IPC handles exchanged over the communicator).
//
// NCCL is loaded at run time (dlopen of libnccl.so.2: the copy already in the process if the host program has one,
// e.g. the NCCL bundled with torch, else the system library): the library has no link-time dependency on it, and a
// single-GPU user never needs it.  Only a handful of long-stable entry points are used, declared below with NCCL's
// own ABI (ncclUniqueId is 128 bytes; ncclDataType_t / ncclRedOp_t values are fixed by nccl.h since 2.0).
#include <cuda.h>
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "ctx.hpp"
#include "kernels.cuh"

namespace mdim {

namespace {

struct NcclId { char internal[128]; };
typedef void* NcclComm;
enum { kNcclSuccess = 0 };
// ncclDataType_t
enum { kNcclInt8 = 0, kNcclUint8 = 1, kNcclInt32 = 2, kNcclUint32 = 3, kNcclInt64 = 4, kNcclUint64 = 5, kNcclFloat32 = 7, kNcclFloat64 = 8 };
// ncclRedOp_t
enum { kNcclSum = 0, kNcclProd = 1, kNcclMax = 2, kNcclMin = 3 };

struct NcclApi {
    void* lib = nullptr;
    int (*GetUniqueId)(NcclId*) = nullptr;
    int (*CommInitRank)(NcclComm*, int, NcclId, int) = nullptr;
    int (*CommDestroy)(NcclComm) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, NcclComm, cudaStream_t) = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, NcclComm, cudaStream_t) = nullptr;
    int (*GetVersion)(int*) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
    bool ok = false;
    char why[160] = {0};
};

NcclApi& nccl() {
    static NcclApi api = [] {
        NcclApi a;
        const char* names[] = {getenv("MDIM_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
        for (const char* n : names) {
            if (!n || !*n) continue;
            a.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
            if (a.lib) break;
        }
        if (!a.lib) { snprintf(a.why, sizeof a.why, "libnccl.so.2 not found (%s)", dlerror()); return a; }
#define SYM(field, name) *(void**)(&a.field) = dlsym(a.lib, name); if (!a.field) { snprintf(a.why, sizeof a.why, "libnccl lacks %s", name); return a; }
        SYM(GetUniqueId, "ncclGetUniqueId") SYM(CommInitRank, "ncclCommInitRank") SYM(CommDestroy, "ncclCommDestroy") SYM(AllGather, "ncclAllGather")
        SYM(AllReduce, "ncclAllReduce") SYM(GetVersion, "ncclGetVersion") SYM(GetErrorString, "ncclGetErrorString")
#undef SYM
        a.ok = true;
        return a;
    }();
    return api;
}

int nccl_fail(mdim_ctx* ctx, int rc, const char* what) {
    char msg[160];
    snprintf(msg, sizeof msg, "%s: %s", what, nccl().GetErrorString ? nccl().GetErrorString(rc) : "NCCL error");
    return ctx ? set_error(ctx, MDIM_ERR_NCCL, msg) : MDIM_ERR_NCCL;
}

#define NC(ctx, call)                                         \
    do {                                                      \
        int rc_ = (call);                                     \
        if (rc_ != kNcclSuccess) return nccl_fail(ctx, rc_, #call); \
    } while (0)

}  // namespace

struct Comm {
    NcclComm comm = nullptr;
    int rank = 0, world = 1;
    char* scratch = nullptr;  // device staging for the small host-side exchanges (IPC handles, barrier word)
    size_t scratch_bytes = 0;
    struct Opened { cudaIpcMemHandle_t handle; void* base; };  // one mapping per peer ALLOCATION, however many blocks live in it
    std::vector<Opened> opened;  // IPC mappings made by mdim_peer_table, closed by mdim_peer_table_close / shutdown
    // state of the pipelined fold over the sharded axis (k_fold_ring.cu): one allocation per rank, mapped into every rank
    //   [inbox: kRingCap x 16 B][result: kRingCap x 16 B][error: 4 B]   (flag-in-data lines: 2 x the data bytes)
    char* ring = nullptr;
    void* ring_peer[MDIM_MAX_PEERS] = {nullptr};
    uint32_t ring_epoch = 0;
    // packet areas of the in-kernel all-reduce (k_fold_xchg.cu): [slot 0/1][source rank 0..N-1, results][kXchgCapWords x 8 B] + an error word
    char* xchg = nullptr;
    void* xchg_peer[MDIM_MAX_PEERS] = {nullptr};
    uint32_t xchg_epoch = 0;
};
constexpr uint64_t kXchgCapWords = 1ull << 20;     // 32-bit words of columns per launch (4 MiB of a row; wider rows take several launches)
inline size_t xchg_error_off(int world) { return (size_t)2 * (size_t)(world + 1) * kXchgCapWords * 8; }
constexpr uint64_t kRingCap = 1ull << 20;          // columns per launch (a wider result is folded in several launches)
constexpr size_t kRingInboxOff = 0, kRingResultOff = kRingCap * 16, kRingErrorOff = 2 * kRingCap * 16, kRingBytes = kRingErrorOff + 256;

void comm_destroy(mdim_ctx* ctx) {
    Comm* c = ctx->comm;
    if (!c) return;
    for (const Comm::Opened& o : c->opened) cudaIpcCloseMemHandle(o.base);
    if (c->scratch) cudaFree(c->scratch);
    if (c->ring) cudaFree(c->ring);
    if (c->xchg) cudaFree(c->xchg);
    if (c->comm && nccl().ok) nccl().CommDestroy(c->comm);
    delete c;
    ctx->comm = nullptr;
}

namespace {

// all-gather `bytes` of host data per rank through the communicator: -> out[world * bytes]
int exchange_host(mdim_ctx* ctx, const void* mine, size_t bytes, void* out) {
    Comm* c = ctx->comm;
    const size_t need = bytes * (size_t)(c->world + 1);
    if (need > c->scratch_bytes) {
        if (c->scratch) CU(ctx, cudaFree(c->scratch));
        c->scratch = nullptr;
        CU(ctx, cudaMalloc(&c->scratch, need));
        c->scratch_bytes = need;
    }
    char* send = c->scratch + bytes * (size_t)c->world;
    CU(ctx, cudaMemcpyAsync(send, mine, bytes, cudaMemcpyHostToDevice, ctx->stream));
    NC(ctx, nccl().AllGather(send, c->scratch, bytes, kNcclUint8, c->comm, ctx->stream));
    poison_inflight(ctx);
    CU(ctx, cudaMemcpyAsync(out, c->scratch, bytes * (size_t)c->world, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return MDIM_OK;
}

typedef CUresult (*GetAddressRangeFn)(CUdeviceptr*, size_t*, CUdeviceptr);
GetAddressRangeFn address_range_fn() {
    static const GetAddressRangeFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuMemGetAddressRange", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) p = nullptr;
        return (GetAddressRangeFn)p;
    }();
    return fn;
}

struct PeerRecord {  // what every rank publishes about its block
    cudaIpcMemHandle_t handle;  // of the ALLOCATION the block lives in (cudaIpcGetMemHandle ignores interior offsets)
    uint64_t offset;            // of the block inside that allocation
    uint64_t bytes;
};

}  // namespace
}  // namespace mdim

using namespace mdim;

extern "C" {

int mdim_comm_unique_id(uint8_t id[MDIM_COMM_ID_BYTES]) {
    if (!id) return MDIM_ERR_INVALID;
    static_assert(sizeof(NcclId) == MDIM_COMM_ID_BYTES, "ncclUniqueId is 128 bytes");
    if (!nccl().ok) return MDIM_ERR_NCCL;
    NcclId u;
    if (nccl().GetUniqueId(&u) != kNcclSuccess) return MDIM_ERR_NCCL;
    memcpy(id, &u, sizeof u);
    return MDIM_OK;
}

int mdim_comm_init(mdim_ctx* ctx, int rank, int world, const uint8_t id[MDIM_COMM_ID_BYTES]) {
    if (!ctx || !id || world < 1 || rank < 0 || rank >= world || world > MDIM_MAX_PEERS) return MDIM_ERR_INVALID;
    if (ctx->comm) return set_error(ctx, MDIM_ERR_INVALID, "the context already has a communicator");
    if (!nccl().ok) return set_error(ctx, MDIM_ERR_NCCL, nccl().why);
    CU(ctx, cudaSetDevice(ctx->device));
    Comm* c = new (std::nothrow) Comm();
    if (!c) return MDIM_ERR_NOMEM;
    c->rank = rank; c->world = world;
    NcclId u;
    memcpy(&u, id, sizeof u);
    const int rc = nccl().CommInitRank(&c->comm, world, u, rank);
    if (rc != kNcclSuccess) { delete c; return nccl_fail(ctx, rc, "ncclCommInitRank"); }
    ctx->comm = c;
    return MDIM_OK;
}

int mdim_comm_destroy(mdim_ctx* ctx) {
    if (!ctx) return MDIM_ERR_INVALID;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    comm_destroy(ctx);
    return MDIM_OK;
}

int mdim_comm_info(mdim_ctx* ctx, int* rank, int* world, int* nccl_version) {
    if (!ctx) return MDIM_ERR_INVALID;
    if (rank) *rank = ctx->comm ? ctx->comm->rank : 0;
    if (world) *world = ctx->comm ? ctx->comm->world : 1;
    if (nccl_version) { *nccl_version = 0; if (nccl().ok) nccl().GetVersion(nccl_version); }
    return MDIM_OK;
}

// ncclAllGather of every rank's `block_bytes` into `recv` (rank-major), on the context's stream, asynchronous.
int mdim_allgather(mdim_ctx* ctx, const void* send_device, void* recv_device, size_t block_bytes) {
    if (!ctx || !ctx->comm) return ctx ? set_error(ctx, MDIM_ERR_INVALID, "no communicator: call mdim_comm_init") : MDIM_ERR_INVALID;
    if (!block_bytes) return MDIM_OK;
    if (!send_device || !recv_device) return MDIM_ERR_INVALID;
    CU(ctx, cudaSetDevice(ctx->device));
    NC(ctx, nccl().AllGather(send_device, recv_device, block_bytes, kNcclUint8, ctx->comm->comm, ctx->stream));
    poison_inflight(ctx);
    return MDIM_OK;
}

// ncclAllReduce in place over `n` elements of `dtype` with the fold's operator (ADD, MUL, or the min / max of the
// MDIM_REDUCE_* codes), on the context's stream, asynchronous.  f32 sums are reassociated: 1e-6 relative tolerance.
int mdim_allreduce(mdim_ctx* ctx, void* data_device, size_t n, int dtype, int op) {
    if (!ctx || !ctx->comm) return ctx ? set_error(ctx, MDIM_ERR_INVALID, "no communicator: call mdim_comm_init") : MDIM_ERR_INVALID;
    if (!n) return MDIM_OK;
    if (!data_device) return MDIM_ERR_INVALID;
    int nt, no;
    switch (dtype) {
        case MDIM_U8: nt = kNcclUint8; break;
        case MDIM_I8: nt = kNcclInt8; break;
        case MDIM_I16: case MDIM_U16: return set_error(ctx, MDIM_ERR_UNSUPPORTED, "all-reduce: NCCL has no 16-bit integer type");
        case MDIM_I32: nt = kNcclInt32; break;
        case MDIM_U32: nt = kNcclUint32; break;
        case MDIM_I64: nt = kNcclInt64; break;
        case MDIM_U64: nt = kNcclUint64; break;
        case MDIM_F32: nt = kNcclFloat32; break;
        case MDIM_F64: nt = kNcclFloat64; break;
        default: return set_error(ctx, MDIM_ERR_INVALID, "bad dtype");
    }
    switch (op) {
        case MDIM_ADD: no = kNcclSum; break;
        case MDIM_MUL: no = kNcclProd; break;
        case MDIM_REDUCE_MIN: no = kNcclMin; break;
        case MDIM_REDUCE_MAX: no = kNcclMax; break;
        default: return set_error(ctx, MDIM_ERR_UNSUPPORTED, "all-reduce supports ADD, MUL, MIN and MAX");
    }
    CU(ctx, cudaSetDevice(ctx->device));
    NC(ctx, nccl().AllReduce(data_device, data_device, n, nt, no, ctx->comm->comm, ctx->stream));
    poison_inflight(ctx);
    return MDIM_OK;
}

// Every rank has finished everything it enqueued before its own call (a 4-byte all-reduce + stream sync).
int mdim_barrier(mdim_ctx* ctx) {
    if (!ctx || !ctx->comm) return ctx ? set_error(ctx, MDIM_ERR_INVALID, "no communicator: call mdim_comm_init") : MDIM_ERR_INVALID;
    uint32_t one = 1, all[MDIM_MAX_PEERS];
    CU(ctx, cudaSetDevice(ctx->device));
    return exchange_host(ctx, &one, sizeof one, all);
}

// Collective.  Every rank passes its own block (device memory, any interior pointer of a cudaMalloc allocation);
// on return peers[p] addresses rank p's block from THIS process (peers[rank] == local_device), mapped with CUDA IPC
// and readable by the kernels over NVLink / NVSwitch (mdim_node.peer[]).
int mdim_peer_table(mdim_ctx* ctx, void* local_device, size_t block_bytes, void* peers[MDIM_MAX_PEERS]) {
    if (!ctx || !ctx->comm) return ctx ? set_error(ctx, MDIM_ERR_INVALID, "no communicator: call mdim_comm_init") : MDIM_ERR_INVALID;
    if (!local_device || !peers) return MDIM_ERR_INVALID;
    Comm* c = ctx->comm;
    CU(ctx, cudaSetDevice(ctx->device));
    PeerRecord mine;
    memset(&mine, 0, sizeof mine);
    CUdeviceptr base = (CUdeviceptr)(uintptr_t)local_device;
    size_t alloc_size = 0;
    if (GetAddressRangeFn fn = address_range_fn()) {
        if (fn(&base, &alloc_size, (CUdeviceptr)(uintptr_t)local_device) != CUDA_SUCCESS) base = (CUdeviceptr)(uintptr_t)local_device;
    }
    CU(ctx, cudaIpcGetMemHandle(&mine.handle, (void*)(uintptr_t)base));
    mine.offset = (uint64_t)((uintptr_t)local_device - (uintptr_t)base);
    mine.bytes = block_bytes;
    std::vector<PeerRecord> all((size_t)c->world);
    int st = exchange_host(ctx, &mine, sizeof mine, all.data());
    if (st) return st;
    for (int p = 0; p < MDIM_MAX_PEERS; ++p) peers[p] = nullptr;
    for (int p = 0; p < c->world; ++p) {
        if (p == c->rank) { peers[p] = local_device; continue; }
        void* mapped = nullptr;
        for (const Comm::Opened& o : c->opened)
            if (memcmp(&o.handle, &all[(size_t)p].handle, sizeof o.handle) == 0) mapped = o.base;
        if (!mapped) {
            CU(ctx, cudaIpcOpenMemHandle(&mapped, all[(size_t)p].handle, cudaIpcMemLazyEnablePeerAccess));
            c->opened.push_back({all[(size_t)p].handle, mapped});
        }
        peers[p] = (char*)mapped + all[(size_t)p].offset;
    }
    return MDIM_OK;
}

// Collective.  `local_rows` = this rank's rows of an Array whose OUTERMOST axis is sharded over the ranks in rank order
// (dense row-major, n_rows_local x n_cols, device memory); `out` (n_cols elements, device memory, on EVERY rank) receives
//   out[c] = (((init (op) x[0][c]) (op) x[1][c]) ... (op) x[I-1][c])   over ALL ranks' rows in index order
// — the reference's sequential fold (src/view.rs:617-622, 250-252) bit for bit, unlike partial folds + all-reduce.  One fused
// kernel per GPU: the running values travel from rank to rank through peer-mapped HBM, pipelined over column slices
// (csrc/k_fold_ring.cu).  op: ADD, SUB, MUL, AND, OR, XOR; 4- and 8-byte dtypes.  Asynchronous on the context's stream.
int mdim_fold_sharded_axis(mdim_ctx* ctx, const void* local_rows, uint64_t n_rows_local, uint64_t n_cols, int dtype, int op, mdim_scalar init, void* out_device) {
    if (!ctx || !ctx->comm) return ctx ? set_error(ctx, MDIM_ERR_INVALID, "no communicator: call mdim_comm_init") : MDIM_ERR_INVALID;
    if (!local_rows || !out_device) return MDIM_ERR_INVALID;
    const int es = dtype_size(dtype);
    if (es != 4 && es != 8) return set_error(ctx, MDIM_ERR_UNSUPPORTED, "fold over the sharded axis: 4- and 8-byte element types");
    if (!(op == MDIM_ADD || op == MDIM_SUB || op == MDIM_MUL || op == MDIM_AND || op == MDIM_OR || op == MDIM_XOR))
        return set_error(ctx, MDIM_ERR_UNSUPPORTED, "fold over the sharded axis: ADD, SUB, MUL, AND, OR, XOR");
    if ((dtype == MDIM_F32 || dtype == MDIM_F64) && op >= MDIM_AND) return set_error(ctx, MDIM_ERR_INVALID, "bitwise fold of floats");
    if (n_cols == 0 || n_rows_local == 0) return set_error(ctx, MDIM_ERR_UNSUPPORTED, "fold over the sharded axis: every rank must hold at least one row");
    Comm* c = ctx->comm;
    CU(ctx, cudaSetDevice(ctx->device));
    if (!c->ring) {  // first use: allocate the ring state, zero the flags, map everyone's into everyone (collective)
        CU(ctx, cudaMalloc(&c->ring, kRingBytes));
        CU(ctx, cudaMemsetAsync(c->ring, 0, kRingBytes, ctx->stream));
        CU(ctx, cudaStreamSynchronize(ctx->stream));
        int st = mdim_peer_table(ctx, c->ring, kRingBytes, c->ring_peer);
        if (st) return st;
        st = mdim_barrier(ctx);
        if (st) return st;
    }
    const int next = (c->rank + 1) % c->world;
    for (uint64_t c0 = 0; c0 < n_cols; c0 += kRingCap) {
        FoldRingArgs A;
        memset(&A, 0, sizeof A);
        A.n_rows = n_rows_local; A.n_cols = std::min<uint64_t>(kRingCap, n_cols - c0);
        A.dtype = dtype; A.op = op; A.esize = es; A.rank = c->rank; A.world = c->world;
        A.epoch = ++c->ring_epoch;
        A.init = 0; memcpy(&A.init, &init, (size_t)es);
        A.inbox = c->ring + kRingInboxOff;
        A.next_inbox = (char*)c->ring_peer[next] + kRingInboxOff;
        for (int p = 0; p < c->world; ++p) A.result[p] = (char*)c->ring_peer[p] + kRingResultOff;
        A.out = (char*)out_device + c0 * (uint64_t)es;
        A.error = (uint32_t*)(c->ring + kRingErrorOff);
        if (n_cols > kRingCap) return set_error(ctx, MDIM_ERR_UNSUPPORTED, "fold over the sharded axis: more than 2^20 columns per call (strided column windows: fold the result in blocks)");
        const int rc = launch_fold_ring(A, local_rows, ctx->sm_count, ctx->stream);
        if (rc == -1) return set_error(ctx, MDIM_ERR_UNSUPPORTED, "fold over the sharded axis: the rows must be 16-byte aligned with a 16-byte multiple row length");
        if (rc) return cuda_fail(ctx, (cudaError_t)rc, "k_fold_ring");
        ctx->launches++;
        snprintf(ctx->last_kernel, sizeof ctx->last_kernel, "k_fold_ring");
    }
    poison_inflight(ctx);
    return MDIM_OK;
}

// Collective.  The all-reduce route of the same fold (SURVEY.md §8e) as ONE fused kernel per GPU (csrc/k_fold_xchg.cu):
//   P_r = rank r's rows folded sequentially (rank 0 from `init`, the others from the operator's identity);
//   out = ((P_0 (op) P_1) (op) P_2) ... (op) P_{N-1}, the same order on every rank.
// Bit-identical to the reference for integer / bitwise folds; float sums are reassociated at the rank boundaries only:
// deterministic, as accurate as the reference's order, ~1e-6 relative away from it over 1024 f32 terms (like ncclAllReduce).  op: ADD, MUL, AND, OR, XOR.  Asynchronous on the context's stream.
int mdim_fold_sharded_axis_blocked(mdim_ctx* ctx, const void* local_rows, uint64_t n_rows_local, uint64_t n_cols, int dtype, int op, mdim_scalar init,
                                   void* out_device) {
    if (!ctx || !ctx->comm) return ctx ? set_error(ctx, MDIM_ERR_INVALID, "no communicator: call mdim_comm_init") : MDIM_ERR_INVALID;
    if (!local_rows || !out_device) return MDIM_ERR_INVALID;
    const int es = dtype_size(dtype);
    if (es != 4 && es != 8) return set_error(ctx, MDIM_ERR_UNSUPPORTED, "fold over the sharded axis: 4- and 8-byte element types");
    if (!(op == MDIM_ADD || op == MDIM_MUL || op == MDIM_AND || op == MDIM_OR || op == MDIM_XOR))
        return set_error(ctx, MDIM_ERR_UNSUPPORTED, "blocked fold over the sharded axis: ADD, MUL, AND, OR, XOR (the operator needs an identity)");
    if ((dtype == MDIM_F32 || dtype == MDIM_F64) && op >= MDIM_AND) return set_error(ctx, MDIM_ERR_INVALID, "bitwise fold of floats");
    if (n_cols == 0 || n_rows_local == 0) return set_error(ctx, MDIM_ERR_UNSUPPORTED, "fold over the sharded axis: every rank must hold at least one row");
    Comm* c = ctx->comm;
    CU(ctx, cudaSetDevice(ctx->device));
    const size_t area_bytes = xchg_error_off(c->world) + 256;
    if (!c->xchg) {  // first use: allocate the packet areas (zero = no epoch), map everyone's into everyone (collective)
        CU(ctx, cudaMalloc(&c->xchg, area_bytes));
        CU(ctx, cudaMemsetAsync(c->xchg, 0, area_bytes, ctx->stream));
        CU(ctx, cudaStreamSynchronize(ctx->stream));
        int st = mdim_peer_table(ctx, c->xchg, area_bytes, c->xchg_peer);
        if (st) return st;
        st = mdim_barrier(ctx);
        if (st) return st;
    }
    uint64_t identity = 0;  // x (op) identity == x for EVERY x: for a float sum that is -0.0 (+0.0 would turn a partial of -0.0 into +0.0)
    if (op == MDIM_ADD && dtype == MDIM_F32) identity = 0x80000000ull;
    else if (op == MDIM_ADD && dtype == MDIM_F64) identity = 0x8000000000000000ull;
    else if (op == MDIM_AND) identity = ~0ull;
    else if (op == MDIM_MUL) {
        if (dtype == MDIM_F32) { const float one = 1.0f; memcpy(&identity, &one, 4); }
        else if (dtype == MDIM_F64) { const double one = 1.0; memcpy(&identity, &one, 8); }
        else identity = 1;
    }
    if (es == 4) identity &= 0xffffffffull;
    const uint64_t row_bytes = n_cols * (uint64_t)es, window = kXchgCapWords * 4;
    for (uint64_t b0 = 0; b0 < row_bytes; b0 += window) {
        FoldXchgArgs A;
        memset(&A, 0, sizeof A);
        A.n_rows = n_rows_local; A.row_bytes = std::min<uint64_t>(window, row_bytes - b0); A.pitch_bytes = row_bytes;
        A.rank = c->rank; A.world = c->world;
        A.epoch = ++c->xchg_epoch; A.slot = A.epoch & 1u;
        if (c->rank == 0) memcpy(&A.start, &init, (size_t)es); else A.start = identity;
        A.cap_words = kXchgCapWords;
        A.rows = (const char*)local_rows + b0;
        for (int p = 0; p < c->world; ++p) A.area[p] = (char*)c->xchg_peer[p];
        A.out = (char*)out_device + b0;
        A.error = (uint32_t*)(c->xchg + xchg_error_off(c->world));
        const int rc = launch_fold_xchg(A, dtype, op, ctx->sm_count, ctx->stream);
        if (rc == -1) return set_error(ctx, MDIM_ERR_UNSUPPORTED, "blocked fold over the sharded axis: rows and out 16-byte aligned, row length a multiple of 16 bytes");
        if (rc) return cuda_fail(ctx, (cudaError_t)rc, "k_fold_xchg");
        ctx->launches++;
        snprintf(ctx->last_kernel, sizeof ctx->last_kernel, "k_fold_xchg");
    }
    poison_inflight(ctx);
    return MDIM_OK;
}

// 1 if a fold over the sharded axis gave up waiting for a peer since the last call (then the outputs are garbage)
int mdim_fold_sharded_axis_status(mdim_ctx* ctx) {
    if (!ctx || !ctx->comm) return MDIM_OK;
    Comm* c = ctx->comm;
    char* words[2] = {c->ring ? c->ring + kRingErrorOff : nullptr, c->xchg ? c->xchg + xchg_error_off(c->world) : nullptr};
    bool lost = false;
    CU(ctx, cudaSetDevice(ctx->device));
    for (char* w : words) {
        if (!w) continue;
        uint32_t err = 0;
        CU(ctx, cudaMemcpyAsync(&err, w, 4, cudaMemcpyDeviceToHost, ctx->stream));
        CU(ctx, cudaStreamSynchronize(ctx->stream));
        if (err) { CU(ctx, cudaMemsetAsync(w, 0, 4, ctx->stream)); lost = true; }
    }
    if (lost) return set_error(ctx, MDIM_ERR_NCCL, "fold over the sharded axis: a peer did not arrive within the time limit");
    return MDIM_OK;
}

// Collective (contains a barrier: nobody unmaps while a peer may still be reading).
int mdim_peer_table_close(mdim_ctx* ctx) {
    if (!ctx || !ctx->comm) return MDIM_ERR_INVALID;
    int st = mdim_barrier(ctx);
    if (st) return st;
    for (const Comm::Opened& o : ctx->comm->opened) CU(ctx, cudaIpcCloseMemHandle(o.base));
    ctx->comm->opened.clear();
    // the folds' exchange state was mapped through the same table: drop it, the next fold sets it up again
    if (ctx->comm->ring) { CU(ctx, cudaFree(ctx->comm->ring)); ctx->comm->ring = nullptr; }
    if (ctx->comm->xchg) { CU(ctx, cudaFree(ctx->comm->xchg)); ctx->comm->xchg = nullptr; }
    return mdim_barrier(ctx);
}

}  // extern "C"
