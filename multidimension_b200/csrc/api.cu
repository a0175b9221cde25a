// api.cu — the C ABI of include/mdim.h: context, device-resident boxed buffers, and the
// View::collect entry points (device-resident and host-buffer forms).
//
// Everything that computes runs one of the hand-written sm_100a kernels of this directory; there
// is no CPU fallback: without a usable sm_100 device mdim_init fails with MDIM_ERR_CUDA and no
// other compute entry point can be reached (they all need a context).
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <memory>
#include <new>
#include <vector>

#include "ctx.hpp"
#include "kernels.cuh"
#include "program.hpp"

using namespace mdim;

namespace {

// The k_eval kernel of instantiation `variant` (Plan::variant), or nullptr if the four k_eval_*.cu lists do not add up to the
// planner's table.
EvalKernel eval_kernel(int variant) {
    static const std::vector<EvalKernel> all = [] {
        std::vector<EvalKernel> v;
        for (auto part : {eval_kernels_s32_static, eval_kernels_s64_static, eval_kernels_s32_interp, eval_kernels_s64_interp}) {
            int n = 0;
            const EvalKernel* k = part(&n);
            v.insert(v.end(), k, k + n);
        }
        if ((int)v.size() != kNumEvalVariants) v.clear();
        return v;
    }();
    return variant >= 0 && variant < (int)all.size() ? all[variant] : nullptr;
}

bool plan_can_fail(const Plan& p) {
    if (p.kind != KK_GENERIC && p.kind != KK_STREAM) return false;
    for (int i = 0; i < p.prog.n_instr; ++i) {
        const Instr& I = p.prog.instr[i];
        if (I.opc == OPC_GATHER) return true;
        if ((I.opc == OPC_BINARY || I.opc == OPC_FOLD_STEP) && (I.op == MDIM_DIV || I.op == MDIM_REM) && I.dtype != MDIM_F32 && I.dtype != MDIM_F64)
            return true;
    }
    return false;
}

// May this launch start before its predecessor in the stream has finished?  Yes iff nothing it reads was written, and
// nothing it writes was touched, by a kernel that may still be running.  Either way the launch is recorded.
bool may_skip_wait(mdim_ctx* ctx, const Plan& p, const void* out) {
    const bool usable = ctx->dep_tracking && pdl_enabled() && ctx->stream == ctx->own_stream && p.n_in_ranges >= 0;
    mdim_ctx::Touched mine[kMaxRanges + 2];
    int n = 0;
    if (p.n_in_ranges >= 0)
        for (int i = 0; i < p.n_in_ranges; ++i) mine[n++] = {p.in_range[i].lo, p.in_range[i].hi, false};
    mine[n++] = {(uint64_t)(uintptr_t)out, (uint64_t)(uintptr_t)out + p.out_elems * (uint64_t)p.out_esize, true};
    if (p.kind == KK_FOLD_SPLIT)  // its tickets and partials: a second split fold must wait for this one
        mine[n++] = {(uint64_t)(uintptr_t)ctx->split_scratch, (uint64_t)(uintptr_t)ctx->split_scratch + ctx->split_scratch_bytes, true};
    bool conflict = !usable || ctx->inflight.size() + (size_t)n > 256 || p.n_out > 1;  // several output runs: simply wait
    for (size_t k = 0; k < ctx->inflight.size() && !conflict; ++k) {
        const mdim_ctx::Touched& t = ctx->inflight[k];
        for (int i = 0; i < n; ++i)
            if ((t.write || mine[i].write) && mine[i].lo < t.hi && t.lo < mine[i].hi) { conflict = true; break; }
    }
    if (conflict) ctx->inflight.clear();  // this kernel waits, so everything before it will have completed
    if (p.n_out > 1) ctx->inflight.push_back({0, ~0ull, true});  // (its other runs are not in `mine`: conflicts with everything)
    else if (usable) ctx->inflight.insert(ctx->inflight.end(), mine, mine + n);
    else if (p.n_in_ranges < 0) ctx->inflight.push_back({0, ~0ull, true});  // untracked operands: conflicts with everything
    return !conflict;
}

int launch_eval(mdim_ctx* ctx, const Plan& p, void* out, ErrWord* err, bool explain, uint64_t explain_pos, bool nowait = false) {
    if (p.variant < 0) return set_error(ctx, MDIM_ERR_UNSUPPORTED, "no evaluator instantiation for this expression");
    const EvalKernel fn = eval_kernel(p.variant);
    if (!fn) return set_error(ctx, MDIM_ERR_INVALID, "the k_eval kernels do not match the planner's instantiation table");
    uint64_t g0 = 0, g1 = p.prog.n_vec;
    int grid;
    // an op tree without a pre-built signature is specialised on first use (jit.cu); else the interpreter runs
    void* jit = nullptr;
    int jit_level = 0;
    if (!(p.flags & (MDIM_COLLECT_NO_STATIC | MDIM_COLLECT_NO_JIT))) jit = jit_kernel_for(p, &jit_level, explain);
    if (jit) snprintf(ctx->last_kernel, sizeof ctx->last_kernel, "%s", jit_level == 2 ? "mdim_jit_kernel[ops+shape]" : "mdim_jit_kernel[ops]");
    else eval_variant_name(p.variant, ctx->last_kernel, sizeof ctx->last_kernel);
    Program q = p.prog;
    if (p.vec256_ok && ((uintptr_t)out % 32) == 0) q.flags |= PF_VEC256;
    if (nowait && !explain) q.flags |= PF_NOWAIT;
    if (explain) {
        q.flags |= PF_EXPLAIN;
        q.explain_pos = explain_pos;
        g0 = explain_pos / (uint64_t)p.vec;
        g1 = g0 + 1;
        grid = 1;
    } else {
        grid = (int)std::min<uint64_t>((g1 + kEvalThreads - 1) / kEvalThreads, 0x7fffffffull);
    }
    if (jit) {
        unsigned long long a0 = g0, a1 = g1;
        void* args[] = {(void*)&q, (void*)&out, (void*)&err, (void*)&a0, (void*)&a1};
        cudaLaunchConfig_t cfg; cudaLaunchAttribute attr;
        pdl_config(cfg, attr, dim3((unsigned)grid), dim3(kEvalThreads), 0, ctx->stream);
        CU(ctx, cudaLaunchKernelExC(&cfg, (const void*)jit, args));
    } else {
        CU(ctx, launch_pdl(fn, dim3((unsigned)grid), dim3(kEvalThreads), 0, ctx->stream, q, out, err, g0, g1));
    }
    ctx->launches++;
    CU(ctx, cudaGetLastError());
    return MDIM_OK;
}

// Scratch for k_fold_split of at least `bytes` (tickets included).  A new allocation waits for the stream (the old one may still
// be in use) and zeroes the tickets before any split fold reads them.
int ensure_split_scratch(mdim_ctx* ctx, size_t bytes) {
    if (bytes <= ctx->split_scratch_bytes) return MDIM_OK;
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->split_scratch) { CU(ctx, cudaFree(ctx->split_scratch)); ctx->split_scratch = nullptr; ctx->split_scratch_bytes = 0; }
    bytes = std::max<size_t>(bytes, (size_t)1 << 20);
    CU(ctx, cudaMalloc((void**)&ctx->split_scratch, bytes));
    CU(ctx, cudaMemsetAsync(ctx->split_scratch, 0, kSplitMaxOuts * sizeof(unsigned int), ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->split_scratch_bytes = bytes;
    ctx->inflight.clear();  // the stream is idle
    return MDIM_OK;
}

int launch_plan(mdim_ctx* ctx, const Plan& p, void* out, ErrWord* err) {
    if (p.kind == KK_EMPTY) return MDIM_OK;
    if (p.kind == KK_FOLD_SPLIT) {
        int st = ensure_split_scratch(ctx, fold_split_scratch_bytes(p.fs, ctx->sm_count));
        if (st) return st;
    }
    const bool nowait = may_skip_wait(ctx, p, out);
    const char* name;
    switch (p.kind) {
        case KK_TRANSPOSE: name = launch_transpose(p, out, nowait, ctx->stream, ctx->sm_count); break;
        case KK_FOLD_ROWS: name = launch_fold_rows(p, out, nowait, ctx->stream, ctx->sm_count); break;
        case KK_FOLD_COLS: name = launch_fold_cols(p, out, nowait, ctx->stream, ctx->sm_count); break;
        case KK_FOLD_SPLIT: name = launch_fold_split(p, out, nowait, ctx->stream, ctx->sm_count, ctx->split_scratch); break;
        default: return launch_eval(ctx, p, out, err, false, 0, nowait);
    }
    if (!name) return cuda_fail(ctx, cudaGetLastError(), "kernel launch");
    snprintf(ctx->last_kernel, sizeof ctx->last_kernel, "%s", name);
    ctx->launches++;
    CU(ctx, cudaGetLastError());
    return MDIM_OK;
}

// Fill ctx->last from a failed collect: rerun the failing element alone with PF_EXPLAIN.
int explain(mdim_ctx* ctx, const Plan& p, void* out, int slot, uint64_t pos) {
    ErrWord* d = ctx->d_err + slot;
    ErrWord* h = ctx->h_err + slot;
    memset(h, 0, sizeof *h);
    h->pos = ~0ull;
    CU(ctx, cudaMemcpyAsync(d, h, sizeof *h, cudaMemcpyHostToDevice, ctx->stream));
    int st = launch_eval(ctx, p, out, d, true, pos);
    if (st) return st;
    CU(ctx, cudaMemcpyAsync(h, d, sizeof *h, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    explain_failure(*h, pos, &ctx->last);
    // reset the slot for reuse
    h->pos = ~0ull; h->status = 0;
    CU(ctx, cudaMemcpyAsync(d, h, sizeof *h, cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return ctx->last.status;
}

// Wait for the stream and resolve every pending (fallible) collect in submission order.
int drain(mdim_ctx* ctx) {
    if (!ctx->pending.empty())
        CU(ctx, cudaMemcpyAsync(ctx->h_err, ctx->d_err, sizeof(ErrWord) * kErrSlots, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->inflight.clear();  // nothing is running any more
    int result = MDIM_OK;
    std::vector<Pending> pend;
    pend.swap(ctx->pending);
    ctx->next_slot = 0;
    for (Pending& pd : pend) {
        if (result == MDIM_OK && ctx->h_err[pd.slot].pos != ~0ull) {
            result = explain(ctx, *pd.plan, pd.out, pd.slot, ctx->h_err[pd.slot].pos);
            ctx->last.position += pd.pos_base;
        }
        else if (ctx->h_err[pd.slot].pos != ~0ull) {
            ctx->h_err[pd.slot].pos = ~0ull;
            cudaMemcpyAsync(ctx->d_err + pd.slot, ctx->h_err + pd.slot, sizeof(ErrWord), cudaMemcpyHostToDevice, ctx->stream);
        }
        delete pd.plan;
    }
    if (!pend.empty()) CU(ctx, cudaStreamSynchronize(ctx->stream));
    return result;
}

int env_int(const char* name, int dflt) {
    const char* e = getenv(name);
    return e && *e ? atoi(e) : dflt;
}

}  // namespace

extern "C" {

int mdim_abi_version(void) { return MDIM_ABI_VERSION; }

const char* mdim_status_string(int status) { return status_string(status); }

int mdim_init(int device, mdim_ctx** out) {
    if (!out) return MDIM_ERR_INVALID;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || device < 0 || device >= n) return MDIM_ERR_CUDA;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return MDIM_ERR_CUDA;
    if (prop.major != 10) return MDIM_ERR_CUDA;  // sm_100a SASS only: no other device can run it, and nothing else is tried
    mdim_ctx* ctx = new (std::nothrow) mdim_ctx();
    if (!ctx) return MDIM_ERR_NOMEM;
    memset(&ctx->last, 0, sizeof ctx->last);
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    ctx->cc_major = prop.major;
    ctx->cc_minor = prop.minor;
    ctx->hbm = prop.totalGlobalMem;
    ctx->dep_tracking = env_int("MDIM_DEP_TRACK", 1) != 0;
    ctx->host_chunk_bytes = (size_t)std::max(1, env_int("MDIM_HOST_CHUNK_MB", 128)) << 20;
    bool ok = cudaSetDevice(device) == cudaSuccess && cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking) == cudaSuccess &&
              cudaMalloc(&ctx->d_err, sizeof(ErrWord) * kErrSlots) == cudaSuccess &&
              cudaMallocHost(&ctx->h_err, sizeof(ErrWord) * kErrSlots) == cudaSuccess;
    if (ok) {
        ctx->stream = ctx->own_stream;
        for (int i = 0; i < kErrSlots; ++i) { memset(&ctx->h_err[i], 0, sizeof(ErrWord)); ctx->h_err[i].pos = ~0ull; }
        ok = cudaMemcpy(ctx->d_err, ctx->h_err, sizeof(ErrWord) * kErrSlots, cudaMemcpyHostToDevice) == cudaSuccess;
    }
    if (!ok) {
        if (ctx->d_err) cudaFree(ctx->d_err);
        if (ctx->h_err) cudaFreeHost(ctx->h_err);
        if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
        delete ctx;
        return MDIM_ERR_CUDA;
    }
    *out = ctx;
    return MDIM_OK;
}

int mdim_shutdown(mdim_ctx* ctx) {
    if (!ctx) return MDIM_ERR_INVALID;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    for (Pending& pd : ctx->pending) delete pd.plan;
    comm_destroy(ctx);
    HostPipe& hp = ctx->pipe;
    for (int i = 0; i < 2; ++i) {
        if (hp.up[i]) cudaEventDestroy(hp.up[i]);
        if (hp.done[i]) cudaEventDestroy(hp.done[i]);
        if (hp.down[i]) cudaEventDestroy(hp.down[i]);
    }
    if (hp.h2d) cudaStreamDestroy(hp.h2d);
    if (hp.d2h) cudaStreamDestroy(hp.d2h);
    if (hp.arena) cudaFree(hp.arena);
    if (ctx->split_scratch) cudaFree(ctx->split_scratch);
    cudaFree(ctx->d_err);
    cudaFreeHost(ctx->h_err);
    cudaStreamDestroy(ctx->own_stream);
    delete ctx;
    return MDIM_OK;
}

int mdim_set_stream(mdim_ctx* ctx, void* cuda_stream) {
    if (!ctx) return MDIM_ERR_INVALID;
    int st = drain(ctx);
    ctx->stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->own_stream;
    return st;
}

int mdim_get_stream(mdim_ctx* ctx, void** cuda_stream) {
    if (!ctx || !cuda_stream) return MDIM_ERR_INVALID;
    *cuda_stream = (void*)ctx->stream;
    return MDIM_OK;
}

int mdim_last_kernel(mdim_ctx* ctx, char* buf, size_t buf_len) {
    if (!ctx || !buf || !buf_len) return MDIM_ERR_INVALID;
    snprintf(buf, buf_len, "%s", ctx->last_kernel);
    return MDIM_OK;
}

int mdim_sync(mdim_ctx* ctx) {
    if (!ctx) return MDIM_ERR_INVALID;
    CU(ctx, cudaSetDevice(ctx->device));
    return drain(ctx);
}

int mdim_last_error(mdim_ctx* ctx, mdim_error_info* info) {
    if (!ctx || !info) return MDIM_ERR_INVALID;
    *info = ctx->last;
    return MDIM_OK;
}

uint64_t mdim_launch_count(mdim_ctx* ctx) { return ctx ? ctx->launches : 0; }

int mdim_device_info(mdim_ctx* ctx, int* sm_count, int* cc_major, int* cc_minor, size_t* hbm_bytes) {
    if (!ctx) return MDIM_ERR_INVALID;
    if (sm_count) *sm_count = ctx->sm_count;
    if (cc_major) *cc_major = ctx->cc_major;
    if (cc_minor) *cc_minor = ctx->cc_minor;
    if (hbm_bytes) *hbm_bytes = ctx->hbm;
    return MDIM_OK;
}

// ---- buffers --------------------------------------------------------------------------------------
int mdim_buf_alloc(mdim_ctx* ctx, size_t bytes, void** dptr) {
    if (!ctx || !dptr) return MDIM_ERR_INVALID;
    *dptr = nullptr;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaMalloc(dptr, bytes ? bytes : 16));
    return MDIM_OK;
}

int mdim_buf_free(mdim_ctx* ctx, void* dptr) {
    if (!ctx) return MDIM_ERR_INVALID;
    if (!dptr) return MDIM_OK;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    CU(ctx, cudaFree(dptr));
    return MDIM_OK;
}

int mdim_upload(mdim_ctx* ctx, void* dst_device, const void* src_host, size_t bytes) {
    if (!ctx || (bytes && (!dst_device || !src_host))) return MDIM_ERR_INVALID;
    if (!bytes) return MDIM_OK;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaMemcpyAsync(dst_device, src_host, bytes, cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return MDIM_OK;
}

int mdim_download(mdim_ctx* ctx, void* dst_host, const void* src_device, size_t bytes) {
    if (!ctx || (bytes && (!dst_host || !src_device))) return MDIM_ERR_INVALID;
    CU(ctx, cudaSetDevice(ctx->device));
    int st = drain(ctx);  // a failed async collect must not hand out its garbage silently
    if (st) return st;
    if (!bytes) return MDIM_OK;
    CU(ctx, cudaMemcpyAsync(dst_host, src_device, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return MDIM_OK;
}

int mdim_host_alloc(mdim_ctx* ctx, size_t bytes, void** hptr) {
    if (!ctx || !hptr) return MDIM_ERR_INVALID;
    *hptr = nullptr;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaHostAlloc(hptr, bytes ? bytes : 16, cudaHostAllocDefault));
    return MDIM_OK;
}

int mdim_host_free(mdim_ctx* ctx, void* hptr) {
    if (!ctx) return MDIM_ERR_INVALID;
    if (!hptr) return MDIM_OK;
    CU(ctx, cudaFreeHost(hptr));
    return MDIM_OK;
}

// ---- the hot path ---------------------------------------------------------------------------------
static int collect_planned(mdim_ctx* ctx, Plan* plan, void* out_device, uint32_t flags) {
    if (plan->kind == KK_EMPTY) return MDIM_OK;
    const bool fallible = plan_can_fail(*plan);
    int slot = 0;
    if (fallible) {
        if (ctx->next_slot >= kErrSlots) { int st = drain(ctx); if (st) return st; }
        slot = ctx->next_slot++;
    }
    int st = launch_plan(ctx, *plan, out_device, ctx->d_err + slot);
    if (st) return st;
    if (fallible) {
        Plan* copy = new (std::nothrow) Plan(*plan);
        if (!copy) return MDIM_ERR_NOMEM;
        ctx->pending.push_back(Pending{copy, out_device, slot, ctx->pos_base});
    }
    if (flags & MDIM_COLLECT_ASYNC) return MDIM_OK;
    return drain(ctx);
}

// Plan, then launch on the context's device.  One Plan is several KB: it lives on the heap.
static int collect(mdim_ctx* ctx, const mdim_expr* e, void* const* outs, int n_outs, uint32_t flags) {
    std::unique_ptr<Plan> plan(new (std::nothrow) Plan());
    if (!plan) return MDIM_ERR_NOMEM;
    char why[160];
    int st = plan_collect(e, flags, outs, n_outs, plan.get(), why, sizeof why);
    if (st) return set_error(ctx, st, why);
    if (plan->kind == KK_EMPTY) return MDIM_OK;
    cudaError_t ce = cudaSetDevice(ctx->device);
    if (ce != cudaSuccess) return cuda_fail(ctx, ce, "cudaSetDevice");
    return collect_planned(ctx, plan.get(), outs[0], flags);
}

int mdim_collect(mdim_ctx* ctx, const mdim_expr* e, void* out_device, uint32_t flags) {
    if (!ctx) return MDIM_ERR_INVALID;
    return collect(ctx, e, &out_device, 1, flags);
}

int mdim_collect_tuple(mdim_ctx* ctx, const mdim_expr* e, void* const* outs_device, int n_outs, uint32_t flags) {
    if (!ctx || !outs_device || n_outs < 1 || n_outs > MDIM_MAX_OUTS) return MDIM_ERR_INVALID;
    return collect(ctx, e, outs_device, n_outs, flags);
}

int mdim_plan_describe_nodevice(const mdim_expr* e, uint32_t flags, char* buf, size_t buf_len) {
    if (!buf || !buf_len) return MDIM_ERR_INVALID;
    std::unique_ptr<Plan> plan(new (std::nothrow) Plan());
    if (!plan) return MDIM_ERR_NOMEM;
    char why[160];
    int st = plan_expr(e, flags, plan.get(), why, sizeof why);
    if (st) snprintf(buf, buf_len, "%s", why);
    else if ((plan->kind == KK_GENERIC || plan->kind == KK_STREAM) && plan->variant >= 0) {
        const bool may_jit = plan->static_id < 0 && !(flags & (MDIM_COLLECT_NO_STATIC | MDIM_COLLECT_NO_JIT));
        const EvalVariant& v = kEvalVariants[plan->variant];
        snprintf(buf, buf_len, "%s [%s r%d%s]", plan->describe, v.name, v.maxr, may_jit ? ", specialised on first use" : "");
    } else snprintf(buf, buf_len, "%s", plan->describe);
    return st;
}

int mdim_jit_check_nodevice(const mdim_expr* e, uint32_t flags, char* log, size_t log_len) {
    std::unique_ptr<Plan> plan(new (std::nothrow) Plan());
    if (!plan) return MDIM_ERR_NOMEM;
    char why[160];
    int st = plan_expr(e, flags, plan.get(), why, sizeof why);
    if (st) { if (log && log_len) snprintf(log, log_len, "%s", why); return st; }
    return jit_compile_check(*plan, log, log_len);
}

int mdim_plan_describe(mdim_ctx* ctx, const mdim_expr* e, uint32_t flags, char* buf, size_t buf_len) {
    (void)ctx;
    return mdim_plan_describe_nodevice(e, flags, buf, buf_len);
}

// ---- peer memory ------------------------------------------------------------------------------------
int mdim_ipc_export(mdim_ctx* ctx, void* dptr, uint8_t handle[MDIM_IPC_HANDLE_BYTES]) {
    if (!ctx || !dptr || !handle) return MDIM_ERR_INVALID;
    static_assert(sizeof(cudaIpcMemHandle_t) <= MDIM_IPC_HANDLE_BYTES, "handle size");
    cudaIpcMemHandle_t h;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaIpcGetMemHandle(&h, dptr));
    memset(handle, 0, MDIM_IPC_HANDLE_BYTES);
    memcpy(handle, &h, sizeof h);
    return MDIM_OK;
}

int mdim_ipc_open(mdim_ctx* ctx, const uint8_t handle[MDIM_IPC_HANDLE_BYTES], void** dptr) {
    if (!ctx || !dptr || !handle) return MDIM_ERR_INVALID;
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof h);
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaIpcOpenMemHandle(dptr, h, cudaIpcMemLazyEnablePeerAccess));
    return MDIM_OK;
}

int mdim_ipc_close(mdim_ctx* ctx, void* dptr) {
    if (!ctx || !dptr) return MDIM_ERR_INVALID;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaIpcCloseMemHandle(dptr));
    return MDIM_OK;
}

}  // extern "C"


// ---- host-buffer form: Array::new(..) → collect → to_raw() (src/array.rs:28-30,54) ----------------
namespace {

struct HostBuf {       // one distinct host operand (several nodes may view the same Array)
    const char* base;  // host pointer as given in the descriptor
    int esize;
    int64_t lo, hi;    // element range [lo, hi) touched by any node
    bool chunked;      // every node walks it in disjoint slabs along iteration axis 0
    int64_t stride0;   // elements per step of axis 0 (chunked only)
    int64_t slab_lo, slab_hi;  // element range of ONE step of axis 0 relative to r*stride0 (chunked only)
    char* dev;         // resident copy (not chunked)
    char* stage[2];    // staging (chunked)
};

int ensure_pipe(mdim_ctx* ctx, size_t arena_bytes) {
    HostPipe& hp = ctx->pipe;
    if (!hp.h2d) {
        CU(ctx, cudaStreamCreateWithFlags(&hp.h2d, cudaStreamNonBlocking));
        CU(ctx, cudaStreamCreateWithFlags(&hp.d2h, cudaStreamNonBlocking));
        for (int i = 0; i < 2; ++i) {
            CU(ctx, cudaEventCreateWithFlags(&hp.up[i], cudaEventDisableTiming));
            CU(ctx, cudaEventCreateWithFlags(&hp.done[i], cudaEventDisableTiming));
            CU(ctx, cudaEventCreateWithFlags(&hp.down[i], cudaEventDisableTiming));
        }
    }
    if (arena_bytes > hp.arena_bytes) {
        if (hp.arena) { CU(ctx, cudaDeviceSynchronize()); CU(ctx, cudaFree(hp.arena)); hp.arena = nullptr; hp.arena_bytes = 0; }
        CU(ctx, cudaMalloc((void**)&hp.arena, arena_bytes));
        hp.arena_bytes = arena_bytes;
    }
    return MDIM_OK;
}

size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

}  // namespace

extern "C" int mdim_collect_host(mdim_ctx* ctx, const mdim_expr* e, void* out_host, uint32_t flags) {
    if (!ctx) return MDIM_ERR_INVALID;
    std::unique_ptr<Plan> plan(new (std::nothrow) Plan());  // validates the descriptor here, then plans each chunk
    if (!plan) return MDIM_ERR_NOMEM;
    char why[160];
    int st = plan_expr(e, flags, plan.get(), why, sizeof why);
    if (st) return set_error(ctx, st, why);
    if (plan->kind == KK_EMPTY) return MDIM_OK;
    if (!out_host) return set_error(ctx, MDIM_ERR_INVALID, "null output buffer");
    if (plan->n_out > 1) return set_error(ctx, MDIM_ERR_INVALID, "a tuple-typed root in a host collect (mdim_collect_tuple collects its runs)");
    CU(ctx, cudaSetDevice(ctx->device));
    st = drain(ctx);
    if (st) return st;

    const int total = e->rank + e->red_rank;
    const int root = e->n_nodes - 1;
    const int out_es = dtype_size(e->nodes[root].dtype);
    uint64_t row_elems = 1;
    for (int a = 1; a < e->rank; ++a) row_elems *= e->length[a];
    const uint64_t n0 = e->rank > 0 ? e->length[0] : 1;

    // ---- distinct host operands and how each is walked along axis 0 -------------------------------
    std::vector<HostBuf> bufs;
    std::vector<int> node_buf(e->n_nodes, -1);
    bool can_chunk = e->rank >= 1 && n0 >= 2;
    std::vector<AxisRange> ranges(e->n_nodes);
    node_axis_ranges(e, ranges.data());
    for (int i = 0; i < e->n_nodes; ++i) {
        const mdim_node& n = e->nodes[i];
        if (n.kind == MDIM_NODE_CONCAT && n.axis_a[0] == 0) can_chunk = false;  // range test on the chunked coordinate
        if (n.kind == MDIM_NODE_DIAG) {
            for (int p = 0; p < n.n_comp; ++p)
                if (n.axis_a[p] == 0 || n.axis_b[p] == 0) can_chunk = false;  // predicate on the chunked coordinate
            continue;
        }
        if (n.kind != MDIM_NODE_LEAF && n.kind != MDIM_NODE_GATHER) continue;
        if (n.n_peers > 1) return set_error(ctx, MDIM_ERR_INVALID, "peer-sharded source in a host collect");
        const ElemRange all = operand_reach(e, n, ranges[i], 0);
        int b = -1;
        for (size_t k = 0; k < bufs.size(); ++k) if (bufs[k].base == (const char*)n.data) b = (int)k;
        const int es = dtype_size(n.dtype);
        const bool slabbed = n.kind == MDIM_NODE_LEAF && n.stride[0] > 0;
        const ElemRange slab = slabbed ? operand_reach(e, n, ranges[i], 1) : ElemRange{0, 0};
        bool disjoint = slabbed && slab.hi - slab.lo <= n.stride[0];
        for (int a = 1; a < total && disjoint; ++a) if (n.stride[a] < 0) disjoint = false;
        if (b < 0) {
            HostBuf hb;
            memset(&hb, 0, sizeof hb);
            hb.base = (const char*)n.data; hb.esize = es; hb.lo = all.lo; hb.hi = all.hi;
            hb.chunked = disjoint; hb.stride0 = n.stride[0]; hb.slab_lo = slab.lo; hb.slab_hi = slab.hi;
            bufs.push_back(hb);
            b = (int)bufs.size() - 1;
        } else {
            HostBuf& hb = bufs[b];
            if (hb.esize != es) return set_error(ctx, MDIM_ERR_INVALID, "one host buffer viewed with two element sizes");
            hb.lo = std::min(hb.lo, all.lo); hb.hi = std::max(hb.hi, all.hi);
            if (hb.chunked && disjoint && hb.stride0 == n.stride[0]) {
                hb.slab_lo = std::min(hb.slab_lo, slab.lo); hb.slab_hi = std::max(hb.slab_hi, slab.hi);
                if (hb.slab_hi - hb.slab_lo > hb.stride0) hb.chunked = false;
            } else hb.chunked = false;
        }
        node_buf[i] = b;
    }
    for (const HostBuf& hb : bufs) if (hb.lo < 0) return set_error(ctx, MDIM_ERR_INVALID, "operand reaches before its base pointer");

    // ---- chunk geometry -----------------------------------------------------------------------------
    uint64_t per_row = row_elems * (uint64_t)out_es;
    for (const HostBuf& hb : bufs) if (hb.chunked) per_row += (uint64_t)hb.stride0 * hb.esize;
    uint64_t rows = std::max<uint64_t>(1, ctx->host_chunk_bytes / std::max<uint64_t>(per_row, 1));
    if (rows >= 4096) rows &= ~1023ull;  // keep chunk boundaries vector-aligned when axis 0 is also the innermost
    if (!can_chunk || rows >= n0) { rows = n0; can_chunk = false; }
    if (!can_chunk) for (HostBuf& hb : bufs) hb.chunked = false;
    const uint64_t n_chunks = (n0 + rows - 1) / rows;
    const int n_sets = n_chunks > 1 ? 2 : 1;

    // ---- arena layout ---------------------------------------------------------------------------------
    size_t need = 0;
    std::vector<size_t> off_res(bufs.size(), 0), off_stage(bufs.size(), 0);
    for (size_t k = 0; k < bufs.size(); ++k) {
        const HostBuf& hb = bufs[k];
        if (!hb.chunked) { off_res[k] = need; need = align_up(need + (size_t)(hb.hi - hb.lo) * hb.esize, 256); }
    }
    size_t set_bytes = 0;
    for (size_t k = 0; k < bufs.size(); ++k) {
        const HostBuf& hb = bufs[k];
        if (hb.chunked) {
            off_stage[k] = set_bytes;
            set_bytes = align_up(set_bytes + (size_t)((int64_t)(rows - 1) * hb.stride0 + (hb.slab_hi - hb.slab_lo)) * hb.esize, 256);
        }
    }
    const size_t off_out = set_bytes;
    set_bytes = align_up(set_bytes + (size_t)(rows * row_elems) * out_es, 256);
    const size_t sets_at = need;
    need += set_bytes * n_sets;
    st = ensure_pipe(ctx, need);
    if (st) return st;
    HostPipe& hp = ctx->pipe;
    for (size_t k = 0; k < bufs.size(); ++k) {
        bufs[k].dev = hp.arena + off_res[k];
        for (int s = 0; s < 2; ++s) bufs[k].stage[s] = hp.arena + sets_at + set_bytes * (s % n_sets) + off_stage[k];
    }

    // ---- resident operands: one upload, ahead of the first chunk ----------------------------------------
    cudaStream_t compute = ctx->stream;
    for (const HostBuf& hb : bufs)
        if (!hb.chunked) CU(ctx, cudaMemcpyAsync(hb.dev, hb.base + hb.lo * hb.esize, (size_t)(hb.hi - hb.lo) * hb.esize, cudaMemcpyHostToDevice, hp.h2d));

    std::vector<mdim_node> nodes(e->nodes, e->nodes + e->n_nodes);
    mdim_expr sub = *e;
    sub.nodes = nodes.data();
    // Issue chunk c: uploads on the h2d stream, the fused kernel on the compute stream, the
    // download on the d2h stream, double-buffered over two staging sets.
    auto run_chunk = [&](uint64_t c, bool pipelined) -> int {
        const int s = (int)(c % (uint64_t)n_sets);
        const uint64_t r0 = c * rows, r1 = std::min(n0, r0 + rows);
        // the staging set must no longer be read by chunk c-2's kernel
        if (pipelined && c >= (uint64_t)n_sets) CU(ctx, cudaStreamWaitEvent(hp.h2d, hp.done[s], 0));
        for (const HostBuf& hb : bufs)
            if (hb.chunked) {
                const int64_t first = (int64_t)r0 * hb.stride0 + hb.slab_lo;
                const int64_t count = (int64_t)(r1 - r0 - 1) * hb.stride0 + (hb.slab_hi - hb.slab_lo);
                CU(ctx, cudaMemcpyAsync(hb.stage[s], hb.base + first * hb.esize, (size_t)count * hb.esize, cudaMemcpyHostToDevice, hp.h2d));
            }
        CU(ctx, cudaEventRecord(hp.up[s], hp.h2d));
        // the chunk's expression: same nodes over device pointers, axis 0 restricted to [r0, r1)
        if (e->rank > 0) sub.length[0] = r1 - r0;
        for (int i = 0; i < e->n_nodes; ++i) {
            mdim_node& n = nodes[i];
            const mdim_node& src = e->nodes[i];
            if (src.kind == MDIM_NODE_IOTA) n.offset = src.offset + (int64_t)r0 * src.stride[0];
            const int b = node_buf[i];
            if (b < 0) continue;
            const HostBuf& hb = bufs[b];
            if (hb.chunked) { n.data = hb.stage[s]; n.offset = src.offset - hb.slab_lo; }
            else { n.data = hb.dev; n.offset = src.offset - hb.lo + (e->rank > 0 ? (int64_t)r0 * src.stride[0] : 0); }
        }
        char* out_dev = hp.arena + sets_at + set_bytes * s + off_out;
        CU(ctx, cudaStreamWaitEvent(compute, hp.up[s], 0));
        if (pipelined && c >= (uint64_t)n_sets) CU(ctx, cudaStreamWaitEvent(compute, hp.down[s], 0));
        void* outs[1] = {out_dev};
        int rc = plan_collect(&sub, flags, outs, 1, plan.get(), why, sizeof why);
        if (rc) return set_error(ctx, rc, why);
        ctx->pos_base = r0 * row_elems;
        rc = collect_planned(ctx, plan.get(), out_dev, pipelined ? (flags | MDIM_COLLECT_ASYNC) : (flags & ~MDIM_COLLECT_ASYNC));
        ctx->pos_base = 0;
        if (rc) return rc;
        CU(ctx, cudaEventRecord(hp.done[s], compute));
        CU(ctx, cudaStreamWaitEvent(hp.d2h, hp.done[s], 0));
        CU(ctx, cudaMemcpyAsync((char*)out_host + r0 * row_elems * out_es, out_dev, (size_t)((r1 - r0) * row_elems) * out_es, cudaMemcpyDeviceToHost, hp.d2h));
        CU(ctx, cudaEventRecord(hp.down[s], hp.d2h));
        return MDIM_OK;
    };
    int result = MDIM_OK;
    for (uint64_t c = 0; c < n_chunks && result == MDIM_OK; ++c) result = run_chunk(c, true);
    CU(ctx, cudaStreamSynchronize(hp.h2d));
    const int dst = drain(ctx);  // waits for the compute stream and surfaces device-side panics
    CU(ctx, cudaStreamSynchronize(hp.d2h));
    if (result == MDIM_OK) result = dst;
    if ((result == MDIM_ERR_OOB || result == MDIM_ERR_ARITH || result == MDIM_ERR_INVALID) && n_chunks > 1) {
        // The staging sets have been reused since the failing chunk ran, so the details recorded by
        // the explain pass may describe other data: replay that one chunk on its own.
        const uint64_t c = ctx->last.position / (rows * row_elems);
        CU(ctx, cudaDeviceSynchronize());
        result = run_chunk(std::min(c, n_chunks - 1), false);
        CU(ctx, cudaDeviceSynchronize());
        if (result == MDIM_OK) result = set_error(ctx, MDIM_ERR_INVALID, "device-side failure did not reproduce");
    }
    return result;
}
