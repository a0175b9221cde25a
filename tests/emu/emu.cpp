// emu.cpp — TEST INFRASTRUCTURE (never linked into the product): compiles the product's host
// planner (plan.cpp) and the product's per-thread evaluator (exec.cuh, host mode) with g++ and runs
// the evaluator one "thread" at a time.  It lets the CPU-only test suite check descriptor ->
// Program lowering, coordinate decode, vector/broadcast/strided loads, predicates, gather and fold
// control flow, and error reporting against the oracle without a GPU.  The dedicated CUDA kernels
// (tiled transpose, row fold) have no host form; the generic program stands in for them here.
#include <stdlib.h>
#include <string.h>

#include "../../multidimension_b200/csrc/exec.cuh"
#include "../../multidimension_b200/csrc/plan.cpp"

namespace mdim {
// No static signatures on the host.
int find_static_signature(const char*, int, int, int, int, int) { return -1; }

template <class S, int V, int MAXD, bool WIDE, int MAXR>
static void run_all(const Program& P, void* out, ErrWord* err, uint64_t g0, uint64_t g1) {
    for (uint64_t g = g0; g < g1; ++g) eval_vector<NoSig, S, V, MAXD, WIDE, MAXR>(P, out, err, g);
}

// the same MAXR choices the device registry offers (variants_s32.inc / variants_s64.inc), plus the
// stream form MAXR = 1 that the static signatures use
template <class S, int V, int MAXD, bool WIDE>
static void run_r(const Plan& p, const Program& P, void* out, ErrWord* err, uint64_t g0, uint64_t g1) {
    const int need = p.kind == KK_STREAM ? 1 : (p.n_axes < 1 ? 1 : p.n_axes);
    if (need <= 1) run_all<S, V, MAXD, WIDE, 1>(P, out, err, g0, g1);
    else if (need <= 3) run_all<S, V, MAXD, WIDE, 3>(P, out, err, g0, g1);
    else run_all<S, V, MAXD, WIDE, 8>(P, out, err, g0, g1);
}

template <class S, int V, int MAXD>
static void run_w(const Plan& p, const Program& P, void* out, ErrWord* err, uint64_t g0, uint64_t g1) {
    if (p.wide) run_r<S, V, MAXD, true>(p, P, out, err, g0, g1);
    else run_r<S, V, MAXD, false>(p, P, out, err, g0, g1);
}

static int run(const Plan& p, const Program& P, void* out, ErrWord* err, uint64_t g0, uint64_t g1) {
    if (p.slot_bytes == 4) {
        if (p.vec == 8 && p.max_depth <= 4) run_w<uint32_t, 8, 4>(p, P, out, err, g0, g1);
        else if (p.vec == 4 && p.max_depth <= 4) run_w<uint32_t, 4, 4>(p, P, out, err, g0, g1);
        else if (p.vec == 1 && p.max_depth <= 4) run_w<uint32_t, 1, 4>(p, P, out, err, g0, g1);
        else if (p.vec == 1) run_w<uint32_t, 1, 8>(p, P, out, err, g0, g1);
        else return MDIM_ERR_UNSUPPORTED;
    } else {
        if (p.vec == 4 && p.max_depth <= 4) run_w<uint64_t, 4, 4>(p, P, out, err, g0, g1);
        else if (p.vec == 2 && p.max_depth <= 4) run_w<uint64_t, 2, 4>(p, P, out, err, g0, g1);
        else if (p.vec == 1 && p.max_depth <= 4) run_w<uint64_t, 1, 4>(p, P, out, err, g0, g1);
        else if (p.vec == 1) run_w<uint64_t, 1, 8>(p, P, out, err, g0, g1);
        else return MDIM_ERR_UNSUPPORTED;
    }
    return MDIM_OK;
}
}  // namespace mdim

static void* const* g_more_outs = nullptr;  // set by mdim_emu_collect_tuple for the duration of one call

extern "C" int mdim_emu_collect(const mdim_expr* e, void* out, uint32_t flags, mdim_error_info* info, char* describe, size_t describe_len);
extern "C" int mdim_emu_collect_tuple(const mdim_expr* e, void* const* outs, int n_outs, uint32_t flags, mdim_error_info* info, char* describe, size_t describe_len) {
    g_more_outs = outs;
    const int st = mdim_emu_collect(e, outs[0], flags, info, describe, describe_len);
    g_more_outs = nullptr;
    (void)n_outs;
    return st;
}

extern "C" int mdim_emu_collect(const mdim_expr* e, void* out, uint32_t flags, mdim_error_info* info, char* describe, size_t describe_len) {
    using namespace mdim;
    Plan* plan = new Plan();
    char why[160];
    if (info) memset(info, 0, sizeof *info);
    int st = plan_expr(e, flags, plan, why, sizeof why);
    if (describe && describe_len) snprintf(describe, describe_len, "%s", st ? why : plan->describe);
    if (st) { if (info) { info->status = st; snprintf(info->message, sizeof info->message, "%s", why); } delete plan; return st; }
    if (plan->kind == KK_EMPTY) { delete plan; return MDIM_OK; }
    if (plan->n_out > 1) {
        if (!g_more_outs) { delete plan; return MDIM_ERR_INVALID; }
        for (int k = 1; k < plan->n_out; ++k) plan->prog.out_more[k - 1] = g_more_outs[k];
    }
    ErrWord err;
    memset(&err, 0, sizeof err);
    err.pos = ~0ull;
    if (plan->vec256_ok && ((uintptr_t)out % 32) == 0) plan->prog.flags |= PF_VEC256;  // as mdim_collect does at launch
    st = run(*plan, plan->prog, out, &err, 0, plan->prog.n_vec);
    if (st == MDIM_OK && err.pos != ~0ull) {
        const uint64_t pos = err.pos;
        Program q = plan->prog;
        q.flags |= PF_EXPLAIN;
        q.explain_pos = pos;
        memset(&err, 0, sizeof err);
        err.pos = ~0ull;
        const uint64_t item = pos / (uint64_t)plan->vec;
        run(*plan, q, out, &err, item, item + 1);
        st = err.status ? err.status : MDIM_ERR_INVALID;
        if (info) {
            info->status = st; info->node = err.node; info->position = pos; info->value = err.value; info->bound = err.bound;
            info->component = err.component;
            if (st == MDIM_ERR_OOB) snprintf(info->message, sizeof info->message, "Index %llu is out of bounds for size %llu",
                                             (unsigned long long)err.value, (unsigned long long)err.bound);
            else if (st == MDIM_ERR_ARITH) snprintf(info->message, sizeof info->message, "attempt to divide by zero or with overflow");
        }
    }
    delete plan;
    return st;
}
