// emu.cpp — TEST INFRASTRUCTURE (never linked into the product): compiles the product's host
// planner (plan.cpp) and the product's per-thread evaluator (exec.cuh, host mode) with g++ and runs
// the evaluator one "thread" at a time.  It lets the CPU-only test suite check descriptor ->
// Program lowering, coordinate decode, vector/broadcast/strided loads, predicates, gather and fold
// control flow, and error reporting against the oracle without a GPU.  Every evaluator instantiation
// the library builds (pre-built signatures through run_static, the interpreter through run_interp)
// has a host form here, picked by the library's rules.  The dedicated CUDA kernels (tiled transpose,
// row fold) have none; the generic program stands in for them here.
#include <stdlib.h>
#include <string.h>

#include "../../multidimension_b200/csrc/sigs.hpp"
#include "../../multidimension_b200/csrc/plan.cpp"

namespace mdim {
template <class Sig, class S, int V, int MAXD, bool WIDE, int MAXR>
static void run_all(const Program& P, void* out, ErrWord* err, uint64_t g0, uint64_t g1) {
    for (uint64_t g = g0; g < g1; ++g) eval_vector<Sig, S, V, MAXD, WIDE, MAXR>(P, out, err, g);
}

// The host form of every instantiation the library builds, in the library's registry order (api.cu: registry()), from the
// same variants_*.inc lists: a pre-built signature runs run_static here exactly where the GPU runs it.
struct HostVariant {
    const char* name;
    int slot_bytes, vec, max_depth, wide, maxr;
    const SigInstr* sig;  // nullptr = interpreter
    int sig_n;
    void (*fn)(const Program&, void*, ErrWord*, uint64_t, uint64_t);
};
template <class Sig> constexpr const SigInstr* sig_code() { if constexpr (Sig::n > 0) return Sig::code; else return nullptr; }

static const HostVariant kVariants[] = {
#define X(Sig, S, V, MAXD, WIDE, MAXR) \
    {#Sig, (int)sizeof(S), V, MAXD, WIDE ? 1 : 0, MAXR, sig_code<Sig>(), Sig::n, &run_all<Sig, S, V, MAXD, WIDE, MAXR>},
#include "../../multidimension_b200/csrc/variants_s32_static.inc"
#include "../../multidimension_b200/csrc/variants_s64_static.inc"
#include "../../multidimension_b200/csrc/variants_s32_interp.inc"
#include "../../multidimension_b200/csrc/variants_s64_interp.inc"
#undef X
};
static const int kNumVariants = (int)(sizeof(kVariants) / sizeof(kVariants[0]));

// api.cu's lookup and selection rules, restated over kVariants
static bool sig_matches(const HostVariant& v, const char* sig, int sig_len) {
    if (!v.sig || v.sig_n * 4 != sig_len) return false;
    for (int i = 0; i < v.sig_n; ++i) {
        const unsigned char* s = (const unsigned char*)sig + 4 * i;
        if (v.sig[i].opc != s[0] || v.sig[i].dtype != s[1]) return false;
        const int opc = v.sig[i].opc;
        if ((opc == OPC_LEAF_VEC || opc == OPC_LEAF_BCAST || opc == OPC_LEAF_STRIDED) && v.sig[i].aux != s[3]) return false;
        if ((opc == OPC_BINARY || opc == OPC_UNARY || opc == OPC_FOLD_STEP) && (v.sig[i].op != s[2] || v.sig[i].aux != s[3])) return false;
        if (opc == OPC_GATHER && v.sig[i].aux != s[3]) return false;
    }
    return true;
}

int find_static_signature(const char* sig, int sig_len, int slot_bytes, int vec, int need_maxr, int wide) {
    if (wide) return -1;
    for (int i = 0; i < kNumVariants; ++i)
        if (kVariants[i].slot_bytes == slot_bytes && kVariants[i].vec == vec && kVariants[i].maxr >= need_maxr && !kVariants[i].wide &&
            sig_matches(kVariants[i], sig, sig_len))
            return i;
    return -1;
}

static const HostVariant* select_variant(const Plan& p) {
    const int need = p.kind == KK_STREAM ? 1 : (p.n_axes < 1 ? 1 : p.n_axes);
    const HostVariant* best = nullptr;
    if (p.static_id >= 0 && !p.wide) {
        for (const HostVariant& v : kVariants) {
            if (v.slot_bytes != p.slot_bytes || v.vec != p.vec || v.wide || v.maxr < need || !sig_matches(v, p.sig, p.sig_len)) continue;
            if (!best || v.maxr < best->maxr) best = &v;
        }
        if (best) return best;
    }
    for (const HostVariant& v : kVariants) {
        if (v.sig || v.slot_bytes != p.slot_bytes || v.vec != p.vec || v.wide != p.wide || v.maxr < need || v.max_depth < p.max_depth) continue;
        if (!best || v.maxr < best->maxr || (v.maxr == best->maxr && v.max_depth < best->max_depth)) best = &v;
    }
    return best;
}
}  // namespace mdim

static char g_last_kernel[96];  // the instantiation the last mdim_emu_collect ran, named as mdim_last_kernel names it

static void variant_name(const mdim::HostVariant& v, char* buf, size_t len) {
    snprintf(buf, len, "k_eval<%s,s%d,v%d,d%d%s,r%d>", v.sig ? v.name : "interp", v.slot_bytes * 8, v.vec, v.max_depth, v.wide ? ",wide" : "", v.maxr);
}

// Name of instantiation i of the registry (the four variants_*.inc lists), MDIM_ERR_INVALID past the end.
extern "C" int mdim_emu_variant_name(int i, char* buf, size_t len) {
    if (i < 0 || i >= mdim::kNumVariants) return MDIM_ERR_INVALID;
    variant_name(mdim::kVariants[i], buf, len);
    return MDIM_OK;
}

extern "C" int mdim_emu_last_kernel(char* buf, size_t len) {
    snprintf(buf, len, "%s", g_last_kernel);
    return MDIM_OK;
}

// The planner's magic numbers for q = umulhi(n, mul) >> shr (plan.cpp), so that tests can check them.
extern "C" void mdim_emu_find_divisor(uint32_t d, uint32_t* mul, uint32_t* shr) { mdim::find_divisor(d, mul, shr); }

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
    bool aligned16 = ((uintptr_t)out % 16) == 0;
    for (int k = 1; k < plan->n_out && g_more_outs; ++k) aligned16 = aligned16 && ((uintptr_t)g_more_outs[k] % 16) == 0;
    if (!aligned16 && plan->vec > 1) {  // an element-aligned output: plan again with scalar stores, as mdim_collect does
        st = plan_expr(e, flags | kPlanScalarOut, plan, why, sizeof why);
        if (describe && describe_len) snprintf(describe, describe_len, "%s", st ? why : plan->describe);
        if (st) { if (info) { info->status = st; snprintf(info->message, sizeof info->message, "%s", why); } delete plan; return st; }
    }
    const HostVariant* v = select_variant(*plan);
    if (!v) { delete plan; return MDIM_ERR_UNSUPPORTED; }
    variant_name(*v, g_last_kernel, sizeof g_last_kernel);
    if (plan->n_out > 1) {
        if (!g_more_outs) { delete plan; return MDIM_ERR_INVALID; }
        for (int k = 1; k < plan->n_out; ++k) plan->prog.out_more[k - 1] = g_more_outs[k];
    }
    ErrWord err;
    memset(&err, 0, sizeof err);
    err.pos = ~0ull;
    if (plan->vec256_ok && ((uintptr_t)out % 32) == 0) plan->prog.flags |= PF_VEC256;  // as mdim_collect does at launch
    v->fn(plan->prog, out, &err, 0, plan->prog.n_vec);
    if (st == MDIM_OK && err.pos != ~0ull) {
        const uint64_t pos = err.pos;
        Program q = plan->prog;
        q.flags |= PF_EXPLAIN;
        q.explain_pos = pos;
        memset(&err, 0, sizeof err);
        err.pos = ~0ull;
        const uint64_t item = pos / (uint64_t)plan->vec;
        v->fn(q, out, &err, item, item + 1);
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
