// emu.cpp — TEST INFRASTRUCTURE (never linked into the product): compiles the product's host
// planner (plan.cpp) and the product's per-thread evaluator (exec.cuh, host mode) with g++ and runs
// the evaluator one "thread" at a time.  It lets the CPU-only test suite check descriptor ->
// Program lowering, coordinate decode, vector/broadcast/strided loads, predicates, gather and fold
// control flow, and error reporting against the oracle without a GPU.  Planning, the output checks
// and re-plan of a collect (plan_collect), the choice and name of the k_eval instantiation, and the
// text of a device-side failure are the library's own code; only the kernel table below is the
// emulator's: the host form of every instantiation, which runs where the GPU runs its k_eval.  The
// dedicated CUDA kernels (tiled transpose, row fold) have none; the generic program stands in for
// them here.
#include <stdlib.h>
#include <string.h>

#include <memory>

#include "../../multidimension_b200/csrc/exec.cuh"
#include "../../multidimension_b200/csrc/plan.cpp"

namespace mdim {
template <class Sig, class S, int V, int MAXD, bool WIDE, int MAXR>
static void run_all(const Program& P, void* out, ErrWord* err, uint64_t g0, uint64_t g1) {
    for (uint64_t g = g0; g < g1; ++g) eval_vector<Sig, S, V, MAXD, WIDE, MAXR>(P, out, err, g);
}

// Host form of kEvalVariants[i], from the same variants_*.inc lists in the same order.
static void (*const kHostKernels[])(const Program&, void*, ErrWord*, uint64_t, uint64_t) = {
#define X(Sig, S, V, MAXD, WIDE, MAXR) &run_all<Sig, S, V, MAXD, WIDE, MAXR>,
#include "../../multidimension_b200/csrc/variants_s32_static.inc"
#include "../../multidimension_b200/csrc/variants_s64_static.inc"
#include "../../multidimension_b200/csrc/variants_s32_interp.inc"
#include "../../multidimension_b200/csrc/variants_s64_interp.inc"
#undef X
};
static_assert(sizeof(kHostKernels) / sizeof(kHostKernels[0]) == sizeof(kEvalVariants) / sizeof(kEvalVariants[0]), "one host kernel per instantiation");
}  // namespace mdim

static char g_last_kernel[96];  // the instantiation the last mdim_emu_collect ran, named as mdim_last_kernel names it

// Name of instantiation i of the registry (the four variants_*.inc lists), MDIM_ERR_INVALID past the end.
extern "C" int mdim_emu_variant_name(int i, char* buf, size_t len) {
    if (i < 0 || i >= mdim::kNumEvalVariants) return MDIM_ERR_INVALID;
    mdim::eval_variant_name(i, buf, len);
    return MDIM_OK;
}

extern "C" int mdim_emu_last_kernel(char* buf, size_t len) {
    snprintf(buf, len, "%s", g_last_kernel);
    return MDIM_OK;
}

// The planner's magic numbers for q = umulhi(n, mul) >> shr (plan.cpp), so that tests can check them.
extern "C" void mdim_emu_find_divisor(uint32_t d, uint32_t* mul, uint32_t* shr) { mdim::find_divisor(d, mul, shr); }

static int emu_collect(const mdim_expr* e, void* const* outs, int n_outs, uint32_t flags, mdim_error_info* info, char* describe, size_t describe_len) {
    using namespace mdim;
    std::unique_ptr<Plan> plan(new Plan());
    char why[160];
    mdim_error_info scratch;
    if (!info) info = &scratch;
    memset(info, 0, sizeof *info);
    int st = plan_collect(e, flags, outs, n_outs, plan.get(), why, sizeof why);
    if (describe && describe_len) snprintf(describe, describe_len, "%s", st ? why : plan->describe);
    if (st) { info->status = st; snprintf(info->message, sizeof info->message, "%s", why); return st; }
    if (plan->kind == KK_EMPTY) return MDIM_OK;
    if (plan->variant < 0) return MDIM_ERR_UNSUPPORTED;
    eval_variant_name(plan->variant, g_last_kernel, sizeof g_last_kernel);
    const auto run = kHostKernels[plan->variant];
    ErrWord err;
    memset(&err, 0, sizeof err);
    err.pos = ~0ull;
    if (plan->vec256_ok && ((uintptr_t)outs[0] % 32) == 0) plan->prog.flags |= PF_VEC256;  // as mdim_collect does at launch
    run(plan->prog, outs[0], &err, 0, plan->prog.n_vec);
    if (err.pos == ~0ull) return MDIM_OK;
    const uint64_t pos = err.pos;
    Program q = plan->prog;
    q.flags |= PF_EXPLAIN;
    q.explain_pos = pos;
    memset(&err, 0, sizeof err);
    err.pos = ~0ull;
    const uint64_t item = pos / (uint64_t)plan->vec;
    run(q, outs[0], &err, item, item + 1);
    explain_failure(err, pos, info);
    return info->status;
}

extern "C" int mdim_emu_collect(const mdim_expr* e, void* out, uint32_t flags, mdim_error_info* info, char* describe, size_t describe_len) {
    return emu_collect(e, &out, 1, flags, info, describe, describe_len);
}

extern "C" int mdim_emu_collect_tuple(const mdim_expr* e, void* const* outs, int n_outs, uint32_t flags, mdim_error_info* info, char* describe, size_t describe_len) {
    return emu_collect(e, outs, n_outs, flags, info, describe, describe_len);
}
