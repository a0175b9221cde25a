// k_eval_s32_static.cu — instantiations of the fused evaluator with 32-bit value slots (sm_100a).
#include "kernels.cuh"
#include "sigs.hpp"

namespace mdim {

static const EvalKernel kKernels[] = {
#define X(Sig, S, V, MAXD, WIDE, MAXR) &k_eval<Sig, S, V, MAXD, WIDE, MAXR>,
#include "variants_s32_static.inc"
#undef X
};

const EvalKernel* eval_kernels_s32_static(int* n) {
    *n = (int)(sizeof(kKernels) / sizeof(kKernels[0]));
    return kKernels;
}

}  // namespace mdim
