// k_eval_s64_static.cu — instantiations of the fused evaluator with 64-bit value slots (sm_100a).
#include "kernels.cuh"
#include "sigs.hpp"

namespace mdim {

template <class Sig> constexpr const SigInstr* sig_code() { if constexpr (Sig::n > 0) return Sig::code; else return nullptr; }

static const EvalVariant kVariants[] = {
#define X(Sig, S, V, MAXD, WIDE, MAXR) \
    {#Sig, (int)sizeof(S), V, MAXD, WIDE ? 1 : 0, MAXR, sig_code<Sig>(), Sig::n, &k_eval<Sig, S, V, MAXD, WIDE, MAXR>},
#include "variants_s64_static.inc"
#undef X
};

const EvalVariant* eval_variants_s64_static(int* n) {
    *n = (int)(sizeof(kVariants) / sizeof(kVariants[0]));
    return kVariants;
}

}  // namespace mdim
