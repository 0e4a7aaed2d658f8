// mcmcn_sets_logit.cu -- kernel instantiations (see mcmcn_registry.h).
#include <cuda_runtime.h>
#include "mcmcn_registry.h"
// FP32 production kernels: chains per lane and resident CTAs per SM.  Measured on BASELINE config 5 (ms per
// launch, partial / no pooling; profiles/experiments/r2_logit_occupancy_ab.log): 4 chains x 3 CTAs (168
// registers) 1.756 / 2.004; 4 x 6: 1.586 / 1.728; 4 x 7: 1.554 / 1.778; 2 x 8 (64 registers, no spills)
// 1.560 / 1.723; 2 x 9: 1.590 / 1.650; 2 x 10: 1.608 / 1.679.  The observation loop is bound by the MUFU
// pipe, the decision phases between two loops by latency: resident warps are what overlaps the two.
namespace mcmcn {
static const KernelSet kSets[] = {
    MCMCN_SET_MB(MCMCN_OBJ_BERNOULLI_LOGIT, Logit, 0, 32, float, 2, 8),     // 2 chains per lane x 8 CTAs per SM
    MCMCN_SET(MCMCN_OBJ_BERNOULLI_LOGIT, Logit, 0, 64, double, 2),
};
const KernelSet* sets_logit(int* n) { *n = (int)(sizeof(kSets) / sizeof(kSets[0])); return kSets; }
}  // namespace mcmcn
