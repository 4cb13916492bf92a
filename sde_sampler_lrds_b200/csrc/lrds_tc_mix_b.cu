// The mixture tensor-core kernel (lrds_rollout_mix.cuh): lattice target / ClippedCtrl / Euler-Maruyama with a mixture reference (own translation unit: the
// configurations compile in parallel).
#include "lrds_internal.h"
#include "lrds_rollout_mix.cuh"

namespace lrds {

int launch_mix_b(int cfg, const RolloutArgs& a, const TcPlan& p, cudaStream_t st) {
  switch (cfg) {
    case 4: return launch_mix_cfg<MixCfg<false, 2, 2, false>>(a, p, st);
    case 5: return launch_mix_cfg<MixCfg<false, 0, 2, false>>(a, p, st);
    default: return launch_mix_cfg<MixCfg<false, 1, 2, true>>(a, p, st);
  }
}
}  // namespace lrds
