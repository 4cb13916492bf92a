// The mixture tensor-core kernel (lrds_rollout_mix.cuh): no reference control (PIS / DDS over a mixture target), lattice target with a Gaussian reference (own translation unit: the
// configurations compile in parallel).
#include "lrds_internal.h"
#include "lrds_rollout_mix.cuh"

namespace lrds {

int launch_mix_c(int cfg, const RolloutArgs& a, const TcPlan& p, cudaStream_t st) {
  switch (cfg) {
    case 7: return launch_mix_cfg<MixCfg<false, 1, 0, true>>(a, p, st);
    case 8: return launch_mix_cfg<MixCfg<false, 1, 0, false>>(a, p, st);
    case 10: return launch_mix_cfg<MixCfg<false, 1, 0, true, true>>(a, p, st);
    default: return launch_mix_cfg<MixCfg<false, 2, 1, false>>(a, p, st);
  }
}
}  // namespace lrds
