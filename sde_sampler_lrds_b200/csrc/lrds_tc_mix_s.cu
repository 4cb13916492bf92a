// The small-batch variant of the mixture tensor-core kernel (lrds_rollout_mix_small.cuh), own translation unit.
#include "lrds_internal.h"
#include "lrds_rollout_cmcd_mix.cuh"
#include "lrds_rollout_mix_small.cuh"

namespace lrds {

int launch_mix_small_f16x3(const RolloutArgs& a, const TcPlan& p, cudaStream_t st) {
  return launch_tc(rollout_mix_small_kernel<LRDS_PRECISION_F16X3>, "small-batch mixture rollout", a, p, p.warps * 32, st);
}

int launch_cmcd_mix_f16x3(const RolloutArgs& a, const TcPlan& p, cudaStream_t st) {
  return launch_tc(rollout_cmcd_mix_kernel<LRDS_PRECISION_F16X3>, "CMCD mixture rollout", a, p, p.warps * 32, st, p.tmem_cols);
}
}  // namespace lrds

#ifdef LRDS_MIX_TIMING
extern "C" int lrds_debug_mix_small_timing(unsigned long long* host_out) {  // tools only
  return (int)cudaMemcpyFromSymbol(host_out, lrds::g_mix_timing, sizeof(lrds::g_mix_timing));
}
#endif
