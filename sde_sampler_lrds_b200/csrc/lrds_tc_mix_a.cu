// The mixture tensor-core kernel (lrds_rollout_mix.cuh): the benchmark configuration and its EUBO / Gaussian-reference variants (own translation unit: the
// configurations compile in parallel).
#include "lrds_internal.h"
#include "lrds_rollout_mix.cuh"

namespace lrds {

int launch_mix_b(int cfg, const RolloutArgs& a, const TcPlan& p, cudaStream_t st);  // lrds_tc_mix_b.cu
int launch_mix_c(int cfg, const RolloutArgs& a, const TcPlan& p, cudaStream_t st);  // lrds_tc_mix_c.cu

int launch_mix_f16x3(const RolloutArgs& a, const TcPlan& p, cudaStream_t st) {
  const int cfg = mix_tc_config(a.s);
  switch (cfg) {  // MixCfg<EUBO, TGT, REF, EM>
    case 0: return launch_mix_cfg<MixBench>(a, p, st);
    case 1: return launch_mix_cfg<MixCfg<true, 1, 2, false>>(a, p, st);
    case 2: return launch_mix_cfg<MixCfg<false, 1, 1, false>>(a, p, st);
    case 3: return launch_mix_cfg<MixCfg<false, 1, 1, true>>(a, p, st);
    case 4: case 5: case 6: return launch_mix_b(cfg, a, p, st);
    case 7: case 8: case 9: case 10: return launch_mix_c(cfg, a, p, st);
  }
  return fail(LRDS_ERR_UNSUPPORTED, "mixture tensor-core rollout: configuration not built");
}
}  // namespace lrds

#ifdef LRDS_MIX_TIMING
extern "C" int lrds_debug_mix_timing(unsigned long long* host_out) {  // tools only: 2 CTAs x 16 warps x 16 phase counters
  return (int)cudaMemcpyFromSymbol(host_out, lrds::g_mix_timing, sizeof(lrds::g_mix_timing));
}
#endif
