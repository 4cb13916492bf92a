// Launch of the tensor-core rollout for ONE precision (included by lrds_tc_<precision>.cu so that the precisions
// compile in parallel): kernel selection by loop kind, staging level and compile-time traits.
#pragma once
#include "lrds_internal.h"
#include "lrds_rollout_tc.cuh"

namespace lrds {

// Configurations with a specialised LINEAR kernel (everything else runs the run-time-switched kernel):
//   LRDS: RDS with a mixture reference, exponential-integrator or DDPM-like update, mixture target, ScoreCtrl
//   PIS : Euler-Maruyama, no reference control, lattice target, ScoreCtrl
//   DDS : exponential integrator of Vargas et al., no reference control, lattice target, ScoreCtrl (Ito term at run time)
using TraitsLrds = LinearTraits<LRDS_UPDATE_AXPY, LRDS_ITO_SCALED, LRDS_DISTR_GMM, 1, 2, 1>;
using TraitsPis = LinearTraits<LRDS_UPDATE_EM, LRDS_ITO_EM, LRDS_DISTR_PHI4, 1, 0, 0>;
using TraitsDds = LinearTraits<LRDS_UPDATE_AXPY, -1, LRDS_DISTR_PHI4, 1, 0, 0>;

template <int KIND, int PREC, int STAGE, class TR>
int launch_one(const RolloutArgs& a, const TcPlan& p, cudaStream_t st) {
  return launch_tc(rollout_tc_kernel<KIND, PREC, STAGE, TR>, "tensor-core rollout", a, p, p.warps * 32, st, p.tmem_cols);
}

template <int PREC, int STAGE>
int launch_linear(const RolloutArgs& a, const TcPlan& p, cudaStream_t st) {
  if constexpr (STAGE > 0) {
    if (traits_match<TraitsLrds>(a.s)) return launch_one<LRDS_ROLLOUT_LINEAR, PREC, STAGE, TraitsLrds>(a, p, st);
  }
  if constexpr (STAGE > 0) {
    if (traits_match<TraitsPis>(a.s)) return launch_one<LRDS_ROLLOUT_LINEAR, PREC, STAGE, TraitsPis>(a, p, st);
    if (traits_match<TraitsDds>(a.s)) return launch_one<LRDS_ROLLOUT_LINEAR, PREC, STAGE, TraitsDds>(a, p, st);
  }
  return launch_one<LRDS_ROLLOUT_LINEAR, PREC, STAGE, RuntimeTraits>(a, p, st);
}

template <int PREC>
int launch_prec(const RolloutArgs& a, const TcPlan& p, cudaStream_t st) {
  switch (a.s.kind) {
    case LRDS_ROLLOUT_LINEAR:
      return p.staged == 2   ? launch_linear<PREC, 2>(a, p, st)
             : p.staged == 1 ? launch_linear<PREC, 1>(a, p, st)
                             : launch_linear<PREC, 0>(a, p, st);
    case LRDS_ROLLOUT_CMCD: return launch_one<LRDS_ROLLOUT_CMCD, PREC, 0, RuntimeTraits>(a, p, st);
    case LRDS_ROLLOUT_EUBO_LINEAR: return launch_one<LRDS_ROLLOUT_EUBO_LINEAR, PREC, 0, RuntimeTraits>(a, p, st);
    case LRDS_ROLLOUT_EUBO_CMCD: return launch_one<LRDS_ROLLOUT_EUBO_CMCD, PREC, 0, RuntimeTraits>(a, p, st);
  }
  return fail(LRDS_ERR_INVALID, "unknown rollout kind");
}

}  // namespace lrds
