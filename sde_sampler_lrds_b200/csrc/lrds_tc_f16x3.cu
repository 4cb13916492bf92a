// Tensor-core rollout kernels of one precision (own translation unit: the precisions compile in parallel), plus the
// kernel that also runs the mixture-score contractions on the tensor core (lrds_rollout_mix.cuh).
#include "lrds_rollout_cmcd_tc.cuh"
#include "lrds_rollout_lin.cuh"
#include "lrds_rollout_mix.cuh"
#include "lrds_tc_launch.cuh"

namespace lrds {
template int launch_prec<LRDS_PRECISION_F16X3>(const RolloutArgs&, const TcPlan&, cudaStream_t);

int launch_lin_f16x3(const RolloutArgs& a, const TcPlan& p, cudaStream_t st) {
  const bool em = a.s.update_form == LRDS_UPDATE_EM, phi4 = a.s.target.kind == LRDS_DISTR_PHI4;
  auto kernel = em ? (phi4 ? rollout_lin_kernel<LRDS_PRECISION_F16X3, true, true> : rollout_lin_kernel<LRDS_PRECISION_F16X3, true, false>)
                   : (phi4 ? rollout_lin_kernel<LRDS_PRECISION_F16X3, false, true> : rollout_lin_kernel<LRDS_PRECISION_F16X3, false, false>);
  return launch_tc(kernel, "reference-free tensor-core rollout", a, p, p.warps * 32, st, p.tmem_cols);
}

int launch_cmcd_tc_f16x3(const RolloutArgs& a, const TcPlan& p, cudaStream_t st) {
  auto kernel = a.s.kind == LRDS_ROLLOUT_EUBO_CMCD ? rollout_cmcd_tc_kernel<LRDS_PRECISION_F16X3, 1>
                : a.s.kind == LRDS_ROLLOUT_LINEAR  ? rollout_cmcd_tc_kernel<LRDS_PRECISION_F16X3, 2>
                                                    : rollout_cmcd_tc_kernel<LRDS_PRECISION_F16X3, 0>;
  return launch_tc(kernel, "CMCD tensor-core rollout", a, p, p.warps * 32, st, p.tmem_cols);
}

}  // namespace lrds
