// Tensor-core rollout kernels of one precision (own translation unit: the precisions compile in parallel).
#include "lrds_tc_launch.cuh"

namespace lrds {
template int launch_prec<LRDS_PRECISION_BF16>(const RolloutArgs&, const TcPlan&, cudaStream_t);
}  // namespace lrds
