// Tensor-core rollout: launch planning, dispatch to the per-precision translation units and the weight-image packer.
#include <cuda_runtime.h>

#include <cstdlib>

#include "lrds_internal.h"
#include "lrds_rollout_cmcd_tc.cuh"
#include "lrds_rollout_lin.cuh"
#include "lrds_rollout_cmcd_mix.cuh"
#include "lrds_rollout_mix.cuh"
#include "lrds_rollout_mix_small.cuh"

namespace lrds {

template <int PREC>
int launch_prec(const RolloutArgs& a, const TcPlan& p, cudaStream_t st);  // lrds_tc_<precision>.cu
extern template int launch_prec<LRDS_PRECISION_TF32X3>(const RolloutArgs&, const TcPlan&, cudaStream_t);
extern template int launch_prec<LRDS_PRECISION_BF16>(const RolloutArgs&, const TcPlan&, cudaStream_t);
extern template int launch_prec<LRDS_PRECISION_TF32>(const RolloutArgs&, const TcPlan&, cudaStream_t);
extern template int launch_prec<LRDS_PRECISION_F16X3>(const RolloutArgs&, const TcPlan&, cudaStream_t);

int launch_mix_f16x3(const RolloutArgs& a, const TcPlan& p, cudaStream_t st);      // lrds_tc_f16x3.cu
int launch_mix_small_f16x3(const RolloutArgs& a, const TcPlan& p, cudaStream_t st);  // lrds_tc_mix_s.cu
int launch_cmcd_mix_f16x3(const RolloutArgs& a, const TcPlan& p, cudaStream_t st);   // lrds_tc_mix_s.cu
int launch_cmcd_tc_f16x3(const RolloutArgs& a, const TcPlan& p, cudaStream_t st);  // lrds_tc_f16x3.cu
int launch_lin_f16x3(const RolloutArgs& a, const TcPlan& p, cudaStream_t st);      // lrds_tc_f16x3.cu

int launch_rollout_tc(const RolloutArgs& a, cudaStream_t st) {
  const lrds_spec& s = a.s;
  if (!s.mlp.tc_image) return fail(LRDS_ERR_INVALID, "mlp.tc_image is NULL: pack the weights with lrds_pack_mlp_tc for this precision first");
  const DeviceLimits dl = device_limits();
  const int cap = dl.smem_optin, sms = dl.sms;
  TcPlan p{};
  const char* why = "";
  // latency-bound batches (LRDS_MIX_SMALL=0: tests and A/B timings run them through the throughput kernel)
  const char* small_env = getenv("LRDS_MIX_SMALL");
  if (!(small_env && small_env[0] == '0') && plan_rollout_mix_small(s, cap, sms, &p))
    return launch_mix_small_f16x3(a, p, st);
  if (plan_rollout_mix(s, cap, sms, &p)) return launch_mix_f16x3(a, p, st);
  if (plan_rollout_cmcd_tc(s, cap, &p)) return launch_cmcd_tc_f16x3(a, p, st);
  if (plan_rollout_cmcd_mix(s, cap, sms, &p)) return launch_cmcd_mix_f16x3(a, p, st);
  if (plan_rollout_lin(s, cap, sms, &p)) return launch_lin_f16x3(a, p, st);
  if (int r = plan_rollout_tc(s, cap, sms, &p, &why))
    return fail(r, "tensor-core rollout does not fit (d=%d, precision %d): %s", s.d, s.precision, why);
  switch (s.precision) {
    case LRDS_PRECISION_TF32X3: return launch_prec<LRDS_PRECISION_TF32X3>(a, p, st);
    case LRDS_PRECISION_BF16: return launch_prec<LRDS_PRECISION_BF16>(a, p, st);
    case LRDS_PRECISION_TF32: return launch_prec<LRDS_PRECISION_TF32>(a, p, st);
    case LRDS_PRECISION_F16X3: return launch_prec<LRDS_PRECISION_F16X3>(a, p, st);
  }
  return fail(LRDS_ERR_INVALID, "unknown precision %d", s.precision);
}

size_t tc_image_bytes(int d, int num_hidden, int precision) { return tc_layout(d, num_hidden, precision).bytes; }

int pack_tc_image(const lrds_mlp& w, int precision, void* image, cudaStream_t st) {
  const TcLayout L = tc_layout(w.d, w.num_hidden, precision);
  if (precision == LRDS_PRECISION_F16X3) {
    if (w.num_hidden > 6) return fail(LRDS_ERR_UNSUPPORTED, "pack_tc_image: f16x3 supports at most 6 hidden layers");
    tc_scales_kernel<<<1, 256, 0, st>>>(w, L, static_cast<uint8_t*>(image));
  }
  pack_tc_image_kernel<<<32, 256, 0, st>>>(w, L, static_cast<uint8_t*>(image));
  const cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? LRDS_OK : cuda_fail(e, "pack_tc_image launch");
}

}  // namespace lrds
