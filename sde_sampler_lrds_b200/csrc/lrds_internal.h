// Interfaces between the translation units of liblrds_b200.so (not part of the C ABI).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "../../include/lrds_b200.h"

namespace lrds {
struct RolloutArgs;
struct AdjointArgs;
// lrds_capi.cu: the calling thread's message for lrds_last_error; `code` resp. LRDS_ERR_CUDA is returned, and
// cuda_fail appends ": " and the CUDA error string
int fail(int code, const char* fmt, ...) __attribute__((format(printf, 2, 3)));
int cuda_fail(cudaError_t e, const char* fmt, ...) __attribute__((format(printf, 2, 3)));
// the current device's opt-in shared memory per block and SM count (148 SMs without a device: scratch-size queries)
struct DeviceLimits {
  int smem_optin, sms;
};
DeviceLimits device_limits();
// lrds_tc.cu
int launch_rollout_tc(const RolloutArgs& a, cudaStream_t st);
size_t tc_image_bytes(int d, int num_hidden, int precision);
int pack_tc_image(const lrds_mlp& w, int precision, void* image, cudaStream_t st);
// lrds_adjoint_tc.cu: the tcgen05 adjoint (F16X3 inside lrds_mlp_grad's envelope, when its shared memory fits)
bool adjoint_tc_applicable(const lrds_spec& s);
int launch_adjoint_tc(const AdjointArgs& a, cudaStream_t st);
// lrds_mlp_grad.cu
bool mlp_grad_applicable(int d, int num_hidden);
int mlp_grad_params(int d, int num_hidden);
int64_t mlp_grad_scratch_floats(int d, int num_hidden, int S, int B);
int launch_mlp_grad(const lrds_mlp& mlp, const float* bias1, const float* x, const float* cot, const float* step_w,
                    const float* row_w, float clip, float cot_scale, const float* cot_scale_dev, int S, int B,
                    float* grads, float* dbias1, float* scratch, cudaStream_t st);
}  // namespace lrds
