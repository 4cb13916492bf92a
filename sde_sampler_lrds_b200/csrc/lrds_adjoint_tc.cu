// The adjoint of lrds_adjoint on tcgen05 (F16X3 rollouts inside lrds_mlp_grad's envelope: d <= 64, <= 2 hidden layers).
// A CTA carries a tile of 128 particles through k = K-1 .. 0 with the layout of the weight-gradient kernel (four threads
// per particle, TMEM lane = particle; lrds_mlp_tc.cuh): per step the forward recompute from x_k with GELU' kept in TMEM,
// then the backward-data GEMMs through the output, hidden and input layers on the rollout's own F16X3 weight image read
// MN-major.  lambda stays in shared-memory columns; the per-particle parts shared with the SIMT kernel (lambda_K, J_r of the
// reference mixture) run on one thread per particle while the tensor core computes the forward GEMMs.  The recursion runs
// with w = 1 (it is linear in w_b: the fp16 (hi, lo) operands keep unit-scale cotangents) and cot_out is scaled by w_b.
#include "lrds_adjoint.cuh"
#include "lrds_internal.h"
#include "lrds_mlp_tc.cuh"

namespace lrds {

constexpr uint32_t ADJ_TMEM_COLS = 256;  // A (hi, lo) 64 + D 64 + GELU' 32 per layer (<= 96): 224 used

__host__ __device__ inline uint32_t adj_tc_cols_off(const TcLayout& TL) { return (TL.bytes + TC_TAIL_BYTES + 15u) & ~15u; }
__host__ __device__ inline uint32_t adj_tc_bytes(const lrds_spec& s, const TcLayout& TL) {
  return adj_tc_cols_off(TL) + 128u * (uint32_t)adj_layout(s, false).total * 4u + 128u * 4u;
}

__global__ void __launch_bounds__(MG_THREADS, 1) adjoint_tc_kernel(const AdjointArgs a) {
  extern __shared__ __align__(128) uint8_t adj_smem[];
  uint8_t* const smem = adj_smem;
  const lrds_spec& s = a.r.s;
  const int d = s.d, nh = s.mlp.num_hidden, K = s.K;
  const TcLayout TL = tc_layout(d, nh, LRDS_PRECISION_F16X3);
  const AdjLayout L = adj_layout(s, false);
  float* cols = reinterpret_cast<float*>(smem + adj_tc_cols_off(TL));
  uint32_t* bad = reinterpret_cast<uint32_t*>(cols + 128 * L.total);  // per particle: a non-finite cotangent was seen
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, q = warp & 3, h = warp >> 2;
  const int rloc = 32 * q + lane;
  const int b_raw = blockIdx.x * 128 + rloc;
  const bool live = b_raw < s.B;
  const int b = live ? b_raw : s.B - 1;  // idle rows shadow the last particle, nothing is stored for them
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + TL.bytes);  // [0] image, [1] MMA batches
  uint32_t* slot = reinterpret_cast<uint32_t*>(smem + TL.bytes + 48);
  if (warp == 0) ptx::tmem_alloc(slot, ADJ_TMEM_COLS);
  if (tid == 0) {
    ptx::mbar_init(bars, 1);
    ptx::mbar_init(bars + 1, 1);
    ptx::fence_mbar_init();
  }
  if (tid < 128) bad[tid] = 0u;
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  if (tid == 0) {
    ptx::mbar_expect_tx(bars, TL.bytes);
    ptx::bulk_g2s(smem, s.mlp.tc_image, TL.bytes, bars);
  }
  const Particle P = make_particle(cols, L.c, 128, rloc);
  const Col cm{cols + L.cm * 128 + rloc, 128};
  const Col4 lam{cols + L.lam * 128 + 4 * rloc, 4 * 128}, jr{cols + L.lamn * 128 + 4 * rloc, 4 * 128};
  const bool has_ref = s.has_ref_ctrl != 0;
  if (h == 0) {  // lambda_K (unit weight)
    load_state(a, K, b, P.x);
    adj_terminal(s, P, lam, 1.0f);
  }
  __syncthreads();  // x_K and lambda_K are read by the row's other threads below
  ptx::mbar_wait(bars, 0);
  const uint32_t tmem = *slot;
  const uint32_t tm_lane = tmem + ((uint32_t)(q * 32) << 16);
  const uint32_t img_s = ptx::smem_u32(smem);
  const float* sc = reinterpret_cast<const float*>(smem + TL.off_scale);
  const float* bhid = reinterpret_cast<const float*>(smem + TL.off_bhid);
  const float* bout = reinterpret_cast<const float*>(smem + TL.off_bout);
  const int Kin = TL.Kin, Nout = TL.Nout;
  const float bound = clip_bound(s.clip_model), wb = __ldg(a.row_w + b);
  uint64_t* bar = bars + 1;
  uint32_t phase = 0;
  auto hand = [&](auto&& issue) {  // operands stored -> the batch is issued and committed to `bar`
    ptx::fence_proxy_async();
    ptx::tmem_wait_st();
    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 0) {
      if (ptx::elect_one()) {
        ptx::tc_fence_after();
        issue();
        ptx::mma_commit(bar);
      }
      __syncwarp();
    }
  };
  auto wait = [&]() {
    ptx::mbar_wait(bar, phase);
    phase ^= 1u;
    ptx::tc_fence_after();
  };
  auto store_a = [&](const float (&v)[16]) {  // this thread's 16 columns as the next A operand (hi, lo)
    uint32_t ph[8], pl[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) split_pack(v[2 * i], v[2 * i + 1], ph[i], pl[i]);
    ptx::tmem_st8(tm_lane + MG_A_HI + 8 * h, ph);
    ptx::tmem_st8(tm_lane + MG_A_LO + 8 * h, pl);
  };
  float amax = 0.f, vmax = 0.f;  // largest coordinate / cotangent operand, hidden pre-activation (fp16 saturation)
  bool nonfinite = false;
  for (int k = K - 1; k >= 0; --k) {
    const AdjStep st = adj_step(s, s.steps + (int64_t)k * LRDS_STEP_STRIDE);
    const bool back = k > 0;
    const float* xr = a.traj + ((int64_t)k * s.B + b) * d;
    if (h < Kin / 16) {
      float xv[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const int j = 16 * h + i;
        xv[i] = j < d ? __ldg(xr + j) : 0.f;
        amax = fmaxf(amax, fabsf(xv[i]));
        if (has_ref && back && j < d) P.x(j) = xv[i];
      }
      store_a(xv);
    }
    hand([&] { mg_mma_fwd(tmem, img_s, TL, TL.off_in, Kin, C); });
    if (has_ref && back && h == 0) adj_jr(s, k, P, lam, cm, jr);  // J_r(x_k) lambda_{k+1}, next to the tensor core
    for (int l = 0; l <= nh; ++l) {
      wait();
      uint32_t pg[8];
      mg_forward_layer<true>(tm_lane, h, l, sc[8 + l],
                             l == 0 ? reinterpret_cast<const float4*>(s.steps + (int64_t)k * LRDS_STEP_STRIDE + LRDS_STEP_BIAS1 + 16 * h)
                                    : reinterpret_cast<const float4*>(bhid + (l - 1) * C + 16 * h),
                             pg, vmax);
      if (l < nh) hand([&] { mg_mma_fwd(tmem, img_s, TL, TL.off_hid + (uint32_t)(l * C * C * 2), C, C); });
      else hand([&] { mg_mma_fwd(tmem, img_s, TL, TL.off_out, C, Nout); });
    }
    // ---- output: g_k, gbar_k (to cot_out), the masked cotangent as the A operand of the backward-data GEMMs ----
    wait();
    if (h < Nout / 16) {
      uint32_t rr[16];
      ptx::tmem_ld16(tm_lane + MG_D + 16 * h, rr);
      ptx::tmem_wait_ld();
      float z[16], dl[16];
      noise_chunk(a.r, k, b, 16 * h, reinterpret_cast<float(&)[JC]>(z[0]));
      noise_chunk(a.r, k, b, 16 * h + 8, reinterpret_cast<float(&)[JC]>(z[8]));
      float* cot = a.cot_out + ((int64_t)k * s.B + b) * d;
      const float us = sc[8 + nh + 1];
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const int j = 16 * h + i;
        const float net = fmaf(__uint_as_float(rr[i]), us, bout[j]);
        float gb = 0.f;
        if (j < d) {
          gb = adj_gbar(st, 1.0f, clipb(net, bound), z[i], lam(j));
          if (live) cot[j] = wb * gb;
          nonfinite |= !isfinite(gb);
        }
        dl[i] = fabsf(net) <= bound ? gb : 0.f;
        amax = fmaxf(amax, fabsf(dl[i]));
      }
      store_a(dl);
    }
    if (!back) break;
    hand([&] { mg_mma_bwd(tmem, img_s, TL, TL.off_out, Nout, C); });
    // ---- backward: delta_l = (delta_{l+1} W) GELU'(v_l), then through the input layer ----
    for (int l = nh + 1; l >= 1; --l) {
      wait();
      const float ub = 1.0f / sc[l];
      uint32_t rr[16], gp[8];
      ptx::tmem_ld16(tm_lane + MG_D + 16 * h, rr);
      ptx::tmem_ld8(tm_lane + MG_GP + 32 * (l - 1) + 8 * h, gp);
      ptx::tmem_wait_ld();
      float dl[16];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float2 gd = unpack_gp(gp[i]);
        dl[2 * i] = __uint_as_float(rr[2 * i]) * ub * gd.x;
        dl[2 * i + 1] = __uint_as_float(rr[2 * i + 1]) * ub * gd.y;
        amax = max3abs(amax, dl[2 * i], dl[2 * i + 1]);
      }
      store_a(dl);
      if (l > 1) hand([&] { mg_mma_bwd(tmem, img_s, TL, TL.off_hid + (uint32_t)((l - 2) * C * C * 2), C, C); });
      else hand([&] { mg_mma_bwd(tmem, img_s, TL, TL.off_in, C, Kin); });
    }
    wait();
    // lambda_k = a_k lambda_{k+1} + c_k J_r lambda_{k+1} + W_in^T delta_1 (in place: every reader of lambda_{k+1} is done)
    if (h < Kin / 16) {
      uint32_t rr[16];
      ptx::tmem_ld16(tm_lane + MG_D + 16 * h, rr);
      ptx::tmem_wait_ld();
      const float ub = 1.0f / sc[0];
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const int j = 16 * h + i;
        if (j < d) lam(j) = fmaf(st.ak, lam(j), has_ref ? st.ck * jr(j) : 0.f) + __uint_as_float(rr[i]) * ub;
      }
    }
  }
  if (nonfinite) atomicOr(bad + rloc, 1u);
  ptx::tc_fence_before();
  __syncthreads();
  report_status(s, live, amax > F16X3_MAX_COORD || vmax > F16X3_MAX_PREACT, h == 0 && bad[rloc] != 0u);
  if (warp == 0) ptx::tmem_dealloc(tmem, ADJ_TMEM_COLS);
}

bool adjoint_tc_applicable(const lrds_spec& s) {
  if (s.precision != LRDS_PRECISION_F16X3 || !s.mlp.tc_image || !mlp_grad_applicable(s.d, s.mlp.num_hidden)) return false;
  return adj_tc_bytes(s, tc_layout(s.d, s.mlp.num_hidden, LRDS_PRECISION_F16X3)) <= (uint32_t)device_limits().smem_optin;
}

int launch_adjoint_tc(const AdjointArgs& a, cudaStream_t st) {
  const uint32_t bytes = adj_tc_bytes(a.r.s, tc_layout(a.r.s.d, a.r.s.mlp.num_hidden, LRDS_PRECISION_F16X3));
  cudaError_t e = cudaFuncSetAttribute(adjoint_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e == cudaSuccess) {
    adjoint_tc_kernel<<<(a.r.s.B + 127) / 128, MG_THREADS, bytes, st>>>(a);
    e = cudaGetLastError();
  }
  return e == cudaSuccess ? LRDS_OK : cuda_fail(e, "adjoint_tc launch (%u B smem, %u TMEM columns)", bytes, ADJ_TMEM_COLS);
}

}  // namespace lrds
