// The adjoint of lrds_adjoint_cmcd on tcgen05 (F16X3 rollouts inside lrds_mlp_grad's envelope: d <= 64, <= 2 hidden
// layers), in the layout of adjoint_tc_kernel: 128 particles per CTA, four threads per particle (TMEM lane = particle), the
// rollout's F16X3 weight image, GELU' in TMEM, the backward-data GEMMs reading the image MN-major (lrds_mlp_tc.cuh).
//
// Per point j (the recursion of lrds_adjoint_cmcd.cuh): the network runs twice on the tensor core - at the look-ahead
// point x_{j-1} (u_{j-1}, hence e_{j-1} and q_{j-1} = D_{j-1} / sig - u_{j-1}), then at x_j with its GELU' tape, whose
// output gives ubar_j and the masked cotangent for the backward-data GEMMs.  The GELU' tape is recomputed rather than kept
// from the look-ahead (one tape of 96 TMEM columns, 256 allocated).  The target's part runs on the second thread of every
// particle (warps 4-7) next to the tensor core: the target score at the look-ahead point while its forward GEMMs run, the
// score at x_j (the drift clip's mask) during the forward at x_j, and sig^2/2 (f H_pi + (1 - f) H_0) of the masked Dbar_j
// during the backward-data GEMMs.  The first thread of every particle (warps 0-3) keeps lambda_K.
//
// Shared-memory columns per particle: x, lambda, q and two e columns.  The column of e_j receives ubar_j once e_j is
// used, then Dbar_j = (ubar_j + 2 e_{j-1}) / sig (because [j<K](e_j + sig dt_j lambda_{j+1}) = ubar_j + e_{j-1}), then
// its Hessian-vector product in place.  The look-ahead's D_{j-1} / sig waits in the column that then receives e_{j-1}.
// The recursion runs with w = 1 (it is linear in w_b: the fp16 (hi, lo) operands keep unit-scale cotangents) and cot_out
// is scaled by w_b.
#include "lrds_adjoint_cmcd.cuh"
#include "lrds_internal.h"
#include "lrds_mlp_tc.cuh"

namespace lrds {

constexpr uint32_t ADJ_CMCD_TMEM_COLS = 256;  // A (hi, lo) 64 + D 64 + GELU' 32 per layer (<= 96): 224 used

struct AdjCmcdTcLayout {
  ColLayout c;  // x, rt (target responsibilities)
  int cm, lam, q, ea, eb, total;
};
__host__ __device__ inline AdjCmcdTcLayout adj_cmcd_tc_layout(const lrds_spec& s) {
  AdjCmcdTcLayout L{};
  const int dp = s.mlp.d_pad;
  const int M = s.target.kind == LRDS_DISTR_GMM && s.target.gmm.M > 1 ? (s.target.gmm.M + 3) / 4 * 4 : 0;
  int off = 0;
  L.c.x = off; off += dp;
  L.c.rt = off; off += M;
  L.cm = off; off += M;
  L.c.act = L.c.g = L.c.rr = L.c.rh = L.c.us = L.c.tsd = L.c.db = off;  // unused
  L.lam = off; off += dp;
  L.q = off; off += dp;
  L.ea = off; off += dp;
  L.eb = off; off += dp;
  L.total = L.c.total = off;
  return L;
}
__host__ __device__ inline uint32_t adj_cmcd_tc_cols_off(const TcLayout& TL) { return (TL.bytes + TC_TAIL_BYTES + 15u) & ~15u; }
__host__ __device__ inline uint32_t adj_cmcd_tc_bytes(const lrds_spec& s, const TcLayout& TL) {
  return adj_cmcd_tc_cols_off(TL) + 128u * (uint32_t)adj_cmcd_tc_layout(s).total * 4u + 128u * 4u;
}

__global__ void __launch_bounds__(MG_THREADS, 1) adjoint_cmcd_tc_kernel(const AdjointArgs a) {
  extern __shared__ __align__(128) uint8_t adj_smem[];
  uint8_t* const smem = adj_smem;
  const lrds_spec& s = a.r.s;
  const int d = s.d, nh = s.mlp.num_hidden, K = s.K, tkind = s.target.kind;
  const TcLayout TL = tc_layout(d, nh, LRDS_PRECISION_F16X3);
  const AdjCmcdTcLayout L = adj_cmcd_tc_layout(s);
  float* cols = reinterpret_cast<float*>(smem + adj_cmcd_tc_cols_off(TL));
  uint32_t* bad = reinterpret_cast<uint32_t*>(cols + 128 * L.total);  // per particle: a non-finite cotangent was seen
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, q4 = warp & 3, h = warp >> 2;
  const int rloc = 32 * q4 + lane;
  const int b_raw = blockIdx.x * 128 + rloc;
  const bool live = b_raw < s.B;
  const int b = live ? b_raw : s.B - 1;  // idle rows shadow the last particle, nothing is stored for them
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + TL.bytes);  // [0] image, [1] MMA batches
  uint32_t* slot = reinterpret_cast<uint32_t*>(smem + TL.bytes + 48);
  if (warp == 0) ptx::tmem_alloc(slot, ADJ_CMCD_TMEM_COLS);
  if (tid == 0) {
    ptx::mbar_init(bars, 1);
    ptx::mbar_init(bars + 1, 1);
    ptx::fence_mbar_init();
  }
  if (tid < 128) bad[tid] = 0u;
  for (int i = tid; i < 128 * L.total; i += MG_THREADS) cols[i] = 0.f;  // padded dims stay 0 (the HVP reads them)
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  if (tid == 0) {
    ptx::mbar_expect_tx(bars, TL.bytes);
    ptx::bulk_g2s(smem, s.mlp.tc_image, TL.bytes, bars);
  }
  const Particle P = make_particle(cols, L.c, 128, rloc);
  auto col4 = [&](int off) { return Col4{cols + off * 128 + 4 * rloc, 4 * 128}; };
  const Col cm{cols + L.cm * 128 + rloc, 128};
  const Col4 lam = col4(L.lam), q = col4(L.q);
  Col4 ec = col4(L.ea), en = col4(L.eb);  // e_j (then ubar_j, Dbar_j, its HVP), e_{j-1} (first D_{j-1} / sig)
  const GmmView tv0 = gmm_at(s.target.gmm, 0), prior = gmm_at(s.ref_0, 0);
  const float bound = clip_bound(s.clip_model), dbound = clip_bound(s.cmcd_clip);
  const float sg = s.cmcd_diff, isg = 1.0f / sg, h2 = 0.5f * sg * sg;
  if (h == 0) {  // lambda_K at unit weight: -[|log pi(x_K)| <= clip_target] grad log pi(x_K)
    load_state(a, K, b, P.x);
    const float lt = target_pass1<false>(s, tkind, tv0, P, true);
    const float wt = (s.clip_target > 0.f && !(fabsf(lt) <= s.clip_target)) ? 0.f : 1.0f;
    target_score_loop<false>(s, tkind, tv0, P, [&](int j0, const float(&xr)[JC], const float(&ts)[JC]) {
#pragma unroll
      for (int c = 0; c < JC; ++c) lam(j0 + c) = (j0 + c < d) ? -wt * ts[c] : 0.f;
    });
  }
  __syncthreads();  // x_K is reloaded by the target thread below
  ptx::mbar_wait(bars, 0);
  const uint32_t tmem = *slot;
  const uint32_t tm_lane = tmem + ((uint32_t)(q4 * 32) << 16);
  const uint32_t img_s = ptx::smem_u32(smem);
  const float* sc = reinterpret_cast<const float*>(smem + TL.off_scale);
  const float* bhid = reinterpret_cast<const float*>(smem + TL.off_bhid);
  const float* bout = reinterpret_cast<const float*>(smem + TL.off_bout);
  const int Kin = TL.Kin, Nout = TL.Nout;
  const float wb = __ldg(a.row_w + b), us = sc[8 + nh + 1];
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
  // the network at x of trajectory row `row` up to the output accumulator (MG_D, ready on return); `side` runs on the
  // SIMT pipes while the input layer's GEMMs run
  auto forward = [&](int row, auto&& side) {
    const float* xr = a.traj + ((int64_t)row * s.B + b) * d;
    if (h < Kin / 16) {
      float xv[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const int j = 16 * h + i;
        xv[i] = j < d ? __ldg(xr + j) : 0.f;
        amax = fmaxf(amax, fabsf(xv[i]));
      }
      store_a(xv);
    }
    hand([&] { mg_mma_fwd(tmem, img_s, TL, TL.off_in, Kin, C); });
    side();
    const float* rowp = s.steps + (int64_t)row * LRDS_STEP_STRIDE;
    for (int l = 0; l <= nh; ++l) {
      wait();
      uint32_t pg[8];
      mg_forward_layer<true>(tm_lane, h, l, sc[8 + l],
                             l == 0 ? reinterpret_cast<const float4*>(rowp + LRDS_STEP_BIAS1 + 16 * h)
                                    : reinterpret_cast<const float4*>(bhid + (l - 1) * C + 16 * h),
                             pg, vmax);
      if (l < nh) hand([&] { mg_mma_fwd(tmem, img_s, TL, TL.off_hid + (uint32_t)(l * C * C * 2), C, C); });
      else hand([&] { mg_mma_fwd(tmem, img_s, TL, TL.off_out, C, Nout); });
    }
    wait();
  };
  auto out16 = [&](float (&net)[16]) {  // this thread's 16 network outputs from MG_D
    uint32_t rr[16];
    ptx::tmem_ld16(tm_lane + MG_D + 16 * h, rr);
    ptx::tmem_wait_ld();
#pragma unroll
    for (int i = 0; i < 16; ++i) net[i] = fmaf(__uint_as_float(rr[i]), us, bout[16 * h + i]);
  };

  uint32_t dm0 = 0u, dm1 = 0u;  // target thread: [|D_j before the clip| <= cmcd_clip] of dims 0-31, 32-63
  for (int j = K + 1; j >= 0; --j) {  // j = K + 1 only evaluates q_K
    const bool last = j == K, first = j == 0;
    if (!first) {  // ---- look-ahead at p = j - 1: en <- e_p (p < K), q <- q_p ----
      const int p = j - 1;
      const float* rowp = s.steps + (int64_t)p * LRDS_STEP_STRIDE;
      forward(p, [&] {
        if (h == 1) {  // D_p / sig -> en
          load_state(a, p, b, P.x);
          const float f = __ldg(rowp + LRDS_STEP_FRAC);
          target_pass1<false>(s, tkind, tv0, P, false);
          target_score_loop<false>(s, tkind, tv0, P, [&](int j0, const float(&xr)[JC], const float(&ts)[JC]) {
#pragma unroll
            for (int c = 0; c < JC; ++c) {
              const int i = j0 + c;
              en(i) = i < d ? langevin_drift(s, ts[c], -((xr[c] - prior.mu.ld1(i)) * prior.ivar.ld1(i)), f) * isg : 0.f;
            }
          });
        }
      });
      if (h < Nout / 16) {
        float net[16], z[16];
        out16(net);
        if (p < K) {
          noise_chunk(a.r, p, b, 16 * h, reinterpret_cast<float(&)[JC]>(z[0]));
          noise_chunk(a.r, p, b, 16 * h + 8, reinterpret_cast<float(&)[JC]>(z[8]));
        }
        const float dt = __ldg(rowp + LRDS_STEP_DT), sqdt = __ldg(rowp + LRDS_STEP_SQRT_DT);
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const int jd = 16 * h + i;
          if (jd < d) {
            const float t = en(jd), u = clipb(net[i], bound);
            if (p < K) en(jd) = fmaf(t + u + q(jd), dt, sqdt * z[i]);
            q(jd) = t - u;
          }
        }
      }
      if (j > K) continue;
    }
    // ---- point j: the network at x_j with its GELU' tape; ubar_j; the backward-data GEMMs ----
    const float* row = s.steps + (int64_t)j * LRDS_STEP_STRIDE;
    const float f = __ldg(row + LRDS_STEP_FRAC);
    const float dt = last ? 0.f : __ldg(row + LRDS_STEP_DT);
    forward(j, [&] {
      if (h == 1 && !first) {  // responsibilities at x_j and the drift clip's mask
        load_state(a, j, b, P.x);
        target_pass1<false>(s, tkind, tv0, P, false);
        dm0 = dm1 = 0u;
        target_score_loop<false>(s, tkind, tv0, P, [&](int j0, const float(&xr)[JC], const float(&ts)[JC]) {
#pragma unroll
          for (int c = 0; c < JC; ++c) {
            const int i = j0 + c;
            const float ps = -((xr[c] - prior.mu.ld1(i)) * prior.ivar.ld1(i));
            if (i < d && fabsf((ts[c] * f + ps * (1.0f - f)) * h2) <= dbound) {
              if (i < 32) dm0 |= 1u << i;
              else dm1 |= 1u << (i - 32);
            }
          }
        });
      }
    });
    if (h < Nout / 16) {
      float net[16], dl[16];
      out16(net);
      float* cot = a.cot_out + ((int64_t)j * s.B + b) * d;
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const int jd = 16 * h + i;
        float ub = 0.f;
        if (jd < d) {
          if (!last) ub = fmaf(sg * dt, lam(jd), ec(jd));
          if (!first) ub -= en(jd);
          if (live) cot[jd] = wb * ub;
          nonfinite |= !isfinite(ub);
          ec(jd) = ub;
        }
        dl[i] = fabsf(net[i]) <= bound ? ub : 0.f;
        amax = fmaxf(amax, fabsf(dl[i]));
      }
      store_a(dl);
    }
    if (first) break;  // lambda_0 is not needed: x_0 does not depend on the parameters
    hand([&] { mg_mma_bwd(tmem, img_s, TL, TL.off_out, Nout, C); });
    if (h == 1) {  // Dbar_j masked, the prior's part into lambda, then the target's Hessian-vector product in place
      const float hp = h2 * (1.0f - f);
      for (int i = 0; i < d; ++i) {
        const float v = ((i < 32 ? dm0 : dm1) >> (i & 31)) & 1u ? (ec(i) + 2.0f * en(i)) * isg : 0.f;
        ec(i) = v;
        lam(i) = fmaf(-hp * prior.ivar.ld1(i), v, lam(i));
      }
      target_hvp(s, P, ec, cm);
    }
    // ---- backward: delta_l = (delta_{l+1} W) GELU'(v_l), then through the input layer ----
    for (int l = nh + 1; l >= 1; --l) {
      wait();
      const float ubs = 1.0f / sc[l];
      uint32_t rr[16], gp[8];
      ptx::tmem_ld16(tm_lane + MG_D + 16 * h, rr);
      ptx::tmem_ld8(tm_lane + MG_GP + 32 * (l - 1) + 8 * h, gp);
      ptx::tmem_wait_ld();
      float dl[16];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float2 gd = unpack_gp(gp[i]);
        dl[2 * i] = __uint_as_float(rr[2 * i]) * ubs * gd.x;
        dl[2 * i + 1] = __uint_as_float(rr[2 * i + 1]) * ubs * gd.y;
        amax = max3abs(amax, dl[2 * i], dl[2 * i + 1]);
      }
      store_a(dl);
      if (l > 1) hand([&] { mg_mma_bwd(tmem, img_s, TL, TL.off_hid + (uint32_t)((l - 2) * C * C * 2), C, C); });
      else hand([&] { mg_mma_bwd(tmem, img_s, TL, TL.off_in, C, Kin); });
    }
    wait();
    // lambda_j = lambda_{j+1} (+ the prior's part) + W_in^T delta_1 + sig^2/2 f H_pi Dbar_j
    if (h < Kin / 16) {
      uint32_t rr[16];
      ptx::tmem_ld16(tm_lane + MG_D + 16 * h, rr);
      ptx::tmem_wait_ld();
      const float ubs = 1.0f / sc[0], ht = h2 * f;
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const int jd = 16 * h + i;
        if (jd < d) lam(jd) = fmaf(ht, ec(jd), lam(jd)) + __uint_as_float(rr[i]) * ubs;
      }
    }
    const Col4 t = ec;
    ec = en;
    en = t;
  }
  if (nonfinite) atomicOr(bad + rloc, 1u);
  ptx::tc_fence_before();
  __syncthreads();
  report_status(s, live, amax > F16X3_MAX_COORD || vmax > F16X3_MAX_PREACT, h == 0 && bad[rloc] != 0u);
  if (warp == 0) ptx::tmem_dealloc(tmem, ADJ_CMCD_TMEM_COLS);
}

bool adjoint_cmcd_tc_applicable(const lrds_spec& s) {
  if (s.precision != LRDS_PRECISION_F16X3 || !s.mlp.tc_image || !mlp_grad_applicable(s.d, s.mlp.num_hidden)) return false;
  return adj_cmcd_tc_bytes(s, tc_layout(s.d, s.mlp.num_hidden, LRDS_PRECISION_F16X3)) <= (uint32_t)device_limits().smem_optin;
}

int launch_adjoint_cmcd_tc(const AdjointArgs& a, cudaStream_t st) {
  const uint32_t bytes = adj_cmcd_tc_bytes(a.r.s, tc_layout(a.r.s.d, a.r.s.mlp.num_hidden, LRDS_PRECISION_F16X3));
  cudaError_t e = cudaFuncSetAttribute(adjoint_cmcd_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e == cudaSuccess) {
    adjoint_cmcd_tc_kernel<<<(a.r.s.B + 127) / 128, MG_THREADS, bytes, st>>>(a);
    e = cudaGetLastError();
  }
  return e == cudaSuccess ? LRDS_OK
                          : cuda_fail(e, "adjoint_cmcd_tc launch (%u B smem, %u TMEM columns)", bytes, ADJ_CMCD_TMEM_COLS);
}

}  // namespace lrds
