// The LINEAR loop WITHOUT a reference control - PIS (EMReferenceSDELoss with reference_ctrl=None, losses/oc.py:218-296)
// and DDS (ExponentialIntegratorSDELoss.simulate, oc.py:1319-1397) - over the PhiFour lattice (distr/phi_four.py:45-96)
// or any target without a per-particle pass (none / ClippedCtrl), in the F16X3 precision, written like the benchmark
// kernel (lrds_rollout_mix.cuh): the drift network on tcgen05, everything per dim on packed fp32x2 pairs, no padding
// masks (padded dims have zero output weights, biases and noise, and the lattice score is masked once per chunk), the
// Ito forms folded into one per-step weight.  The general kernel (lrds_rollout_tc.cuh) evaluates the same loop with
// run-time switches per 8-dim chunk and scalar arithmetic: 12.5 k warp-instructions per warp and step against 6 k here.
//
// TWO threads per particle (like lrds_rollout_cmcd_tc.cuh): shared memory (448 B of state per particle at d = 100 plus a
// 90 KB weight image) and TMEM (224 columns per tile) allow only two 128-particle tiles per SM, which leaves the loop
// latency-bound; so a tile is served by 8 warps - warps w and w + W/2 own the same TMEM lanes and split the operand
// columns, the epilogue halves and the 8-dim chunks (contiguous halves of the lattice, whose two boundary sites each
// thread reads before the network runs) - and the partial log-weights are added once at the end.
#pragma once
#include "lrds_rollout_tc.cuh"

namespace lrds {

__host__ __device__ inline bool lin_tc_applicable(const lrds_spec& s) {
  return s.precision == LRDS_PRECISION_F16X3 && s.kind == LRDS_ROLLOUT_LINEAR && !s.has_ref_ctrl && s.ctrl_kind <= LRDS_CTRL_SCORE &&
         !gmm_full_on_path(s) &&
         (s.target.kind == LRDS_DISTR_PHI4 || s.target.kind == LRDS_DISTR_NONE ||
          (s.target.kind == LRDS_DISTR_GMM && s.ctrl_kind == LRDS_CTRL_CLIPPED && s.target.gmm.M == 1));
}

// EM: update form LRDS_UPDATE_EM (else AXPY); PHI4: ScoreCtrl over the lattice target
template <int PREC, bool EM, bool PHI4>
__global__ void __launch_bounds__(512, 1)
rollout_lin_kernel(const RolloutArgs a, const uint8_t* __restrict__ image, const uint32_t tmem_cols) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  const lrds_spec& s = a.s;
  const TcLayout TL = tc_layout(s.d, s.mlp.num_hidden, PREC);
  const int tid = threadIdx.x, warp = tid >> 5;
  const int nwarps = blockDim.x >> 6, NT = blockDim.x >> 1;  // warps / threads that own particles (a multiple of 4 / 128)
  const int half = tid >= NT, ptid = tid - half * NT, pwarp = warp - half * nwarps;  // the particle's two threads
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + TL.bytes);  // [0] image, [1 + t] tile t
  uint32_t* cnts = reinterpret_cast<uint32_t*>(smem_raw + TL.bytes + 64);  // [t] hand-offs of tile t
  float* cols = reinterpret_cast<float*>(smem_raw + TL.bytes + TC_TAIL_BYTES);
  const uint32_t tmem = tc_cta_begin(smem_raw, TL, image, tmem_cols, warp, 5, nullptr, 0, cnts, 4, 0u, []() {});
  const int tile = pwarp >> 2;
  const int bar_id = 1 + tile;  // the tile's named barrier: 4 warps x 2 threads per particle (full tiles only)
  TcMlp<PREC> mlp;
  // one warp of the tile issues every hand-off of its 4 x 2 warps
  mlp.init(TL, smem_raw, tmem + (uint32_t)(tile * TL.tile_cols), warp, bars + 1 + tile, cnts + tile, 8u,
           half == 0 && (pwarp & 3) == 3 ? 3u : 0u, s.mlp.d_pad);

  const int b_raw = blockIdx.x * NT + ptid;
  const bool live = b_raw < s.B;
  const int b = live ? b_raw : s.B - 1;  // idle lanes shadow the last particle, results are not stored
  const int d = s.d, dp = s.mlp.d_pad, K = s.K;
  const Col4 X{cols + 4 * ptid, 4 * NT};
  float* part = cols + (size_t)dp * NT;  // [NT] partial log-weights of the second threads
  for (int j = half; j < dp; j += 2) X(j) = (j < d) ? __ldg(a.x0 + (int64_t)b * d + j) : 0.f;
  if (a.traj_out != nullptr && live)
    for (int j = half; j < d; j += 2) a.traj_out[(int64_t)b * d + j] = __ldg(a.x0 + (int64_t)b * d + j);

  const CtrlConst cc = ctrl_const(s);
  // lattice score: -beta [ (b - x (1 - x^2)) / coef + coef (2 x - x_{j+1} - x_{j-1}) ]  (distr/phi_four.py:81-96)
  //              = x (p1 + p3 x^2) + p0 + pn ((x_{j+1} + x_{j-1}) - 2 x),  p1 = beta / coef = -p3,  pn = beta coef
  // (the lattice Laplacian stays a difference of neighbours: no cancellation between large terms)
  const float coef = s.target.phi4.a * (float)d, beta = s.target.phi4.beta;
  const u64 p0 = f2::pk(-beta * s.target.phi4.b / coef), p1 = f2::pk(beta / coef), p3 = f2::pk(-beta / coef),
            pn = f2::pk(beta * coef), m2 = f2::pk(-2.0f);
  const int nchunk = dp / JC;
  const int c_begin = half ? (nchunk + 1) / 2 : 0, c_end = half ? nchunk : (nchunk + 1) / 2;  // this thread's chunks
  float rnd = 0.f;

  for (int k = 0; k < K; ++k) {
    const float* row = s.steps + (int64_t)k * LRDS_STEP_STRIDE;
    const float A = __ldg(row + LRDS_STEP_A), Bc = __ldg(row + LRDS_STEP_B), Cc = __ldg(row + LRDS_STEP_C);
    const float dt = __ldg(row + LRDS_STEP_DT), sqdt = __ldg(row + LRDS_STEP_SQRT_DT);
    const float wcost = __ldg(row + LRDS_STEP_W_COST), wito = __ldg(row + LRDS_STEP_W_ITO);
    const float gamma = __ldg(row + LRDS_STEP_GAMMA), sigu = __ldg(row + LRDS_STEP_SIGU);
    // one weight for sum(u z): sqrt(omega) (scaled), sqrt(dt) (EM), sigma beta_k (DDS), 0 (none)
    const float wz = s.ito_form == LRDS_ITO_SCALED ? wito
                     : s.ito_form == LRDS_ITO_EM   ? sqdt
                     : s.ito_form == LRDS_ITO_DDS  ? sigu * wito
                                                   : 0.f;
    // update as x' = xa x + xu u + xz z:  AXPY (A, B, C);  EM x + (-(f x) + sigma u) dt + sigma (z sqrt dt)
    const u64 xa2 = f2::pk(EM ? 1.0f - A * dt : A), xu2 = f2::pk(EM ? Bc * dt : Bc), xz2 = f2::pk(EM ? Bc * sqdt : Cc);
    const u64 gs2 = f2::pk(cc.scale_score * gamma);
    ptx::bar_sync(bar_id, 256);  // the pair's writes of x (previous chunk loop / initial load) are visible to both
    // the lattice sites next to this thread's range, before anybody updates them (the barriers of the network's GEMMs
    // separate these reads from the chunk loops)
    float xm = (PHI4 && c_begin > 0) ? X(c_begin * JC - 1) : 0.f;
    const float x_after = (PHI4 && c_end * JC < dp) ? X(c_end * JC) : 0.f;
    {  // the drift network with the operand columns and the epilogue halves split between the pair
      mlp.store_x(X, half, 2);
      mlp.issue(mlp.L.off_in, mlp.L.Kin, C);
      const float* bh = reinterpret_cast<const float*>(mlp.img + mlp.L.off_bhid);
      for (int l = 0; l <= mlp.L.nh; ++l) {
        mlp.wait();
        if (l == 0) mlp.template epilogue_f16<true>(row + LRDS_STEP_BIAS1, 0, 32 * half, 32 * half + 32);
        else mlp.template epilogue_f16<false>(bh + (l - 1) * C, l, 32 * half, 32 * half + 32);
        if (l < mlp.L.nh) mlp.issue(mlp.L.off_hid + (uint32_t)(l * C * C * mlp.L.es), C, C);
      }
      mlp.issue(mlp.L.off_out, C, mlp.L.Nout);
      mlp.wait();
    }
    u64 su2 = 0, sito = 0;
    for (int c = c_begin; c < c_end; ++c) {
      const int j0 = c * JC;
      const ulonglong2 xa = X.ldu(2 * c), xb = X.ldu(2 * c + 1);
      const u64 XV[4] = {xa.x, xa.y, xb.x, xb.y};
      u64 U[4], XN[4];
      float z[JC];
      mlp.out_chunk2(j0, U);
      noise_chunk(a, k, b, j0, z);
      float xs[JC + 2];
      xs[0] = xm;
#pragma unroll
      for (int q = 0; q < 4; ++q) f2::unpack(XV[q], xs[1 + 2 * q], xs[2 + 2 * q]);
      xs[JC + 1] = !PHI4 ? 0.f : (c + 1 < c_end ? X(j0 + JC) : x_after);
      xm = xs[JC];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        float u0, u1;
        f2::unpack(U[q], u0, u1);
        u64 v = f2::pack(clipb(u0, cc.bound_model), clipb(u1, cc.bound_model));
        if constexpr (PHI4) {
          const u64 xq = XV[q];
          const u64 nb = f2::pack(xs[2 * q] + xs[2 * q + 2], xs[2 * q + 1] + xs[2 * q + 3]);  // left + right neighbours
          u64 t = f2::fma(f2::mul(xq, xq), p3, p1);
          t = f2::fma(xq, t, f2::fma(pn, f2::fma(xq, m2, nb), p0));
          float t0, t1;
          f2::unpack(t, t0, t1);
          if (j0 + JC > d) {  // the chunk holding the lattice end: padded sites have no score
            if (j0 + 2 * q >= d) t0 = 0.f;
            if (j0 + 2 * q + 1 >= d) t1 = 0.f;
          }
          if (cc.score) v = f2::fma(f2::pack(clipb(t0, cc.bound_score), clipb(t1, cc.bound_score)), gs2, v);
        }
        const u64 z2 = f2::pack(z[2 * q], z[2 * q + 1]);
        su2 = f2::fma(v, v, su2);
        sito = f2::fma(v, z2, sito);
        XN[q] = f2::fma(xz2, z2, f2::fma(xa2, XV[q], f2::mul(xu2, v)));
      }
      X.stu(2 * c, ulonglong2{XN[0], XN[1]});
      X.stu(2 * c + 1, ulonglong2{XN[2], XN[3]});
      if (a.traj_out != nullptr && live) {
        float xn[JC];
#pragma unroll
        for (int q = 0; q < 4; ++q) f2::unpack(XN[q], xn[2 * q], xn[2 * q + 1]);
        store_traj(a, k + 1, b, j0, xn);
      }
    }
    rnd += wcost * f2::hsum1(su2);
    rnd += wz * f2::hsum1(sito);
  }
  __syncthreads();  // final state complete
  if (half) part[ptid] = rnd;
  __syncthreads();
  // terminal cost: rnd += reference_log_prob(x) - terminal_unnorm_log_prob(x)   (oc.py:290, 1389)
  if (!half) {
    rnd += part[ptid];
    const GmmView r0 = gmm_at(s.ref_0, 0);
    float q = 0.f;
    for (int c = 0; 4 * c < d; ++c) quad4(q, X.ld4(c), r0.mu.ld4(c), r0.ivar.ld4(c));
    // init_cost (DIS): the pre-pass of lrds_rollout left initial_log_prob(x_0) + rnd_offset in rnd_out (oc.py:1164-1168)
    const float lref = s.init_cost ? a.rnd_out[b] : r0.glogc.ld1(0) - 0.5f * q;
    float ltgt = 0.f;
    if (s.target.kind == LRDS_DISTR_PHI4) ltgt = phi4_logp(s.target.phi4, d, X);
    else if (s.target.kind == LRDS_DISTR_GMM) {
      const GmmView t0 = gmm_at(s.target.gmm, 0);
      float qt = 0.f;
      for (int c = 0; 4 * c < d; ++c) quad4(qt, X.ld4(c), t0.mu.ld4(c), t0.ivar.ld4(c));
      ltgt = t0.glogc.ld1(0) - 0.5f * qt;
    }
    rnd += lref - clipf(ltgt, s.clip_target);
    if (live) a.rnd_out[b] = rnd;
  }
  float xsum = 0.f;
  if (live && a.x_out != nullptr)
    for (int j = half; j < d; j += 2) {
      const float v = X(j);
      xsum += v;
      a.x_out[(int64_t)b * d + j] = v;
    }
  report_status(s, live, mlp.saturated(), !isfinite(half ? xsum : rnd + xsum) && !half);  // non-finite: counted once per particle
  tc_cta_end(warp, tmem, tmem_cols);
}

inline bool plan_rollout_lin(const lrds_spec& s, int smem_cap, int sms, TcPlan* out) {
  if (!lin_tc_applicable(s) || s.ref_0.M != 1) return false;
  const TcLayout TL = tc_layout(s.d, s.mlp.num_hidden, s.precision);
  if (TL.tile_cols > 256) return false;
  const size_t fixed = (size_t)TL.bytes + TC_TAIL_BYTES;
  const size_t per_tile = ((size_t)s.mlp.d_pad + 1) * 128 * sizeof(float);  // x columns + the partial log-weights
  if (fixed + per_tile > (size_t)smem_cap) return false;
  // full 128-particle tiles (the pair's warps w and w + W/2 must share TMEM lanes): one or two per CTA
  const bool two = 2 * TL.tile_cols <= 512 && fixed + 2 * per_tile <= (size_t)smem_cap && s.B > 128 * sms;
  const int w = two ? 8 : 4;
  const int need = (s.B + 31) / 32;
  out->warps = 2 * w;  // launched warps: two threads per particle
  out->grid = (need + w - 1) / w;
  out->staged = 0;
  out->tmem_cols = plan_tmem_cols((w / 4) * TL.tile_cols);
  out->smem = fixed + per_tile * (w / 4);
  return true;
}

}  // namespace lrds
