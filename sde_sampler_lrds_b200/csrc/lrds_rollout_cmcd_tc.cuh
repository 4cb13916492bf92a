// CMCD rollout over the Bayesian logistic-regression posterior (ControlledLangevinSDELoss.simulate, losses/oc.py:666-755;
// target distr/logistic_regression.py:41-61 with its autograd score, distr/base.py:146-154) with ALL THREE dense
// contractions of a step on the tensor core:
//     logits    z_n   = sum_j X_nj w_j + b                          [128 x K16] . Img^T      (K-major B operand)
//     gradient  s_j   = sum_n g_n X_nj,  g_n = m_n (y_n - sigma(z_n))   [128 x N16] . Img    (the SAME image, MN-major)
//     drift network (lrds_rollout_tc.cuh)
// in the F16X3 precision (fp16 (hi, lo) 3-pass split, fp32-grade).  The SIMT pipes keep what is not a GEMM: the sigmoid
// and clamp mask per (particle, datum), the GELU epilogues, the noise and the integrator / cost update.
//
// One 128-particle tile per CTA (thread <-> particle <-> TMEM lane), TMEM columns:
//     [0,64) A: x (hi | lo), then the hidden activations      [64,128) D: drift-network accumulator
//     [128, 128+N16) Z: logits, overwritten IN PLACE by g as fp16 (hi | lo) per 16 data (A operand of the gradient GEMM)
//     [.., +K16) T: gradient accumulator                      [.., +d_pad) the Brownian increment of the last step
// so the per-datum residuals g_n (166 / 280 floats per particle, which limit the SIMT kernel to 4 warps per SM through
// shared memory and make it LSU-bound) never leave the tensor memory.  The sigmoid pass is split over the three waits
// of the drift network, whose MMAs it hides.  Shared memory: weight image | data image | columns x, u, drift.
//
// TWO threads per particle: the tile's 128 particles are served by 8 warps; warps w and w + 4 own the same TMEM lanes and
// split every per-particle loop (operand columns, epilogue halves, sigmoid units, 8-dim chunks) - with one 4-warp tile
// per SM the kernel is latency-bound, and halving each thread's work nearly halves the step.  The cost sums are linear,
// so each thread keeps its own partial log-weight and the two are added once, at the end.
//
// The loop is the reference's with the (u_t, drift_t) -> next step's (u_s, drift_s) carry-over (SURVEY 8a row a5) and the
// update fused into the evaluation of the point it starts from: per grid time k the point x_k is evaluated ONCE.
#pragma once
#include "lrds_rollout_tc.cuh"

namespace lrds {

struct CmcdTcLayout {
  int N16, K16, dp;
  uint32_t z_col, t_col, db_col, cols;   // TMEM columns
  uint32_t part_bytes, img_bytes;        // data image: one (hi | lo) part; parts + tail + labels
  uint32_t off_tail, off_y;
};

__host__ __device__ inline CmcdTcLayout cmcd_tc_layout(const lrds_spec& s) {
  CmcdTcLayout L{};
  L.N16 = (s.target.logreg.N + 15) / 16 * 16;
  L.K16 = (s.d + 15) / 16 * 16;
  L.dp = s.mlp.d_pad;
  L.z_col = 128;
  L.t_col = L.z_col + (uint32_t)L.N16;
  L.db_col = L.t_col + (uint32_t)L.K16;
  L.cols = L.db_col + (uint32_t)L.dp;
  L.part_bytes = (uint32_t)L.N16 * (uint32_t)L.K16 * 2u;
  L.off_tail = 2u * L.part_bytes;
  L.off_y = L.off_tail + 16u;
  L.img_bytes = L.off_y + (uint32_t)L.N16 * 4u;
  return L;
}

// per-dim table [4][d_pad]; at least 128 floats (the second threads' partial log-weights at the end)
__host__ __device__ inline int cmcd_tab_floats(int d_pad) { return 4 * d_pad > 128 ? 4 * d_pad : 128; }

// CMCD simulate / compute_eubo, and the LINEAR loop without a reference control (PIS / DDS with ScoreCtrl, the other
// solvers of the reference's experiments/sample_bayesian_logreg_competing.py) over the same posterior
__host__ __device__ inline bool cmcd_tc_applicable(const lrds_spec& s) {
  const bool cmcd = s.kind == LRDS_ROLLOUT_CMCD || s.kind == LRDS_ROLLOUT_EUBO_CMCD;
  const bool lin = s.kind == LRDS_ROLLOUT_LINEAR && !s.has_ref_ctrl && s.ctrl_kind == LRDS_CTRL_SCORE;
  if (!(s.precision == LRDS_PRECISION_F16X3 && (cmcd || lin) && s.target.kind == LRDS_DISTR_LOGREG &&
        s.target.logreg.x_tc != nullptr && s.ref_0.M == 1 && s.mlp.d_pad <= 64 && !gmm_full_on_path(s)))
    return false;
  return cmcd_tc_layout(s).cols <= 512;
}

// log-posterior only (the terminal cost): the SIMT logit pass without storing the residuals
__device__ __forceinline__ float logreg_logp(const lrds_logreg& L, int d, const Col4& x) {
  const float icpt = x(d - 1);
  const float hi = 1.0f - L.eps;
  float ll = 0.f;
  for (int n = 0; n < L.N; n += 4) {
    float z[4] = {0.f, 0.f, 0.f, 0.f};
    const float* xt = L.Xt + n;
    for (int jq = 0; 4 * jq < L.p; ++jq) {
      const float4 xq = x.ld4(jq);
      const float xs[4] = {xq.x, xq.y, xq.z, xq.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int j = 4 * jq + e;
        if (j < L.p) {
          const float4 v = __ldg(reinterpret_cast<const float4*>(xt + (int64_t)j * L.n_pad));
          z[0] = fmaf(v.x, xs[e], z[0]); z[1] = fmaf(v.y, xs[e], z[1]); z[2] = fmaf(v.z, xs[e], z[2]); z[3] = fmaf(v.w, xs[e], z[3]);
        }
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (n + i < L.N) {
        const float yn = __ldg(L.y + n + i);
        const float sig = 1.0f / (1.0f + expf(-(z[i] + icpt)));
        const float ps = fminf(fmaxf(fmaxf(sig, L.threshold), L.eps), hi);
        ll += yn * logf(ps) + (1.0f - yn) * log1pf(-ps);
      }
    }
  }
  const float hl2pi = 0.91893853320467274178f;
  float pr = 0.f;
  const float iw = 1.0f / (2.0f * L.weight_scale * L.weight_scale);
  for (int j = 0; j < L.p; ++j) {
    const float w = x(j);
    pr += -(w * w) * iw;
  }
  pr += (float)L.p * (-logf(L.weight_scale) - hl2pi);
  const float di = icpt - L.intercept_mean;
  pr += -(di * di) / (2.0f * L.intercept_scale * L.intercept_scale) - logf(L.intercept_scale) - hl2pi;
  return ll + pr;
}

struct CmcdTc : TcMlp<LRDS_PRECISION_F16X3> {
  CmcdTcLayout CL;
  int half;              // 0 / 1: which of the particle's two threads this is
  uint32_t ximg_s;       // shared-window address of the data image
  const uint8_t* ximg;   // the same, generic
  float usx;             // its un-scale

  // x -> A; first drift-network layer AND the logit GEMM (N16 may exceed the 256-column MMA limit: split)
  __device__ __forceinline__ void issue_first(const Col4& x) {
    store_x(x, half, 2);  // this thread's 16-dim groups
    arrive_issue([&]() {
      const uint32_t a_hi = tm_tile + a_col(0), a_lo = tm_tile + a_col(1);
      mma_passes<true, false>(tm_tile + d_col(), a_hi, a_lo, 8u, img_s + L.off_in, L.part_bytes, 2u * (uint32_t)C * 16u,
                              (uint32_t)C * 16u, 128u, L.Kin / 16, ptx::make_idesc_f16(128, C));
      const int nsplit = (CL.N16 + 255) / 256;
      const int per = ((CL.N16 / 16 + nsplit - 1) / nsplit) * 16;
      for (int n0 = 0; n0 < CL.N16; n0 += per) {
        const int nn = min(per, CL.N16 - n0);
        mma_passes<true, false>(tm_tile + CL.z_col + (uint32_t)n0, a_hi, a_lo, 8u, ximg_s + (uint32_t)n0 * 16u, CL.part_bytes,
                                2u * (uint32_t)CL.N16 * 16u, (uint32_t)CL.N16 * 16u, 128u, CL.K16 / 16, ptx::make_idesc_f16(128, nn));
      }
    });
  }
  // gradient GEMM: A = g (hi | lo per 16 data, in place of the logits), B = the data image read MN-major
  __device__ __forceinline__ void issue_gradient() {
    arrive_issue([&]() {
      const uint32_t zc = tm_tile + CL.z_col;
      mma_passes<true, false>(tm_tile + CL.t_col, zc, zc + 8u, 16u, ximg_s, CL.part_bytes, 256u, 128u, (uint32_t)CL.N16 * 16u,
                              CL.N16 / 16, ptx::make_idesc_f16(128, CL.K16) | (1u << 16));
    });
  }

  // logits of data [16 t0, 16 t1) -> g = m (y - sigma(z)), m = [eps <= sigma <= 1 - eps] (and >= threshold), as fp16
  // (hi | lo) in place.  Rows beyond N meet zero image rows in the gradient GEMM, whatever g they get.
  __device__ __forceinline__ void sigmoid_units(const lrds_logreg& LR, int t0, int t1) {
    const float kz = -1.4426950408889634f * usx;
    const float hi1 = 1.0f - LR.eps, lo1 = fmaxf(LR.threshold, LR.eps);
    const float* y = reinterpret_cast<const float*>(ximg + CL.off_y);
#pragma unroll 1
    for (int t = t0 + half; t < t1; t += 2) {
      uint32_t zr[16];
      ptx::tmem_ld16(tm_lane + CL.z_col + 16u * (uint32_t)t, zr);
      ptx::tmem_wait_ld();
      uint32_t ph[8], pl[8];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float4 yv = reinterpret_cast<const float4*>(y + 16 * t)[q];
        const float ys[4] = {yv.x, yv.y, yv.z, yv.w};
        float g[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float e, sig;
          asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(__uint_as_float(zr[4 * q + i]) * kz));
          asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(sig) : "f"(1.0f + e));
          const bool inside = (sig >= lo1) && (sig <= hi1);
          g[i] = inside ? (ys[i] - sig) : 0.f;
        }
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          u64 h2, l2;
          f2::split(f2::pack(g[2 * i], g[2 * i + 1]), h2, l2);
          float h0, h1, l0, l1;
          f2::unpack(h2, h0, h1);
          f2::unpack(l2, l0, l1);
          ph[2 * q + i] = ptx::pack_f16x2(h0, h1);
          pl[2 * q + i] = ptx::pack_f16x2(l0, l1);
        }
      }
      ptx::tmem_st8(tm_lane + CL.z_col + 16u * (uint32_t)t, ph);
      ptx::tmem_st8(tm_lane + CL.z_col + 16u * (uint32_t)t + 8u, pl);
    }
  }

  // everything on the tensor core for the point x: afterwards D holds the network output, T the data gradient
  // (the caller generates the step's noise between issue_first() and finish(): it hides the first GEMMs)
  __device__ __forceinline__ void finish(const lrds_logreg& LR, const float* __restrict__ bias1) {
    const int units = CL.N16 / 16, per = (units + L.nh) / (L.nh + 1);
    const float* bh = reinterpret_cast<const float*>(img + L.off_bhid);
    int done = 0;
    for (int l = 0; l < L.nh; ++l) {
      wait();
      if (l == 0) epilogue_f16<true>(bias1, 0, 32 * half, 32 * half + 32);
      else epilogue_f16<false>(bh + (l - 1) * C, l, 32 * half, 32 * half + 32);
      issue(L.off_hid + (uint32_t)(l * C * C * L.es), C, C);
      const int upto = min(units, done + per);
      sigmoid_units(LR, done, upto);  // in the shadow of the layer's MMAs
      done = upto;
    }
    wait();
    if (L.nh == 0) epilogue_f16<true>(bias1, 0, 32 * half, 32 * half + 32);
    else epilogue_f16<false>(bh + (L.nh - 1) * C, L.nh, 32 * half, 32 * half + 32);
    issue(L.off_out, C, L.Nout);
    sigmoid_units(LR, done, units);
    wait();
    issue_gradient();
    wait();
  }
  __device__ __forceinline__ void ld8f(uint32_t col, float (&out)[8]) {
    uint32_t r[8];
    ptx::tmem_ld8(tm_lane + col, r);
    ptx::tmem_wait_ld();
#pragma unroll
    for (int i = 0; i < 8; ++i) out[i] = __uint_as_float(r[i]);
  }
  __device__ __forceinline__ void st8f(uint32_t col, const float (&v)[8]) {
    uint32_t r[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) r[i] = __float_as_uint(v[i]);
    ptx::tmem_st8(tm_lane + col, r);
  }
};

// shared memory: [weight image | mbarriers + TMEM slot | data image | columns x, u, drift]
// EUBO: the noising rollout of compute_eubo (oc.py:757-828): starts at target samples, walks the grid backwards
// (points at rows K, K-1, .., 0), control enters the update with the opposite sign, the cost is subtracted, and the
// drift of the NEW point inside the cost is evaluated at the time of the OLD one (the reference's quirk, oc.py:807).
// MODE 2 (LINEAR): x' = ca x + cu u + cz z with u = clip(net) + gamma clip(score); rnd += w_cost sum u^2 + w_z sum u z per
// step (losses/oc.py:218-296 with reference_ctrl=None, 1319-1397) and the terminal cost reference - target log-density.
template <int PREC, int MODE>  // PREC = LRDS_PRECISION_F16X3 (a template so that only that translation unit instantiates it)
__global__ void __launch_bounds__(256, 1)
rollout_cmcd_tc_kernel(const RolloutArgs a, const uint8_t* __restrict__ image, const uint32_t tmem_cols) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  constexpr bool EUBO = MODE == 1, LIN = MODE == 2;
  const lrds_spec& s = a.s;
  const TcLayout TL = tc_layout(s.d, s.mlp.num_hidden, LRDS_PRECISION_F16X3);
  const CmcdTcLayout CL = cmcd_tc_layout(s);
  const lrds_logreg& LR = s.target.logreg;
  const int tid = threadIdx.x, warp = tid >> 5;
  constexpr int NT = 128;                          // particles per CTA; 256 threads = two per particle
  const int pt = tid & (NT - 1), half = tid >> 7;  // particle slot and which of its two threads
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + TL.bytes);
  uint32_t* cnt = reinterpret_cast<uint32_t*>(smem_raw + TL.bytes + 64);  // the tile's hand-off counter
  uint8_t* ximg = smem_raw + TL.bytes + TC_TAIL_BYTES;
  float* dimtab = reinterpret_cast<float*>(ximg + ((CL.img_bytes + 15u) & ~15u));  // [4][dp] per-dim constants
  float* cols = dimtab + cmcd_tab_floats(a.s.mlp.d_pad);
  auto data = [&]() { ptx::bulk_g2s(ximg, LR.x_tc, CL.img_bytes, bars); };  // the data image, staged with the drift weights
  const uint32_t tmem = tc_cta_begin(smem_raw, TL, image, tmem_cols, warp, 2, nullptr, 0, cnt, 1, CL.img_bytes, data);
  CmcdTc mlp;
  mlp.init(TL, smem_raw, tmem, warp, bars + 1, cnt, (uint32_t)(2 * NT / 32), warp == 0 ? 3u : 0u, s.mlp.d_pad);  // warp 0 issues
  mlp.half = half;
  mlp.CL = CL;
  mlp.ximg = ximg;
  mlp.ximg_s = ptx::smem_u32(ximg);
  mlp.usx = *reinterpret_cast<const float*>(ximg + CL.off_tail);

  const int b_raw = blockIdx.x * NT + pt;
  const bool live = b_raw < s.B;
  const int b = live ? b_raw : s.B - 1;  // idle lanes shadow the last particle, results are not stored
  const int d = s.d, dp = s.mlp.d_pad, K = s.K, p = LR.p;
  const Col4 X{cols + 4 * pt, 4 * NT}, U{cols + dp * NT + 4 * pt, 4 * NT}, DR{cols + 2 * dp * NT + 4 * pt, 4 * NT};
  for (int j = half; j < dp; j += 2) {
    X(j) = (j < d) ? __ldg(a.x0 + (int64_t)b * d + j) : 0.f;
    U(j) = 0.f;
    DR(j) = 0.f;
  }
  if (!EUBO && a.traj_out != nullptr && live)
    for (int j = half; j < d; j += 2) a.traj_out[(int64_t)b * d + j] = __ldg(a.x0 + (int64_t)b * d + j);

  const GmmView prior = gmm_at(s.ref_0, 0);
  const CtrlConst cc = ctrl_const(s);
  const float sg = s.cmcd_diff, isg = 1.0f / sg, hd = 0.5f * sg * sg, cb = clip_bound(s.cmcd_clip);
  {  // per-dim table [4][dp]
    const float iw = 1.0f / (LR.weight_scale * LR.weight_scale), ib = 1.0f / (LR.intercept_scale * LR.intercept_scale);
    for (int j = tid; j < dp; j += 2 * NT) {
      dimtab[j] = j < d ? prior.mu.ld1(j) : 0.f;
      dimtab[dp + j] = j < d ? prior.ivar.ld1(j) : 0.f;
      dimtab[2 * dp + j] = j == p ? LR.intercept_mean : 0.f;
      dimtab[3 * dp + j] = j < p ? iw : (j == p ? ib : 0.f);
    }
    __syncthreads();
  }
  auto prior_logp = [&]() {
    float q = 0.f;
    for (int c = 0; 4 * c < d; ++c) quad4(q, X.ld4(c), prior.mu.ld4(c), prior.ivar.ld4(c));
    return prior.glogc.ld1(0) - 0.5f * q;
  };
  // forward: initial_log_prob(x), oc.py:698; noising: -terminal_unnorm_log_prob(x), oc.py:782 (first thread of the pair;
  // the second one starts its partial sum at zero)
  float rnd = (half || LIN) ? 0.f : (EUBO ? -clipf(logreg_logp(LR, d, X), s.clip_target) : prior_logp());
  const float usign = EUBO ? -sg : sg;  // the control's sign in the update (oc.py:724 / 804)
  float dt_prev = 0.f, frac_prev = 0.f;
  if constexpr (LIN) {
    for (int k = 0; k < K; ++k) {
      const float* row = s.steps + (int64_t)k * LRDS_STEP_STRIDE;
      const float A = __ldg(row + LRDS_STEP_A), Bc = __ldg(row + LRDS_STEP_B), Cc = __ldg(row + LRDS_STEP_C);
      const float dt = __ldg(row + LRDS_STEP_DT), sqdt = __ldg(row + LRDS_STEP_SQRT_DT);
      const float wcost = __ldg(row + LRDS_STEP_W_COST), wito = __ldg(row + LRDS_STEP_W_ITO);
      const float gamma = __ldg(row + LRDS_STEP_GAMMA), sigu = __ldg(row + LRDS_STEP_SIGU);
      const bool em = s.update_form == LRDS_UPDATE_EM;
      const float wz = s.ito_form == LRDS_ITO_SCALED ? wito
                       : s.ito_form == LRDS_ITO_EM   ? sqdt
                       : s.ito_form == LRDS_ITO_DDS  ? sigu * wito
                                                     : 0.f;
      const float ca = em ? 1.0f - A * dt : A, cu = em ? Bc * dt : Bc, cz = em ? Bc * sqdt : Cc;
      __syncthreads();  // the pair's writes of x are visible to both threads
      mlp.issue_first(X);
      float zs[4][JC];
#pragma unroll
      for (int ci = 0; ci < 4; ++ci) {
        const int j0 = JC * (2 * ci + half);
        if (j0 < dp) {
          noise_chunk(a, k, b, j0, zs[ci]);
        } else {
#pragma unroll
          for (int i = 0; i < JC; ++i) zs[ci][i] = 0.f;
        }
      }
      mlp.finish(LR, row + LRDS_STEP_BIAS1);
      float su2 = 0.f, sito = 0.f;
#pragma unroll
      for (int ci = 0; ci < 4; ++ci) {
        const int j0 = JC * (2 * ci + half);
        if (j0 >= dp) break;
        float xr[JC], T[JC], um[JC], xn[JC];
        mlp.ld8f(CL.t_col + (uint32_t)j0, T);
        mlp.out_chunk(j0, um);
        load_chunk(X, j0, xr);
        const float4 s0 = reinterpret_cast<const float4*>(dimtab + 2 * dp + j0)[0], s1 = reinterpret_cast<const float4*>(dimtab + 2 * dp + j0)[1];
        const float4 i0 = reinterpret_cast<const float4*>(dimtab + 3 * dp + j0)[0], i1 = reinterpret_cast<const float4*>(dimtab + 3 * dp + j0)[1];
        const float sm[JC] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
        const float si[JC] = {i0.x, i0.y, i0.z, i0.w, i1.x, i1.y, i1.z, i1.w};
#pragma unroll
        for (int i = 0; i < JC; ++i) {
          const float sc = T[i] * mlp.usx - (xr[i] - sm[i]) * si[i];
          const float v = clipb(um[i], cc.bound_model) + (cc.scale_score * clipb(sc, cc.bound_score)) * gamma;
          su2 = fmaf(v, v, su2);
          sito = fmaf(v, zs[ci][i], sito);
          xn[i] = (ca * xr[i] + cu * v) + cz * zs[ci][i];
        }
        store_chunk(X, j0, xn);
        if (a.traj_out != nullptr && live) store_traj(a, k + 1, b, j0, xn);
      }
      rnd += wcost * su2;
      rnd += wz * sito;
    }
  }
  for (int k = 0; !LIN && k <= K; ++k) {  // forward: point x_k at row k; noising: the k-th point, at row K - k
    const int rk = EUBO ? K - k : k;
    const float* row = s.steps + (int64_t)rk * LRDS_STEP_STRIDE;
    const float gamma = __ldg(row + LRDS_STEP_GAMMA), frac = __ldg(row + LRDS_STEP_FRAC);
    const bool step = k < K;
    const float* rowd = EUBO ? row - LRDS_STEP_STRIDE : row;  // the row holding dt of the step that leaves this point
    const float dt = step ? __ldg(rowd + LRDS_STEP_DT) : 0.f, sqdt = step ? __ldg(rowd + LRDS_STEP_SQRT_DT) : 0.f;
    const float fcost = EUBO ? frac_prev : frac;  // time at which the cost evaluates the new point's drift
    __syncthreads();  // the pair's writes of x (previous chunk loop / initial load) are visible to both threads
    mlp.issue_first(X);
    float zs[4][JC];  // the step's increments for this thread's (at most four) chunks, generated behind the first GEMMs
#pragma unroll
    for (int ci = 0; ci < 4; ++ci) {
      const int j0 = JC * (2 * ci + half);
      if (step && j0 < dp) {
        noise_chunk(a, k, b, j0, zs[ci]);
      } else {
#pragma unroll
        for (int i = 0; i < JC; ++i) zs[ci][i] = 0.f;
      }
    }
    mlp.finish(LR, row + LRDS_STEP_BIAS1);
    float c2 = 0.f, cdb = 0.f;
#pragma unroll
    for (int ci = 0; ci < 4; ++ci) {  // this thread's 8-dim chunks
      const int j0 = JC * (2 * ci + half);
      if (j0 >= dp) break;
      float xr[JC], uo[JC], dro[JC], T[JC], um[JC], dbo[JC], xn[JC], un[JC], drn[JC], dbn[JC];
      const float (&z)[JC] = zs[ci];
      {  // the chunk's three TMEM reads (gradient, network output, last increment) behind one wait
        uint32_t r0[8], r1[8], r2[8];
        ptx::tmem_ld8(mlp.tm_lane + CL.t_col + (uint32_t)j0, r0);
        ptx::tmem_ld8(mlp.tm_lane + mlp.d_col() + (uint32_t)j0, r1);
        if (k > 0) ptx::tmem_ld8(mlp.tm_lane + CL.db_col + (uint32_t)j0, r2);
        ptx::tmem_wait_ld();
        const float4* b4 = reinterpret_cast<const float4*>(mlp.img + mlp.L.off_bout + j0 * 4);
        const float4 ba = b4[0], bb = b4[1];
        const float bs[8] = {ba.x, ba.y, ba.z, ba.w, bb.x, bb.y, bb.z, bb.w};
        const float uso = mlp.unscale(mlp.L.nh + 1);
#pragma unroll
        for (int i = 0; i < JC; ++i) {
          T[i] = __uint_as_float(r0[i]);
          um[i] = fmaf(__uint_as_float(r1[i]), uso, bs[i]);
          dbo[i] = k > 0 ? __uint_as_float(r2[i]) : 0.f;
        }
      }
      load_chunk(X, j0, xr);
      load_chunk(U, j0, uo);
      load_chunk(DR, j0, dro);
      // per-dim constants (prior mean, prior 1/var, score mean, score 1/var) from the shared-memory table; padded dims
      // need no masks: their gradient, output weights, biases, table entries and noise are zero, so everything stays 0
      const float* tb = dimtab + j0;
      float pm[JC], pv[JC], sm[JC], si[JC];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const float4 a0 = reinterpret_cast<const float4*>(tb)[h], a1 = reinterpret_cast<const float4*>(tb + dp)[h];
        const float4 a2 = reinterpret_cast<const float4*>(tb + 2 * dp)[h], a3 = reinterpret_cast<const float4*>(tb + 3 * dp)[h];
        pm[4 * h] = a0.x; pm[4 * h + 1] = a0.y; pm[4 * h + 2] = a0.z; pm[4 * h + 3] = a0.w;
        pv[4 * h] = a1.x; pv[4 * h + 1] = a1.y; pv[4 * h + 2] = a1.z; pv[4 * h + 3] = a1.w;
        sm[4 * h] = a2.x; sm[4 * h + 1] = a2.y; sm[4 * h + 2] = a2.z; sm[4 * h + 3] = a2.w;
        si[4 * h] = a3.x; si[4 * h + 1] = a3.y; si[4 * h + 2] = a3.z; si[4 * h + 3] = a3.w;
      }
#pragma unroll
      for (int i = 0; i < JC; ++i) {
        // target score: sum_n g_n X_nj - w_j / s_w^2 ; intercept: sum_n g_n - (b - m) / s_b^2
        const float sc = T[i] * mlp.usx - (xr[i] - sm[i]) * si[i];
        float v = clipb(um[i], cc.bound_model);
        if (cc.score) v = v + (cc.scale_score * clipb(sc, cc.bound_score)) * gamma;
        const float ps = -((xr[i] - pm[i]) * pv[i]);
        const float dnew = clipb((sc * frac + ps * (1.0f - frac)) * hd, cb);  // ControlledLangevinSDE.drift, eq/sdes.py:101-110
        if (k > 0) {  // cost = (drift_s + drift_t) / sigma + u_s - u_t   (oc.py:737, 816)
          const float dc = EUBO ? clipb((sc * fcost + ps * (1.0f - fcost)) * hd, cb) : dnew;
          const float cst = EUBO ? (dc + dro[i]) * isg + v - uo[i] : (dro[i] + dc) * isg + uo[i] - v;
          c2 = fmaf(cst, cst, c2);
          cdb = fmaf(cst, dbo[i], cdb);
        }
        const float db = sqdt * z[i];
        xn[i] = xr[i] + (dnew + v * usign) * dt + sg * db;  // oc.py:722-724 / 802-804 (dt = 0 beyond the last point)
        un[i] = v;
        drn[i] = dnew;
        dbn[i] = db;
      }
      if (step) {
        store_chunk(X, j0, xn);
        store_chunk(U, j0, un);
        store_chunk(DR, j0, drn);
        mlp.st8f(CL.db_col + (uint32_t)j0, dbn);
        if (!EUBO && a.traj_out != nullptr && live) store_traj(a, k + 1, b, j0, xn);
      }
    }
    if (k > 0) {
      if (EUBO) {
        rnd -= 0.5f * c2 * dt_prev;
        rnd -= cdb;
      } else {
        rnd += 0.5f * c2 * dt_prev;
        rnd += cdb;
      }
    }
    dt_prev = dt;
    frac_prev = frac;
  }
  __syncthreads();  // final state complete; the table is dead: its first 128 floats carry the second threads' partial sums
  if (half) dimtab[pt] = rnd;
  __syncthreads();
  if (!half) {
    rnd += dimtab[pt];
    if (EUBO) rnd += prior_logp();                                   // oc.py:825
    else if (LIN)  // ref_0 - target, oc.py:290, 1389; init_cost (DIS): the pre-pass result in rnd_out replaces ref_0(x_T)
      rnd += (s.init_cost ? a.rnd_out[b] : prior_logp()) - clipf(logreg_logp(LR, d, X), s.clip_target);
    else rnd -= clipf(logreg_logp(LR, d, X), s.clip_target);         // oc.py:750
    if (live) a.rnd_out[b] = rnd;
  }
  if (live && a.x_out != nullptr)
    for (int j = half; j < d; j += 2) a.x_out[(int64_t)b * d + j] = X(j);
  report_status(s, live, mlp.saturated(), !half && !isfinite(rnd));
  tc_cta_end(warp, tmem, tmem_cols);
}

inline bool plan_rollout_cmcd_tc(const lrds_spec& s, int smem_cap, TcPlan* out) {
  if (!cmcd_tc_applicable(s)) return false;
  const TcLayout TL = tc_layout(s.d, s.mlp.num_hidden, s.precision);
  if (TL.tile_cols != 128) return false;
  const CmcdTcLayout CL = cmcd_tc_layout(s);
  const size_t smem = (size_t)TL.bytes + TC_TAIL_BYTES + ((CL.img_bytes + 15u) & ~15u) + ((size_t)cmcd_tab_floats(s.mlp.d_pad) + (size_t)3 * 128 * s.mlp.d_pad) * sizeof(float);
  if (smem > (size_t)smem_cap) return false;
  out->warps = 8;  // two threads per particle
  out->grid = (s.B + 127) / 128;
  out->staged = 0;
  out->tmem_cols = 512;
  out->smem = smem;
  return true;
}

}  // namespace lrds
