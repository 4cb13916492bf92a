// CMCD (ControlledLangevinSDELoss.simulate, losses/oc.py:666-755) over a MIXTURE target - the configuration of
// experiments/sample_many_modes_competing.py:100-115 - on the machinery of the benchmark kernel (lrds_rollout_mix.cuh):
// drift network, the target mixture's logits and its score contraction on tcgen05, counter / mbarrier hand-offs, no
// barrier inside the time loop.  (The logistic-regression posterior has its own CMCD kernel, lrds_rollout_cmcd_tc.cuh;
// every other CMCD configuration runs the general kernel of lrds_rollout_tc.cuh.)
//
// The loop is written over the K + 1 trajectory POINTS: every point is evaluated once (one network pass, one target
// score), which yields the control u_j and the tempered Langevin drift d_j = clip(sigma^2 / 2 (f_j score_target +
// (1 - f_j) score_prior)) (eq/sdes.py:101-110) that END step j - 1 and START step j (the reference evaluates both ends of
// every step, oc.py:716-737: the same values twice).  Per particle only x and s_j = d_j / sigma + u_j stay in shared
// memory; the step's Brownian increment lives in 56 TMEM columns of the particle's lane until the next point needs it
// for the Ito term:
//     cost_{j-1} = (d_{j-1} + d_j) / sigma + u_{j-1} - u_j = s_{j-1} + d_j / sigma - u_j          (oc.py:737)
//     rnd += cost^2 dt_{j-1} / 2 + cost . dB_{j-1}                                                 (oc.py:740-741)
//     x_{j+1} = x_j + (d_j + sigma u_j) dt_j + sigma dB_j                                           (oc.py:722-724)
// TMEM columns of a tile (192): [0,64) A operands / responsibilities + a PAIR of contraction chunks (the target is the
// only mixture: 16 columns per 8-dim chunk, two chunks per batch) | [64,128) accumulator | [128,184) dB.
#pragma once
#include "lrds_rollout_mix.cuh"

namespace lrds {

constexpr int CMX_MAX_WARPS = 8;  // two tiles: x and s in shared memory (448 B per particle at d = 50) next to the weight image
constexpr uint32_t CMX_TILE_COLS = 192, CMX_DB_COL = 128;

__host__ __device__ inline bool cmcd_mix_applicable(const lrds_spec& s) {
  return s.precision == LRDS_PRECISION_F16X3 && s.kind == LRDS_ROLLOUT_CMCD && s.ctrl_kind <= LRDS_CTRL_SCORE && !gmm_full_on_path(s) &&
         s.target.kind == LRDS_DISTR_GMM && s.target.gmm.M > 1 && s.target.gmm.M <= MIX_MAX_M && s.target.gmm.mix_tc != nullptr &&
         s.ref_0.M == 1 && s.mlp.d_pad <= 56 && !s.init_cost;
}

template <int PREC>
__global__ void __launch_bounds__(CMX_MAX_WARPS * 32, 1)
rollout_cmcd_mix_kernel(const RolloutArgs a, const uint8_t* __restrict__ image, const uint32_t tmem_cols) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  const lrds_spec& s = a.s;
  const TcLayout TL = tc_layout(s.d, s.mlp.num_hidden, PREC);
  const int tid = threadIdx.x;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int nwarps = blockDim.x >> 5, NT = blockDim.x;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + TL.bytes);  // [0] image + target block, [1 + t] MMAs of tile t done
  uint32_t* cnts = reinterpret_cast<uint32_t*>(smem_raw + TL.bytes + TC_TAIL_BYTES);
  uint8_t* stage = smem_raw + TL.bytes + TC_TAIL_BYTES + MIX_TAIL_BYTES;  // the static target mixture: logc | sn | tensor-core images
  const StageLayout SL = stage_layout(s, 2, true);
  float* cols = reinterpret_cast<float*>(stage + ((SL.off_buf + 15u) & ~15u));
  const int d = s.d, dp = s.mlp.d_pad, K = s.K;
  const uint32_t mix_off_t = SL.tgt_logc_bytes + SL.tgt_param_bytes;
  auto target = [&]() {  // the target mixture, staged once per CTA with the drift weights
    stage_gmm(stage + SL.off_tgt, gmm_at(s.target.gmm, 0), SL.tgt_logc_bytes, SL.tgt_param_bytes, bars);
    ptx::bulk_g2s(stage + SL.off_tgt + mix_off_t, static_cast<const uint8_t*>(s.target.gmm.mix_tc), SL.tgt_mix_bytes, bars);
  };
  const uint32_t tmem =
      __shfl_sync(0xffffffffu, tc_cta_begin(smem_raw, TL, image, tmem_cols, warp, 3, nullptr, 0, cnts, 4, SL.tgt_bytes, target), 0);
  const int tile = warp >> 2;
  const int tile_warps = min(4, nwarps - 4 * tile);
  MixTc<PREC> mlp;
  mlp.init(TL, smem_raw, tmem + (uint32_t)tile * CMX_TILE_COLS, warp, bars + 1 + tile, cnts + tile, (uint32_t)tile_warps,
           ((warp & 3) == tile_warps - 1 ? 1u : 0u) | ((warp & 3) == max(tile_warps - 2, 0) ? 2u : 0u), dp);
  const int Mt = s.target.gmm.M;
  const uint32_t contr_bytes = gmm_mix_contr_bytes(Mt, dp), lg_part = gmm_mix_logit_part_bytes(Mt, dp);
  mlp.lbo = (uint32_t)(2 * dp) * 16u;
  mlp.part_bytes = (contr_bytes - 16u) / 2u;
  mlp.lg_part = lg_part;

  const int b_raw = blockIdx.x * NT + tid;
  const bool live = b_raw < s.B;
  const int b = live ? b_raw : s.B - 1;  // idle lanes shadow the last particle, results are not stored
  const Col4 X{cols + 4 * tid, 4 * NT};
  const Col4 S{cols + (size_t)dp * NT + 4 * tid, 4 * NT};  // s = d / sigma + u of the step's starting point
  for (int j = 0; j < dp; ++j) X(j) = (j < d) ? __ldg(a.x0 + (int64_t)b * d + j) : 0.f;
  if (a.traj_out != nullptr && live)
    for (int j = 0; j < d; ++j) a.traj_out[(int64_t)b * d + j] = X(j);

  const CtrlConst cc = ctrl_const(s);
  const GmmView tv0 = gmm_at(s.target.gmm, 0);
  const GmmViewT<true> tv = staged_view(stage + SL.off_tgt, tv0, SL.tgt_logc_bytes, SL.tgt_param_bytes);
  const uint32_t tgt_img = ptx::smem_u32(stage + SL.off_tgt + mix_off_t);
  const PPtr<true> tail_t{tgt_img + contr_bytes + 2u * lg_part};
  const bool lg_t = tail_t.ld1(MIX_MAX_M + 3) != 0.f;  // the target's modes share their variances: logits from the GEMM
  const float ust = *reinterpret_cast<const float*>(stage + SL.off_tgt + mix_off_t + contr_bytes - 16u);
  const GmmView prior = gmm_at(s.ref_0, 0);
  const float sg = s.cmcd_diff;
  const u64 sg2 = f2::pk(sg), isg2 = f2::pk(1.0f / sg), hs2 = f2::pk(0.5f * sg * sg), ust2 = f2::pk(ust);
  const float dclip = clip_bound(s.cmcd_clip);
  const float bts = cc.bound_score / ust;
  const int nchunk = dp / JC, npair = (nchunk + 1) >> 1, nq = (d + 3) >> 2;
  __syncwarp();
  float rnd = gmm_logp_any(prior, d, dp, X);  // initial_log_prob(x_0), oc.py:698

  for (int j = 0; j <= K; ++j) {
    const float* row = s.steps + (int64_t)j * LRDS_STEP_STRIDE;
    const float gamma = __ldg(row + LRDS_STEP_GAMMA), frac = __ldg(row + LRDS_STEP_FRAC);
    const bool step = j < K, cost_on = j > 0;
    const float dt = step ? __ldg(row + LRDS_STEP_DT) : 0.f, sqdt = step ? __ldg(row + LRDS_STEP_SQRT_DT) : 0.f;
    const float dt_prev = cost_on ? __ldg(row - LRDS_STEP_STRIDE + LRDS_STEP_DT) : 0.f;
    mlp.store_x(X);
    // responsibilities of the target mixture (lrds_rollout_mix.cuh: logit GEMM + error bound, exact forms as fallback)
    uint32_t r_p[16];
    bool need = true, ok = false;
    if (lg_t) {
      mlp.arrive_issue([&]() { mlp.logit(0, tgt_img + contr_bytes); });
      u64 n2 = 0;
      for (int c = 0; c < nq; ++c) {
        const ulonglong2 xv = X.ldu(c);
        n2 = f2::fma(xv.x, xv.x, n2);
        n2 = f2::fma(xv.y, xv.y, n2);
      }
      const float xnorm = sqrtf(f2::hsum1(n2));
      mlp.wait();
      uint32_t lg[16];
      ptx::tmem_ld16(mlp.tm_lane + mlp.d_col(), lg);
      ptx::tmem_wait_ld();
      ok = mlp.softmax_logits(lg, tail_t, xnorm, r_p);
      need = __any_sync(0xffffffffu, !ok);
    }
    mlp.template hidden_ws<false>(
        row + LRDS_STEP_BIAS1,
        [&]() {
          if (need) {
            float r[MIX_MAX_M];
            uint32_t p[16];
            gmm_pass1_pair(tv, d, dp, X, r);
            mlp.pack_r(r, p);
#pragma unroll
            for (int i = 0; i < 16; ++i) r_p[i] = ok ? r_p[i] : p[i];
          }
        },
        [&]() {});
    mlp.store_r(0, r_p);
    auto issue_pair = [&](int p) {
      mlp.arrive_issue([&]() {
        mlp.template chunk<true, false>(2 * p, tgt_img, tgt_img, 32u);
        if (2 * p + 1 < nchunk) mlp.template chunk<true, false>(2 * p + 1, tgt_img, tgt_img, 48u);
      });
    };
    issue_pair(0);
    const u64 fr2 = f2::pk(frac), omf2 = f2::pk(1.0f - frac), dt2 = f2::pk(dt), sqdt2 = f2::pk(sqdt);
    const u64 gs2 = f2::pk((cc.scale_score * gamma) * ust);
    u64 c2 = 0, cdb = 0;
    for (int p = 0; p < npair; ++p) {
      uint32_t m[32];
      mlp.wait();
      ptx::tmem_ld32(mlp.tm_lane + 32u, m);
      ptx::tmem_wait_ld();
      if (p + 1 < npair) issue_pair(p + 1);
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int c = 2 * p + h;
        if (c >= nchunk) break;
        const int j0 = c * JC;
        const ulonglong2 xa = X.ldu(2 * c), xb = X.ldu(2 * c + 1);
        const u64 XV[4] = {xa.x, xa.y, xb.x, xb.y};
        const ulonglong2 g0 = prior.mu.ld2(2 * c), g1 = prior.mu.ld2(2 * c + 1), i0 = prior.ivar.ld2(2 * c), i1 = prior.ivar.ld2(2 * c + 1);
        const u64 GM[4] = {g0.x, g0.y, g1.x, g1.y}, GI[4] = {i0.x, i0.y, i1.x, i1.y};
        u64 U[4], SP[4] = {0, 0, 0, 0}, DBP[4] = {0, 0, 0, 0}, SN[4], XN[4], DBN[4];
        mlp.out_chunk2(j0, U);
        if (cost_on) {
          const ulonglong2 sa = S.ldu(2 * c), sb = S.ldu(2 * c + 1);
          SP[0] = sa.x; SP[1] = sa.y; SP[2] = sb.x; SP[3] = sb.y;
          uint32_t dbp[8];
          ptx::tmem_ld8(mlp.tm_lane + CMX_DB_COL + (uint32_t)j0, dbp);
          ptx::tmem_wait_ld();
#pragma unroll
          for (int q = 0; q < 4; ++q) DBP[q] = f2::pack(__uint_as_float(dbp[2 * q]), __uint_as_float(dbp[2 * q + 1]));
        }
        float z[JC];
        if (step) noise_chunk(a, j, b, j0, z);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const u64 ta = f2::pack(__uint_as_float(m[16 * h + 2 * q]), __uint_as_float(m[16 * h + 2 * q + 1]));
          const u64 tb = f2::pack(__uint_as_float(m[16 * h + 8 + 2 * q]), __uint_as_float(m[16 * h + 9 + 2 * q]));
          const u64 traw = f2::fma(XV[q], ta, tb);  // target score in image units
          float t0, t1, u0, u1;
          f2::unpack(traw, t0, t1);
          f2::unpack(U[q], u0, u1);
          u64 v = f2::pack(clipb(u0, cc.bound_model), clipb(u1, cc.bound_model));  // control u_j
          if (cc.score) v = f2::fma(f2::pack(clipb(t0, bts), clipb(t1, bts)), gs2, v);
          // tempered Langevin drift (eq/sdes.py:101-110): clip(sigma^2 / 2 (f score_target + (1 - f) score_prior))
          const u64 ps = f2::mul(f2::fma(XV[q], f2::pk(-1.0f), GM[q]), GI[q]);
          u64 dr = f2::mul(f2::fma(ps, omf2, f2::mul(f2::mul(traw, ust2), fr2)), hs2);
          float d0, d1;
          f2::unpack(dr, d0, d1);
          dr = f2::pack(clipb(d0, dclip), clipb(d1, dclip));
          if (cost_on) {  // the step that ends here
            const u64 cst = f2::fma(v, f2::pk(-1.0f), f2::fma(dr, isg2, SP[q]));
            c2 = f2::fma(cst, cst, c2);
            cdb = f2::fma(cst, DBP[q], cdb);
          }
          SN[q] = f2::fma(dr, isg2, v);
          if (step) {     // the step that starts here
            DBN[q] = f2::mul(sqdt2, f2::pack(z[2 * q], z[2 * q + 1]));
            XN[q] = f2::fma(sg2, DBN[q], f2::fma(f2::fma(v, sg2, dr), dt2, XV[q]));
          }
        }
        if (j0 + JC > d) {  // the chunk holding padded dims: keep them at zero (mu = 0, 1/var = 0 there; s must not pick up -0 / NaN)
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            float a0, a1;
            f2::unpack(SN[q], a0, a1);
            SN[q] = f2::pack(j0 + 2 * q < d ? a0 : 0.f, j0 + 2 * q + 1 < d ? a1 : 0.f);
          }
        }
        S.stu(2 * c, ulonglong2{SN[0], SN[1]});
        S.stu(2 * c + 1, ulonglong2{SN[2], SN[3]});
        if (step) {
          X.stu(2 * c, ulonglong2{XN[0], XN[1]});
          X.stu(2 * c + 1, ulonglong2{XN[2], XN[3]});
          uint32_t dbn[8];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            float a0, a1;
            f2::unpack(DBN[q], a0, a1);
            dbn[2 * q] = __float_as_uint(a0);
            dbn[2 * q + 1] = __float_as_uint(a1);
          }
          ptx::tmem_st8(mlp.tm_lane + CMX_DB_COL + (uint32_t)j0, dbn);
          if (a.traj_out != nullptr && live) {
            float xn[JC];
#pragma unroll
            for (int q = 0; q < 4; ++q) f2::unpack(XN[q], xn[2 * q], xn[2 * q + 1]);
            store_traj(a, j + 1, b, j0, xn);
          }
        }
      }
    }
    if (cost_on) {
      rnd += 0.5f * f2::hsum1(c2) * dt_prev;  // oc.py:740
      rnd += f2::hsum1(cdb);                  // oc.py:741
    }
  }
  __syncwarp();  // the partner lane's final coordinates
  {
    float rt[MIX_MAX_M];
    rnd -= clipf(gmm_pass1_pair(tv, d, dp, X, rt), s.clip_target);  // oc.py:750
  }
  float xsum = 0.f;
  if (live) {
    a.rnd_out[b] = rnd;
    if (a.x_out != nullptr)
      for (int j = 0; j < d; ++j) {
        const float v = X(j);
        xsum += v;
        a.x_out[(int64_t)b * d + j] = v;
      }
  }
  report_status(s, live, mlp.saturated(), !isfinite(rnd + xsum));
  tc_cta_end(warp, tmem, tmem_cols);
}

// shared memory: [weight image | barriers | counters | target mixture | x and s columns]
inline bool plan_rollout_cmcd_mix(const lrds_spec& s, int smem_cap, int sms, TcPlan* out) {
  if (!cmcd_mix_applicable(s)) return false;
  const TcLayout TL = tc_layout(s.d, s.mlp.num_hidden, s.precision);
  if (TL.tile_cols != 128) return false;
  const StageLayout SL = stage_layout(s, 2, true);
  const size_t fixed = (size_t)TL.bytes + TC_TAIL_BYTES + MIX_TAIL_BYTES + ((SL.off_buf + 15u) & ~15u);
  const size_t per_warp = (size_t)2 * s.mlp.d_pad * 32 * sizeof(float);
  if (fixed + per_warp > (size_t)smem_cap) return false;
  int wmax = (int)(((size_t)smem_cap - fixed) / per_warp);
  wmax = wmax < CMX_MAX_WARPS ? wmax : CMX_MAX_WARPS;
  const int need = (s.B + 31) / 32;
  const int w = plan_warps(need, sms, wmax);
  out->warps = w;
  out->grid = (need + w - 1) / w;
  out->staged = 2;
  out->tmem_cols = plan_tmem_cols((w + 3) / 4 * (int)CMX_TILE_COLS);
  out->smem = fixed + per_warp * w;
  return true;
}

}  // namespace lrds
