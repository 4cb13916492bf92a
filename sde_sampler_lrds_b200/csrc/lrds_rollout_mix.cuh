// The LRDS benchmark loop with BOTH dense contractions of a step on the tensor core: the drift network
// (lrds_rollout_tc.cuh) and the mixture-score contractions
//     score_j = sum_m r_m mu_mj / var_mj  -  x_j sum_m r_m / var_mj          (distr/gauss.py:97-107)
// of the target mixture (ScoreCtrl, models/reparam.py:112-117) and of the time-marginal reference mixture
// (eq/sdes.py:329-345), as [128 x 16] . [16 x 16] fp16 (hi, lo) 3-pass GEMMs per 8-dim chunk.  The responsibilities
// r = softmax_m(logc_m - q_m / 2) stay on the SIMT pipes: their quadratic forms q_m cannot be expanded into a GEMM
// at fp32 parity (cancellation).  They never touch shared memory: registers -> TMEM (A operand) -> accumulator.
//
// Configuration: LINEAR kind, exponential-integrator / DDPM-like update (LRDS_UPDATE_AXPY, LRDS_ITO_SCALED), ScoreCtrl
// over a mixture target, mixture reference, both with 2..16 components, precision F16X3 (traits_match<TraitsLrds> and
// mix_tc_applicable below); everything else runs the kernels of lrds_rollout_tc.cuh.
//
// TMEM columns of a tile (F16X3, d <= 64; wider A / D regions beyond): [0,32) A hi | [32,64) A lo | [64,128) accumulator D.  After the output
// GEMM of the network the A region is free: [0,32) holds R = (r_target hi | lo | r_reference hi | lo), 8 packed columns
// each, [32,64) the 8-dim chunk of the contraction (target a8 b8 | reference a8 b8) while D still holds the network's
// output.  One chunk is in flight at a time: chunk c+1 is issued as soon as every warp of the tile has read chunk c.
//
// Hand-offs.  A tile's tensor-core batches (the network's GEMMs, the logit GEMM, the contraction chunks) are issued by
// its last warp: every warp stores its operand rows / reads its accumulator rows, increments the tile's shared-memory
// counter (release) and goes on; the issuer warp polls the counter (acquire), issues the batch from warp-uniform
// registers (elect.sync) and commits it to the tile's mbarrier, on which the tile's warps wait only when they need
// the result.  With 14 warps per SM the last warp of a full tile sits on a sub-partition with three particle warps
// instead of four, so the issue work stays off the sub-partitions that bound the kernel.  The per-step operand buffers are refilled (TMA) by the CTA's last warp to finish a
// step.  There is no CTA-wide or tile-wide barrier inside the time loop: warps run out of phase.
//
// Responsibilities.  r = softmax_m(logc_m - q_m / 2).  For a mixture whose modes share their variances (every
// ManyModes / TwoModes target of the reference, and the VP time-marginal of a reference built from one) the x^2 term of
// q_m is mode-independent, so logit_m = c_m + x . wc_m up to a common shift: one more [128 x K] . [K x 16] GEMM per
// mixture on the x operand the network's first GEMM needs anyway.  Its rounding error grows with |x| |wc| (fp32
// accumulation of large terms), which only matters when two modes are close to a tie; so every particle checks the
// bound  (kappa |x|_2 max_m |wc_m|_2 + kappa_c max_m |c_m|) min(1, 4 (1 - r_max)) <= tau  and a warp with one particle over it
// (or a mixture with per-mode variances) evaluates the exact quadratic forms on the SIMT pipes instead
// (gmm_pass1_pair), behind the first two GEMMs of the network.
#pragma once
#include "lrds_rollout_tc.cuh"

namespace lrds {

constexpr int MIX_MAX_WARPS = 16;   // 3.5 tiles = 14 warps: one wave for 65536 particles on 148 SMs (128 registers)
constexpr int MIX_TAIL_BYTES = 32;  // the kernel's hand-off counters: tile[4] | step buffer[2]
constexpr float MIX_LOGIT_KAPPA = 9.5367431640625e-07f;  // 2^-20: error of a 3-pass fp16 dot product per unit of |x|_2 |wc|_2 (emulated worst case 2^-21.4)
constexpr float MIX_LOGIT_KAPPA_C = 2.384185791015625e-07f;  // 2^-22: c_m enters by one fp32 rounding of itself and one of the sum
constexpr float MIX_LOGIT_TAU = 2e-5f;                   // accepted logit error where modes tie (= the exact forms' own fp32 error at q ~ 50)

// Compile-time configuration of the kernel: which of the two score contractions run on the tensor core, and the update.
//   TGT  1: ScoreCtrl over a mixture target (contraction on tcgen05)   2: ScoreCtrl over the PhiFour lattice (stencil)
//        0: ClippedCtrl (no target score)
//   REF  2: the time-marginal reference is a mixture (contraction on tcgen05)   1: a single Gaussian (one FMA per dim)
//        0: no reference control (PIS / DDS over a mixture target)
//   EM   Euler-Maruyama update and Ito term (losses/oc.py:277-284) instead of the exponential-integrator axpy
//   DIS  the control is one of the DIS parametrisations over a mixture target (TGT 1): CancelDriftCtrl or LerpCtrl
//        (models/reparam.py:131-147, 189-199; which one is a warp-uniform run-time switch)
template <bool EUBO_, int TGT_, int REF_, bool EM_, bool DIS_ = false>
struct MixCfg {
  static constexpr bool kEubo = EUBO_, kEm = EM_, kDis = DIS_;
  static constexpr int kTgt = TGT_, kRef = REF_;
};
using MixBench = MixCfg<false, 1, 2, false>;  // the benchmark configuration

// index of the configuration that serves `s` (see launch_mix_f16x3), or -1
__host__ __device__ inline int mix_tc_config(const lrds_spec& s) {
  if (s.precision != LRDS_PRECISION_F16X3 || s.mlp.d_pad > 128 || gmm_full_on_path(s)) return -1;
  const bool tmix = s.ctrl_kind == LRDS_CTRL_SCORE && s.target.kind == LRDS_DISTR_GMM && s.target.gmm.M > 1 &&
                    s.target.gmm.M <= MIX_MAX_M && s.target.gmm.mix_tc != nullptr;
  const bool tdis = s.ctrl_kind >= LRDS_CTRL_CANCEL_DRIFT && s.target.kind == LRDS_DISTR_GMM && s.target.gmm.M > 1 &&
                    s.target.gmm.M <= MIX_MAX_M && s.target.gmm.mix_tc != nullptr;
  const bool tphi = s.ctrl_kind == LRDS_CTRL_SCORE && s.target.kind == LRDS_DISTR_PHI4;
  const bool tnone = s.ctrl_kind == LRDS_CTRL_CLIPPED &&
                     (s.target.kind != LRDS_DISTR_GMM || s.target.gmm.M <= MIX_MAX_M) && s.target.kind != LRDS_DISTR_LOGREG;
  const bool rnone = !s.has_ref_ctrl;
  const bool rmix = s.has_ref_ctrl && s.ref_t.M > 1 && s.ref_t.M <= MIX_MAX_M && s.ref_t.mix_tc != nullptr;
  const bool rgauss = s.has_ref_ctrl && s.ref_t.M == 1;
  const bool axpy = s.update_form == LRDS_UPDATE_AXPY && (s.ito_form == LRDS_ITO_SCALED || (rnone && s.ito_form != LRDS_ITO_EM));
  // Euler-Maruyama; without a reference control also with the Ito term switched off (DIS with compute_weights=False)
  const bool em = s.update_form == LRDS_UPDATE_EM && (s.ito_form == LRDS_ITO_EM || (rnone && s.ito_form == LRDS_ITO_NONE));
  if (s.ref_0.M > MIX_MAX_M) return -1;
  if (s.target.kind == LRDS_DISTR_GMM && s.target.gmm.M > 1 && s.target.gmm.mix_tc == nullptr) return -1;  // staged with the target
  if (s.kind == LRDS_ROLLOUT_EUBO_LINEAR) return (tmix && rmix && axpy) ? 1 : -1;
  if (s.kind != LRDS_ROLLOUT_LINEAR) return -1;
  if (tmix && rmix && axpy) return 0;
  if (tmix && rgauss && axpy) return 2;
  if (tmix && rgauss && em) return 3;
  if (tphi && rmix && axpy) return 4;
  if (tnone && rmix && axpy) return 5;
  if (tmix && rmix && em) return 6;
  if (tmix && rnone && em) return 7;    // PIS over a mixture target
  if (tmix && rnone && axpy) return 8;  // DDS over a mixture target (any Ito form but EM)
  if (tphi && rgauss && axpy) return 9;
  if (tdis && rnone && em) return 10;   // DIS with CancelDriftCtrl / LerpCtrl over a mixture target
  return -1;
}
__host__ __device__ inline bool mix_tc_applicable(const lrds_spec& s) { return mix_tc_config(s) >= 0; }

// log-density of a reference / prior block that may be a single Gaussian (the terminal cost)
__device__ __forceinline__ float gmm_logp_any(const GmmView& g, int d, int dp, const Col4& x) {
  if (g.M == 1) {
    const int nq = (d + 3) >> 2;
    float q = 0.f;
    for (int c = 0; c < nq; ++c) quad4(q, x.ld4(c), g.mu.ld4(c), g.ivar.ld4(c));
    return g.glogc.ld1(0) - 0.5f * q;
  }
  float r[MIX_MAX_M];
  return gmm_pass1_pair(g, d, dp, x, r);
}

// Optional phase timers (-DLRDS_MIX_TIMING, tools only): lane 0 of every particle warp accumulates the cycles between
// consecutive marks in shared memory; CTAs 0 and gridDim.x / 2 dump them to g_mix_timing at the end.
#ifdef LRDS_MIX_TIMING
static __device__ unsigned long long g_mix_timing[2 * 16 * 16];
struct MixTm {
  unsigned long long* w = nullptr;  // (kernels that do not collect timings leave it unset)
  long long t;
  __device__ __forceinline__ void start() { t = clock64(); }
  __device__ __forceinline__ void mark(int i) {
    const long long n = clock64();
    if (w != nullptr && (threadIdx.x & 31) == 0) w[i] += (unsigned long long)(n - t);
    t = n;
  }
  __device__ __forceinline__ void count(int i, bool hit) {  // warp-steps that evaluated the exact quadratic forms
    if (w != nullptr && (threadIdx.x & 31) == 0 && hit) w[i] += 1ull;
  }
};
#else
struct MixTm {
  __device__ __forceinline__ void start() {}
  __device__ __forceinline__ void mark(int) {}
  __device__ __forceinline__ void count(int, bool) {}
};
#endif

// ---- tensor-core side: operand stores, hand-offs, batches, accumulator reads ------------------------------------------
template <int PREC>
struct MixTc : TcMlp<PREC> {
  using Base = TcMlp<PREC>;
  static constexpr uint32_t kRCol = 0, kDCol = 32;
  uint32_t lbo, part_bytes;  // contraction image: bytes between the K chunks (modes 0-7 | 8-15), bytes of one (hi | lo) part
  uint32_t lg_part;          // logit image: bytes of one (hi | lo) part
  MixTm tm;

  // logits of mixture `which` (0 target, 1 reference): accumulator columns [16 which, 16 which + 16) <- x . wc^T
  __device__ __forceinline__ void logit(int which, uint32_t img, int col = -1) const {
    const uint32_t dcol = this->tm_tile + (col < 0 ? this->d_col() : (uint32_t)col) + (uint32_t)which * MIX_MAX_M;
    mma_passes<true, true>(dcol, this->tm_tile + this->a_col(0), this->tm_tile + this->a_col(1), 8u, img, lg_part,
                           2u * MIX_MAX_M * 16u, MIX_MAX_M * 16u, 128u, this->L.Kin / 16, ptx::make_idesc_f16(128, MIX_MAX_M));
  }
  // chunk c of the contractions -> columns [32, 64) of the tile; images = shared-window addresses of the (hi | lo) blocks
  template <bool TGT, bool REF>
  __device__ __forceinline__ void chunk(int c, uint32_t tgt_img, uint32_t ref_img, uint32_t col = kDCol, uint32_t rcol = kRCol) const {
    const uint32_t idesc = ptx::make_idesc_f16(128, 16);
#pragma unroll
    for (int which = TGT ? 0 : 1; which < (REF ? 2 : 1); ++which) {
      const uint32_t img = (which ? ref_img : tgt_img) + (uint32_t)c * 256u;  // 16 rows of 16 bytes per chunk
      const uint32_t dcol = this->tm_tile + col + which * 16;
      const uint32_t a_hi = this->tm_tile + rcol + which * 16, a_lo = a_hi + 8;
      const uint64_t b_hi = ptx::make_smem_desc(img, lbo, 128u), b_lo = ptx::make_smem_desc(img + part_bytes, lbo, 128u);
      ptx::mma_bf16_ts(dcol, a_lo, b_hi, idesc, 0);
      ptx::mma_bf16_ts(dcol, a_hi, b_lo, idesc, 1);
      ptx::mma_bf16_ts(dcol, a_hi, b_hi, idesc, 1);
    }
  }

  // r (16 responsibilities) -> packed fp16 (hi [0,8) | lo [8,16)) A-operand words
  static __device__ __forceinline__ void pack_r(const float (&r)[MIX_MAX_M], uint32_t (&p)[16]) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      u64 hi, lo;
      f2::split(f2::pack(r[2 * i], r[2 * i + 1]), hi, lo);
      float h0, h1, l0, l1;
      f2::unpack(hi, h0, h1);
      f2::unpack(lo, l0, l1);
      p[i] = ptx::pack_f16x2(h0, h1);
      p[8 + i] = ptx::pack_f16x2(l0, l1);
    }
  }
  // A operand `which` (0 target, 1 reference) of the contraction <- packed responsibilities
  __device__ __forceinline__ void store_r(int which, const uint32_t (&p)[16], uint32_t rcol = kRCol) {
    ptx::tmem_st16(this->tm_lane + rcol + which * 16, p);
  }
  __device__ __forceinline__ void load_chunk(uint32_t (&m)[32]) {
    ptx::tmem_ld32(this->tm_lane + kDCol, m);
    ptx::tmem_wait_ld();
  }

  // Responsibilities from the logit accumulator (16 raw columns `acc` of this particle).  `tail` = the logit image's
  // c_m | {un-scale, max |wc_m|_2, max |c_m|, shared}.  Returns whether the error bound accepts them for this particle.
  static __device__ __forceinline__ bool softmax_logits(const uint32_t* acc, const PPtr<true>& tail, float xnorm, uint32_t (&p)[16]) {
    float r[MIX_MAX_M];
    const float4 t2 = tail.ld4(MIX_MAX_M / 4);
#pragma unroll
    for (int q = 0; q < MIX_MAX_M / 4; ++q) {
      const float4 c = tail.ld4(q);
      r[4 * q + 0] = fmaf(__uint_as_float(acc[4 * q + 0]), t2.x, c.x);
      r[4 * q + 1] = fmaf(__uint_as_float(acc[4 * q + 1]), t2.x, c.y);
      r[4 * q + 2] = fmaf(__uint_as_float(acc[4 * q + 2]), t2.x, c.z);
      r[4 * q + 3] = fmaf(__uint_as_float(acc[4 * q + 3]), t2.x, c.w);
    }
    float mx = r[0];
#pragma unroll
    for (int i = 1; i < MIX_MAX_M; ++i) mx = fmaxf(mx, r[i]);
    float s = 0.f;
#pragma unroll
    for (int mb = 0; mb < MIX_MAX_M / 4; ++mb) {
#pragma unroll
      for (int i = 0; i < 4; ++i) r[4 * mb + i] = __expf(r[4 * mb + i] - mx);
      s += (r[4 * mb] + r[4 * mb + 1]) + (r[4 * mb + 2] + r[4 * mb + 3]);
    }
    const float inv = 1.0f / s;
#pragma unroll
    for (int i = 0; i < MIX_MAX_M; ++i) r[i] *= inv;
    pack_r(r, p);
    // 1 - r_max = (s - 1) / s (the largest term of s is exactly 1)
    const float eps = fmaf(MIX_LOGIT_KAPPA * xnorm, t2.y, MIX_LOGIT_KAPPA_C * t2.z);
    const float amb = fminf(1.0f, 4.0f * (s - 1.0f) * inv);
    return eps * amb <= MIX_LOGIT_TAU && xnorm < 3.0e4f;  // (false for NaN; beyond 3e4 the fp16 operands saturate)
  }

  // The drift network up to the completed output GEMM (A region free afterwards); the A operand x is already stored.
  // slot0 / slot1 run behind the first / second GEMM of the network (work that needs x but not the network).
  template <bool BIAS_SH, class S0, class S1>
  __device__ __forceinline__ void hidden_ws(const float* __restrict__ bias1, S0&& slot0, S1&& slot1) {
    const TcLayout& L = this->L;
    this->issue(L.off_in, L.Kin, C);
    tm.mark(1);
    slot0();
    tm.mark(2);
    const float* bh = reinterpret_cast<const float*>(this->img + L.off_bhid);
    const int nh = L.nh;
    for (int l = 0; l <= nh; ++l) {
      if (l == 1) {
        slot1();
        tm.mark(5);
      }
      this->wait();
      tm.mark(l == 0 ? 3 : l == 1 ? 6 : 8);
      if (l == 0) this->template epilogue_f16<!BIAS_SH>(bias1, 0);
      else this->template epilogue_f16<false>(bh + (l - 1) * C, l);
      if (l < nh) this->issue(L.off_hid + (uint32_t)(l * C * C * L.es), C, C);
      else this->issue(L.off_out, C, L.Nout);
      tm.mark(l == 0 ? 4 : 7);
    }
    if (nh == 0) slot1();
    this->wait();
    tm.mark(8);
  }
};

// Operands of step k -> step buffer k & 1, completion on its mbarrier (one thread): table row | reference mixture block |
// its tensor-core images; step 0 also stages the static target mixture (whether or not the control uses its score:
// the terminal cost does).  Stage layout: [step-buffer mbarriers | target | buffers] (stage_layout).
template <bool RMIX>
__device__ __forceinline__ void mix_load_step(const lrds_spec& s, const StageLayout& SL, uint8_t* stage, int k) {
  uint64_t* sbar = reinterpret_cast<uint64_t*>(stage) + (k & 1);
  uint8_t* dst = stage + SL.off_buf + (k & 1) * SL.buf_bytes;
  const bool tgt = k == 0 && SL.tgt_bytes;
  ptx::mbar_expect_tx(sbar, SL.buf_bytes + (tgt ? SL.tgt_bytes : 0u));
  if (tgt) {
    stage_gmm(stage + SL.off_tgt, gmm_at(s.target.gmm, 0), SL.tgt_logc_bytes, SL.tgt_param_bytes, sbar);
    ptx::bulk_g2s(stage + SL.off_tgt + SL.tgt_logc_bytes + SL.tgt_param_bytes, static_cast<const uint8_t*>(s.target.gmm.mix_tc),
                  SL.tgt_mix_bytes, sbar);
  }
  stage_step(dst, s, SL, k, sbar);
  if constexpr (RMIX)
    ptx::bulk_g2s(dst + SL.row_bytes + SL.ref_logc_bytes + SL.ref_param_bytes,
                  static_cast<const uint8_t*>(s.ref_t.mix_tc) + (int64_t)k * s.ref_t.step_stride_mix_tc, SL.ref_mix_bytes, sbar);
}

// ---- the loop ------------------------------------------------------------------------------------------------------
// EUBO: the noising rollout of compute_eubo (losses/oc.py:512-568): per step x <- mean x + std z first, then the
// control and the reference score at the new point enter the cost; x is not integrated by the control.  The step's
// increments are generated twice (for the update and for the cost) instead of being kept per particle.
template <int PREC, class CFG>
__device__ __forceinline__ void rollout_body_mix(const RolloutArgs& a, float* smem, uint8_t* stage, uint32_t* step_cnt, const int nwarps,
                                                 MixTc<PREC>& mlp) {
  constexpr bool EUBO = CFG::kEubo, TMIX = CFG::kTgt == 1, TPHI = CFG::kTgt == 2, RMIX = CFG::kRef == 2, RGAUSS = CFG::kRef == 1, EM = CFG::kEm, DIS = CFG::kDis;
  const lrds_spec& s = a.s;
  const int NT = nwarps * 32;  // particle threads
  const int tid = threadIdx.x;
  const int b_raw = blockIdx.x * NT + tid;
  const bool live = b_raw < s.B;
  const int b = live ? b_raw : s.B - 1;  // idle lanes shadow the last particle, results are not stored
  const int d = s.d, dp = s.mlp.d_pad, K = s.K;
  const ColLayout L = col_layout(s, true);
  const Particle P = make_particle(smem, L, NT, tid);

  for (int j = 0; j < dp; ++j) P.x(j) = (j < d) ? __ldg(a.x0 + (int64_t)b * d + j) : 0.f;
  if (!EUBO && a.traj_out != nullptr && live)
    for (int j = 0; j < d; ++j) a.traj_out[(int64_t)b * d + j] = P.x(j);

  CtrlConst cc = ctrl_const(s);
  const GmmView tv0 = gmm_at(s.target.gmm, 0);
  const StageLayout SL = stage_layout(s, 2, true);
  uint64_t* sbar = reinterpret_cast<uint64_t*>(stage);  // [i]: step buffer i filled (TMA transaction bytes)
  const uint32_t mix_off_t = SL.tgt_logc_bytes + SL.tgt_param_bytes;                // inside the target area
  const uint32_t mix_off_r = SL.row_bytes + SL.ref_logc_bytes + SL.ref_param_bytes;  // inside a step buffer
  // a block of mix_tc: [contraction hi | lo | 16 B][logit hi | lo][c_m | 16 B]  (gmm_mix_tc_bytes)
  const int Mt = TMIX ? s.target.gmm.M : s.ref_t.M;  // both are padded to 16 modes: equal block geometry
  const uint32_t contr_bytes = gmm_mix_contr_bytes(Mt, dp), lg_part = gmm_mix_logit_part_bytes(Mt, dp);
  const uint32_t lg_tail_off = contr_bytes + 2u * lg_part;
  const GmmViewT<true> tv = staged_view(stage + SL.off_tgt, tv0, SL.tgt_logc_bytes, SL.tgt_param_bytes);
  const uint32_t tgt_img = ptx::smem_u32(stage + SL.off_tgt + mix_off_t);
  mlp.lbo = (uint32_t)(2 * dp) * 16u;
  mlp.part_bytes = (contr_bytes - 16u) / 2u;
  mlp.lg_part = lg_part;
  // terminal_unnorm_log_prob(x) of whatever the target is (clipped by the caller)
  auto target_logp = [&]() -> float {
    if (s.target.kind == LRDS_DISTR_GMM) {
      if (s.target.gmm.M == 1) return gmm_logp_any(tv0, d, dp, P.x);
      float rt[MIX_MAX_M];
      return gmm_pass1_pair(tv, d, dp, P.x, rt);
    }
    if (s.target.kind == LRDS_DISTR_PHI4) return phi4_logp(s.target.phi4, d, P.x);
    return 0.f;
  };
  // lattice score (lrds_rollout_lin.cuh): x (p1 + p3 x^2) + p0 + pn ((x_{j+1} + x_{j-1}) - 2 x)
  const float coef = s.target.phi4.a * (float)d, beta = s.target.phi4.beta;
  const u64 p0 = f2::pk(-beta * s.target.phi4.b / coef), p1 = f2::pk(beta / coef), p3 = f2::pk(-beta / coef),
            pn = f2::pk(beta * coef), m2 = f2::pk(-2.0f);
  const int nchunk = dp / JC;
  const int nq = (d + 3) >> 2;
  float rnd = 0.f;
  __syncwarp();  // the quadratic forms read the partner lane's coordinates
  if constexpr (EUBO) {  // rnd = reference_log_prob(x) - terminal_unnorm_log_prob(x)   (oc.py:536)
    ptx::mbar_wait(sbar, 0);  // the staged target mixture (the same phase as the first step's buffer)
    const float lref = gmm_logp_any(gmm_at(s.ref_0, 0), d, dp, P.x);
    rnd = lref - clipf(target_logp(), s.clip_target);
  }

  mlp.tm.start();
  for (int k = 0; k < K; ++k) {
    ptx::mbar_wait(sbar + (k & 1), (uint32_t)(k >> 1) & 1u);
    mlp.tm.mark(0);
    const uint8_t* buf = stage + SL.off_buf + (k & 1) * SL.buf_bytes;
    const float* row = reinterpret_cast<const float*>(buf);
    const PPtr<true> rowp{ptx::smem_u32(buf)};
    const GmmViewT<true> rv = staged_view(buf + SL.row_bytes, gmm_at(s.ref_t, k), SL.ref_logc_bytes, SL.ref_param_bytes);
    const uint32_t ref_img = ptx::smem_u32(buf + mix_off_r);
    const float A = rowp.ld1(LRDS_STEP_A), Bc = rowp.ld1(LRDS_STEP_B), Cc = rowp.ld1(LRDS_STEP_C);
    const float wcost = rowp.ld1(LRDS_STEP_W_COST), wito = rowp.ld1(LRDS_STEP_W_ITO);
    const float gamma = rowp.ld1(LRDS_STEP_GAMMA);
    const float ust = TMIX ? *reinterpret_cast<const float*>(stage + SL.off_tgt + mix_off_t + contr_bytes - 16u) : 1.0f;
    const float usr = RMIX ? *reinterpret_cast<const float*>(buf + mix_off_r + contr_bytes - 16u) : 1.0f;
    const GmmView rg = gmm_at(s.ref_t, k);  // single-Gaussian reference: read from global memory (!RMIX)

    if constexpr (EUBO) {  // x <- mean x + std z   (oc.py:550-552)
      const u64 mean2 = f2::pk(rowp.ld1(LRDS_STEP_EU_A)), std2 = f2::pk(rowp.ld1(LRDS_STEP_EU_B));
      for (int c = 0; c < nchunk; ++c) {
        float z[JC];
        noise_chunk(a, k, b, c * JC, z);
        const ulonglong2 xa = P.x.ldu(2 * c), xb = P.x.ldu(2 * c + 1);
        P.x.stu(2 * c, ulonglong2{f2::fma(std2, f2::pack(z[0], z[1]), f2::mul(xa.x, mean2)),
                                  f2::fma(std2, f2::pack(z[2], z[3]), f2::mul(xa.y, mean2))});
        P.x.stu(2 * c + 1, ulonglong2{f2::fma(std2, f2::pack(z[4], z[5]), f2::mul(xb.x, mean2)),
                                      f2::fma(std2, f2::pack(z[6], z[7]), f2::mul(xb.y, mean2))});
      }
    }
    mlp.store_x(P.x);
    // Responsibilities of the two mixtures (packed fp16 hi | lo).  Shared-variance mixtures: from the logit GEMM, unless
    // the error bound of a particle of this warp refuses; otherwise the exact quadratic forms behind the network's GEMMs.
    // A particle's choice depends on its own bound only (results must not depend on which particles share a warp);
    // the exact forms are evaluated by the whole warp (the half-warps serve each other) as soon as one lane needs them.
    uint32_t rt_p[16], rr_p[16];
    bool need_t = TMIX, need_r = RMIX;   // warp-uniform: some lane needs the exact forms
    bool ok_t = false, ok_r = false;     // this lane keeps the responsibilities of the logit GEMM
    if constexpr (TMIX || RMIX) {
      const PPtr<true> tail_t{tgt_img + lg_tail_off}, tail_r{ref_img + lg_tail_off};
      const bool lg_t = TMIX && tail_t.ld1(MIX_MAX_M + 3) != 0.f, lg_r = RMIX && tail_r.ld1(MIX_MAX_M + 3) != 0.f;  // CTA-uniform
      if (lg_t || lg_r) {
        mlp.arrive_issue([&]() {
          if (lg_t) mlp.logit(0, tgt_img + contr_bytes);
          if (lg_r) mlp.logit(1, ref_img + contr_bytes);
        });
        u64 n2 = 0;  // |x|^2 while the batch runs
        for (int c = 0; c < nq; ++c) {
          const ulonglong2 xv = P.x.ldu(c);
          n2 = f2::fma(xv.x, xv.x, n2);
          n2 = f2::fma(xv.y, xv.y, n2);
        }
        const float xnorm = sqrtf(f2::hsum1(n2));
        mlp.wait();
        uint32_t lg[32];
        ptx::tmem_ld32(mlp.tm_lane + mlp.d_col(), lg);
        ptx::tmem_wait_ld();
        if (lg_t) {
          ok_t = mlp.softmax_logits(lg, tail_t, xnorm, rt_p);
          need_t = __any_sync(0xffffffffu, !ok_t);
        }
        if (lg_r) {
          ok_r = mlp.softmax_logits(lg + MIX_MAX_M, tail_r, xnorm, rr_p);
          need_r = __any_sync(0xffffffffu, !ok_r);
        }
      }
    }
    mlp.tm.count(14, need_t);
    mlp.tm.count(15, need_r);
    mlp.template hidden_ws<true>(
        row + LRDS_STEP_BIAS1,
        [&]() {
          if constexpr (TMIX) {
            if (need_t) {
              float r[MIX_MAX_M];
              uint32_t p[16];
              gmm_pass1_pair(tv, d, dp, P.x, r);
              mlp.pack_r(r, p);
#pragma unroll
              for (int i = 0; i < 16; ++i) rt_p[i] = ok_t ? rt_p[i] : p[i];
            }
          }
        },
        [&]() {
          if constexpr (RMIX) {
            if (need_r) {
              float r[MIX_MAX_M];
              uint32_t p[16];
              gmm_pass1_pair(rv, d, dp, P.x, r);
              mlp.pack_r(r, p);
#pragma unroll
              for (int i = 0; i < 16; ++i) rr_p[i] = ok_r ? rr_p[i] : p[i];
            }
          }
        });
    // the output GEMM is complete: the A region is free for the responsibilities and the contraction chunks
    if constexpr (TMIX) mlp.store_r(0, rt_p);
    if constexpr (RMIX) mlp.store_r(1, rr_p);
    mlp.arrive_issue([&]() { mlp.template chunk<TMIX, RMIX>(0, tgt_img, ref_img); });
    mlp.tm.mark(9);
    // The integrator update on packed fp32x2 pairs of dims.  The images hold -1/var, so a score is one FFMA2; their
    // power-of-two un-scales are folded into the ScoreCtrl factor / the clip bound (target) and into the FFMA that
    // adds the control (reference).  Padded dims need no masks: their image rows, output weights, biases and noise
    // are zero, so u = scores = z = 0 and x stays 0.
    // update x' = ca x + cr r + cu u + cz z:  axpy (A, B, B, C);  EM x + ((-(f x) + sigma^2 r) + sigma u) dt + sigma (z sqrt dt)
    const float dt = EM ? rowp.ld1(LRDS_STEP_DT) : 0.f, sqdt = EM ? rowp.ld1(LRDS_STEP_SQRT_DT) : 0.f;
    const u64 A2 = f2::pk(EM ? 1.0f - A * dt : A), B2 = f2::pk(EM ? Bc * dt : Bc), C2 = f2::pk(EM ? Bc * sqdt : Cc);
    const u64 usr2 = f2::pk(usr), R2 = f2::pk((EM ? Cc * dt : Bc) * usr);
    // DIS parametrisations: u = (clip(net) + CX x) + GSCALE ((scale clip(sc)) gamma), sc = the target score (CancelDriftCtrl)
    // or lerp(prior score, target score, LERP) evaluated in true units (LerpCtrl)
    const bool lerp = DIS && s.ctrl_kind == LRDS_CTRL_LERP;
    const float gsc = DIS ? rowp.ld1(LRDS_STEP_GSCALE) : 1.0f, wl = DIS ? rowp.ld1(LRDS_STEP_LERP) : 0.f;
    const u64 cx2 = f2::pk(DIS ? rowp.ld1(LRDS_STEP_CX) : 0.f), ust2 = f2::pk(ust);
    const u64 wl2 = f2::pk(wl < 0.5f ? wl : -(1.0f - wl));
    const GmmView pg = gmm_at(s.ref_0, 0);  // LerpCtrl: the prior (a diagonal Gaussian)
    const u64 gs2 = f2::pk(((cc.scale_score * gamma) * gsc) * (lerp ? 1.0f : ust));
    const float bts = lerp ? cc.bound_score : cc.bound_score / ust;
    // weight of sum(u z) in the log-weight (oc.py:284 / 499); without a reference control also the DDS forms (oc.py:1380-1383)
    const float wz = EM ? (s.ito_form == LRDS_ITO_NONE ? 0.f : sqdt)
                     : (RMIX || RGAUSS || s.ito_form == LRDS_ITO_SCALED) ? wito
                     : s.ito_form == LRDS_ITO_DDS ? rowp.ld1(LRDS_STEP_SIGU) * wito
                                                  : 0.f;
    u64 su2 = 0, sito = 0;
    float xm = 0.f;  // lattice target: x_{j0-1} of the state before this step's update
    for (int c = 0; c < nchunk; ++c) {
      const int j0 = c * JC;
      uint32_t m[32];
      mlp.wait();
      mlp.tm.mark(10);
      mlp.load_chunk(m);
      if (c + 1 < nchunk) mlp.arrive_issue([&]() { mlp.template chunk<TMIX, RMIX>(c + 1, tgt_img, ref_img); });
      mlp.tm.mark(11);
      const ulonglong2 xa = P.x.ldu(2 * c), xb = P.x.ldu(2 * c + 1);
      const u64 X[4] = {xa.x, xa.y, xb.x, xb.y};
      u64 U[4], XN[4];
      float z[JC];
      mlp.out_chunk2(j0, U);
      noise_chunk(a, k, b, j0, z);
      float xs[JC + 2];  // lattice target: the chunk with its two neighbours (state before the update)
      if constexpr (TPHI) {
        xs[0] = xm;
#pragma unroll
        for (int q = 0; q < 4; ++q) f2::unpack(X[q], xs[1 + 2 * q], xs[2 + 2 * q]);
        xs[JC + 1] = (j0 + JC < dp) ? P.x(j0 + JC) : 0.f;
        xm = xs[JC];
      }
      u64 GM[4], GI[4];  // single-Gaussian reference: mean and 1/var of the chunk
      if constexpr (RGAUSS) {
        const ulonglong2 g0 = rg.mu.ld2(2 * c), g1 = rg.mu.ld2(2 * c + 1), i0 = rg.ivar.ld2(2 * c), i1 = rg.ivar.ld2(2 * c + 1);
        GM[0] = g0.x; GM[1] = g0.y; GM[2] = g1.x; GM[3] = g1.y;
        GI[0] = i0.x; GI[1] = i0.y; GI[2] = i1.x; GI[3] = i1.y;
      }
      if constexpr (DIS) {
        if (lerp) {
          const ulonglong2 g0 = pg.mu.ld2(2 * c), g1 = pg.mu.ld2(2 * c + 1), i0 = pg.ivar.ld2(2 * c), i1 = pg.ivar.ld2(2 * c + 1);
          GM[0] = g0.x; GM[1] = g0.y; GM[2] = g1.x; GM[3] = g1.y;
          GI[0] = i0.x; GI[1] = i0.y; GI[2] = i1.x; GI[3] = i1.y;
        }
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const u64 ta = f2::pack(__uint_as_float(m[2 * q]), __uint_as_float(m[2 * q + 1]));
        const u64 tb = f2::pack(__uint_as_float(m[8 + 2 * q]), __uint_as_float(m[9 + 2 * q]));
        const u64 ra = f2::pack(__uint_as_float(m[16 + 2 * q]), __uint_as_float(m[17 + 2 * q]));
        const u64 rb = f2::pack(__uint_as_float(m[24 + 2 * q]), __uint_as_float(m[25 + 2 * q]));
        float t0 = 0.f, t1 = 0.f, u0, u1;
        if constexpr (TMIX) f2::unpack(f2::fma(X[q], ta, tb), t0, t1);  // raw target score (image units)
        if constexpr (DIS) {
          if (lerp) {  // torch.lerp(prior_score, target_score, w): a + w (b - a) for w < 1/2, else b - (b - a)(1 - w)
            const u64 tt = f2::mul(f2::pack(t0, t1), ust2);
            const u64 pr = f2::mul(f2::fma(X[q], f2::pk(-1.0f), GM[q]), GI[q]);
            const u64 df = f2::fma(pr, f2::pk(-1.0f), tt);
            f2::unpack(f2::fma(df, wl2, wl < 0.5f ? pr : tt), t0, t1);
          }
        }
        if constexpr (TPHI) {
          const u64 nb = f2::pack(xs[2 * q] + xs[2 * q + 2], xs[2 * q + 1] + xs[2 * q + 3]);
          const u64 t = f2::fma(X[q], f2::fma(f2::mul(X[q], X[q]), p3, p1), f2::fma(pn, f2::fma(X[q], m2, nb), p0));
          f2::unpack(t, t0, t1);
          if (j0 + JC > d) {  // padded lattice sites have no score
            if (j0 + 2 * q >= d) t0 = 0.f;
            if (j0 + 2 * q + 1 >= d) t1 = 0.f;
          }
        }
        f2::unpack(U[q], u0, u1);
        const u64 uc = f2::pack(clipb(u0, cc.bound_model), clipb(u1, cc.bound_model));
        u64 v = uc;  // control u
        if constexpr (DIS) v = f2::fma(X[q], cx2, v);
        if constexpr (TMIX || TPHI) v = f2::fma(f2::pack(clipb(t0, bts), clipb(t1, bts)), gs2, v);
        // reference score in the units of R2: mixture = accumulator (image units), Gaussian = -(x - mu) / var
        const u64 rraw = RMIX ? f2::fma(X[q], ra, rb) : RGAUSS ? f2::mul(f2::fma(X[q], f2::pk(-1.0f), GM[q]), GI[q]) : 0ull;
        const u64 z2 = f2::pack(z[2 * q], z[2 * q + 1]);
        if constexpr (EUBO) {  // cost += u (r + u / 2),  gz += u z   (oc.py:556-563; g = u for the axpy updates)
          su2 = f2::fma(v, f2::fma(v, f2::pk(0.5f), f2::mul(rraw, usr2)), su2);
          sito = f2::fma(v, z2, sito);
          continue;
        }
        su2 = f2::fma(v, v, su2);
        sito = f2::fma(v, z2, sito);
        if constexpr (!RMIX && !RGAUSS) {
          XN[q] = f2::fma(C2, z2, f2::fma(A2, X[q], f2::mul(B2, v)));
        } else if constexpr (EM) {
          XN[q] = f2::fma(C2, z2, f2::fma(A2, X[q], f2::fma(R2, rraw, f2::mul(B2, v))));
        } else {
          const u64 rv2 = f2::fma(rraw, usr2, v);  // reference score + u
          XN[q] = f2::fma(C2, z2, f2::fma(A2, X[q], f2::mul(B2, rv2)));
        }
      }
      if constexpr (EUBO) {
        mlp.tm.mark(12);
        continue;
      }
      P.x.stu(2 * c, ulonglong2{XN[0], XN[1]});
      P.x.stu(2 * c + 1, ulonglong2{XN[2], XN[3]});
      if (a.traj_out != nullptr && live) {
        float xn[JC];
#pragma unroll
        for (int q = 0; q < 4; ++q) f2::unpack(XN[q], xn[2 * q], xn[2 * q + 1]);
        store_traj(a, k + 1, b, j0, xn);
      }
      mlp.tm.mark(12);
    }
    if constexpr (EUBO) {
      rnd -= f2::hsum1(su2) * wcost;
      rnd -= f2::hsum1(sito) * wito;
    } else {
      rnd += wcost * f2::hsum1(su2);
      rnd += wz * f2::hsum1(sito);
    }
    // This warp is done with the step's buffer (the last contraction, which reads its image, has completed: wait()
    // above).  The CTA's last warp to get here refills it with the operands of step k + 2.
    __syncwarp();
    if ((tid & 31) == 0) {
      const uint32_t old = ptx::atom_add_acq_rel(step_cnt + (k & 1), 1u);
      if (old == (uint32_t)((k >> 1) * nwarps + nwarps - 1) && k + 2 < K) mix_load_step<RMIX>(s, SL, stage, k + 2);
    }
    mlp.tm.mark(13);
  }
  __syncwarp();  // the partner lane's final coordinates
  if constexpr (!EUBO) {  // terminal cost: rnd += reference_log_prob(x) - terminal_unnorm_log_prob(x)   (oc.py:290, 505, 645)
    // init_cost (DIS): the pre-pass of lrds_rollout left initial_log_prob(x_0) + rnd_offset in rnd_out (oc.py:1164-1168)
    const float lref = s.init_cost ? a.rnd_out[b] : gmm_logp_any(gmm_at(s.ref_0, 0), d, dp, P.x);
    rnd += lref - clipf(target_logp(), s.clip_target);
  }

  float xsum = 0.f;
  if (live) {
    a.rnd_out[b] = rnd;
    if (a.x_out != nullptr)
      for (int j = 0; j < d; ++j) {
        const float v = P.x(j);
        xsum += v;
        a.x_out[(int64_t)b * d + j] = v;
      }
  }
  report_status(s, live, mlp.saturated(), !isfinite(rnd + xsum));
}

// The auxiliary warp of a CTA whose last tile is partial: it owns no particles and issues that tile's batches, in the
// order the tile's warps hand them off (rollout_body_mix), so that the issue work stays off the tile's own warps - both
// of which share their SM sub-partitions with three other particle warps and would otherwise bound the kernel.
template <int PREC, class CFG>
__device__ __forceinline__ void mix_aux_issuer(const RolloutArgs& a, uint8_t* stage, MixTc<PREC>& mlp) {
  constexpr bool TMIX = CFG::kTgt == 1, RMIX = CFG::kRef == 2;
  const lrds_spec& s = a.s;
  const int dp = s.mlp.d_pad, K = s.K, nchunk = dp / JC, nh = mlp.L.nh;
  const StageLayout SL = stage_layout(s, 2, true);
  uint64_t* sbar = reinterpret_cast<uint64_t*>(stage);
  const uint32_t mix_off_t = SL.tgt_logc_bytes + SL.tgt_param_bytes;
  const uint32_t mix_off_r = SL.row_bytes + SL.ref_logc_bytes + SL.ref_param_bytes;
  const int Mt = TMIX ? s.target.gmm.M : s.ref_t.M;
  const uint32_t contr_bytes = gmm_mix_contr_bytes(Mt, dp), lg_part = gmm_mix_logit_part_bytes(Mt, dp);
  const uint32_t lg_tail_off = contr_bytes + 2u * lg_part;
  const uint32_t tgt_img = ptx::smem_u32(stage + SL.off_tgt + mix_off_t);
  mlp.lbo = (uint32_t)(2 * dp) * 16u;
  mlp.part_bytes = (contr_bytes - 16u) / 2u;
  mlp.lg_part = lg_part;
  const TcLayout& L = mlp.L;
  for (int k = 0; k < K; ++k) {
    ptx::mbar_wait(sbar + (k & 1), (uint32_t)(k >> 1) & 1u);  // the step's flags and images (read-only use)
    const uint8_t* buf = stage + SL.off_buf + (k & 1) * SL.buf_bytes;
    const uint32_t ref_img = ptx::smem_u32(buf + mix_off_r);
    if constexpr (TMIX || RMIX) {
      const PPtr<true> tail_t{tgt_img + lg_tail_off}, tail_r{ref_img + lg_tail_off};
      const bool lg_t = TMIX && tail_t.ld1(MIX_MAX_M + 3) != 0.f, lg_r = RMIX && tail_r.ld1(MIX_MAX_M + 3) != 0.f;
      if (lg_t || lg_r)
        mlp.issue_when_ready([&]() {
          if (lg_t) mlp.logit(0, tgt_img + contr_bytes);
          if (lg_r) mlp.logit(1, ref_img + contr_bytes);
        });
    }
    mlp.issue_when_ready([&]() { mlp.gemm(L.off_in, L.Kin, C); });
    for (int l = 0; l < nh; ++l) mlp.issue_when_ready([&]() { mlp.gemm(L.off_hid + (uint32_t)(l * C * C * L.es), C, C); });
    mlp.issue_when_ready([&]() { mlp.gemm(L.off_out, C, L.Nout); });
    for (int c = 0; c < nchunk; ++c) mlp.issue_when_ready([&]() { mlp.template chunk<TMIX, RMIX>(c, tgt_img, ref_img); });
  }
}

// shared memory: [weight image | mbarriers + TMEM slot | hand-off counters | operand stage | particle columns]
template <int PREC, class CFG>
__global__ void __launch_bounds__(MIX_MAX_WARPS * 32, 1)
rollout_mix_kernel(const RolloutArgs a, const uint8_t* __restrict__ image, const uint32_t tmem_cols, const int nwarps) {
  // nwarps = particle warps; blockDim.x / 32 = nwarps + 1 when the last tile is partial (the auxiliary issuer warp)
  extern __shared__ __align__(128) uint8_t smem_raw[];
  constexpr bool RMIX = CFG::kRef == 2;
  const lrds_spec& s = a.s;
  const TcLayout TL = tc_layout(s.d, s.mlp.num_hidden, PREC);
  const int tid = threadIdx.x;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);  // warp-uniform for the compiler as well
  const bool has_aux = (int)(blockDim.x >> 5) > nwarps;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + TL.bytes);  // [0] image, [1 + t] MMAs of tile t done
  uint32_t* cnts = reinterpret_cast<uint32_t*>(smem_raw + TL.bytes + TC_TAIL_BYTES);  // [t] tile hand-offs, [4 + i] step buffer i released
  uint8_t* stage = smem_raw + TL.bytes + TC_TAIL_BYTES + MIX_TAIL_BYTES;
  const StageLayout SL = stage_layout(s, 2, true);
  float* cols = reinterpret_cast<float*>(stage + ((SL.total + 15u) & ~15u));
  auto steps01 = [&]() {  // the static target mixture and steps 0, 1, staged with the drift weights
    for (int k = 0; k < 2 && k < s.K; ++k) mix_load_step<RMIX>(s, SL, stage, k);
  };
  const uint32_t tmem = __shfl_sync(
      0xffffffffu, tc_cta_begin(smem_raw, TL, image, tmem_cols, warp, 5, reinterpret_cast<uint64_t*>(stage), 2, cnts, 6, 0u, steps01), 0);
  const bool aux = warp == nwarps;              // the auxiliary issuer serves the partial last tile
  const int tile = aux ? (nwarps - 1) >> 2 : warp >> 2;
  const int tile_warps = min(4, nwarps - 4 * tile);
  // even hand-offs: the tile's last warp; odd ones: the one before it (the same warp in a one-warp tile); none in a
  // partial tile served by the auxiliary warp
  uint32_t issue_mask = ((warp & 3) == tile_warps - 1 ? 1u : 0u) | ((warp & 3) == max(tile_warps - 2, 0) ? 2u : 0u);
  if (has_aux && tile_warps < 4) issue_mask = 0u;
  MixTc<PREC> mlp;
  mlp.init(TL, smem_raw, tmem + (uint32_t)(tile * TL.tile_cols), warp, bars + 1 + tile, cnts + tile, (uint32_t)tile_warps, issue_mask,
           s.mlp.d_pad);
#ifdef LRDS_MIX_TIMING
  unsigned long long* tmw = reinterpret_cast<unsigned long long*>(cols + (size_t)col_layout(s, true).total * 32 * nwarps) + warp * 16;
  if ((tid & 31) < 16) tmw[tid & 31] = 0;
  __syncwarp();
  mlp.tm.w = tmw;
#endif
  if (aux) mix_aux_issuer<PREC, CFG>(a, stage, mlp);
  else rollout_body_mix<PREC, CFG>(a, cols, stage, cnts + 4, nwarps, mlp);
#ifdef LRDS_MIX_TIMING
  __syncwarp();
  if ((blockIdx.x == 0 || blockIdx.x == gridDim.x / 2) && (tid & 31) < 16)
    g_mix_timing[((blockIdx.x ? 1 : 0) * 16 + warp) * 16 + (tid & 31)] = tmw[tid & 31];
#endif
  tc_cta_end(warp, tmem, tmem_cols);
}

// Launch shape of the mix kernel: one CTA per SM, warps per CTA as plan_warps picks them.
inline bool plan_rollout_mix(const lrds_spec& s, int smem_cap, int sms, TcPlan* out) {
  if (!mix_tc_applicable(s)) return false;
  const TcLayout TL = tc_layout(s.d, s.mlp.num_hidden, s.precision);
  if (TL.tile_cols > 512 || TL.parts * TL.a_cols < 64) return false;  // R and the chunk live in 64 columns of the A region
  const ColLayout CL = col_layout(s, true);
  size_t fixed = (size_t)TL.bytes + TC_TAIL_BYTES + MIX_TAIL_BYTES + ((stage_layout(s, 2, true).total + 15u) & ~15u);
#ifdef LRDS_MIX_TIMING
  fixed += 16 * 16 * 8;
#endif
  const size_t per_warp = (size_t)CL.total * 32 * sizeof(float);
  if (fixed + per_warp > (size_t)smem_cap) return false;
  int wmax = (int)(((size_t)smem_cap - fixed) / per_warp);
  wmax = wmax < MIX_MAX_WARPS ? wmax : MIX_MAX_WARPS;
  wmax = wmax < 4 * (512 / TL.tile_cols) ? wmax : 4 * (512 / TL.tile_cols);
  const int need = (s.B + 31) / 32;
  const int w = plan_warps(need, sms, wmax);
  out->warps = w;
  out->grid = (need + w - 1) / w;
  out->staged = 2;
  out->tmem_cols = plan_tmem_cols((w + 3) / 4 * TL.tile_cols);
  out->smem = fixed + per_warp * w;
  return true;
}

template <class CFG>
int launch_mix_cfg(const RolloutArgs& a, const TcPlan& p, cudaStream_t st) {
  // a partial last tile gets the auxiliary issuer warp when the CTA has room for it
  const int aux = (p.warps % 4 != 0 && p.warps < MIX_MAX_WARPS) ? 1 : 0;
  return launch_tc(rollout_mix_kernel<LRDS_PRECISION_F16X3, CFG>, "mixture tensor-core rollout", a, p, (p.warps + aux) * 32, st,
                   p.tmem_cols, p.warps);
}

}  // namespace lrds
