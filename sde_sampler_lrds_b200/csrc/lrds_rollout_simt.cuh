// The rollout body: one thread integrates one particle through all K steps.  Particle state (x, mixture
// responsibilities, CMCD carry-over) lives in shared-memory columns for the whole rollout; HBM is touched only
// for x0, the optional recorded noise / trajectory, and the results.  Per-step tables and distribution
// parameters are warp-uniform broadcast loads served by L1/L2.
//
// The drift network is a policy (template parameter MLP) with two hooks:
//   mlp.hidden(bias1, x)      run the network up to (and, on tensor cores, including) the output GEMM
//   mlp.out_chunk(j0, out)    out_layer(x)[j0 .. j0+8) including its bias
// SimtMlp (below) is the fp32 FFMA parity anchor (LRDS_PRECISION_FP32_SIMT); TcMlp (lrds_rollout_tc.cuh) runs the
// four GEMMs on tcgen05 with TMEM-resident operands.  Everything else is shared between the two.
#pragma once
#include "lrds_device.cuh"
#include "lrds_tc_ptx.cuh"

namespace lrds {

struct RolloutArgs {
  lrds_spec s;
  const float* x0;
  const float* noise;
  uint64_t seed;
  uint64_t particle_offset;
  float* x_out;
  float* rnd_out;
  float* traj_out;
};

// spec.status (include/lrds_b200.h): [0] += this thread saw a saturating fp16 operand, [1] += non-finite result
__device__ __forceinline__ void report_status(const lrds_spec& s, bool live, bool saturated, bool nonfinite) {
  if (s.status != nullptr && live) {
    if (saturated) atomicAdd(s.status, 1u);
    if (nonfinite) atomicAdd(s.status + 1, 1u);
  }
}

// shared-memory floats per particle for a spec (host + device agree through this one function)
struct ColLayout {
  int x, act, rt, rr, rh, g, us, tsd, db, total;
};

// a full-covariance reference (lrds_gmm.layout) on the time-marginal path resp. as the terminal term
__host__ __device__ inline bool ref_t_full(const lrds_spec& s) { return s.has_ref_ctrl && s.ref_t.layout == LRDS_GMM_FULL; }
__host__ __device__ inline bool gmm_full_on_path(const lrds_spec& s) {
  return ref_t_full(s) || s.ref_0.layout == LRDS_GMM_FULL || (s.target.kind == LRDS_DISTR_GMM && s.target.gmm.layout == LRDS_GMM_FULL);
}

// mix_tc: the mixture-score contractions run on the tensor core (lrds_rollout_mix.cuh): responsibilities live in
// registers / TMEM, not in shared-memory columns
__host__ __device__ inline ColLayout col_layout(const lrds_spec& s, bool mix_tc = false) {
  ColLayout L{};
  int off = 0;
  const int dp = s.mlp.d_pad;
  L.x = off; off += dp;
  L.act = off;
  if (s.precision == LRDS_PRECISION_FP32_SIMT) off += C;  // hidden activations: tensor-core backends keep them in TMEM
  L.rt = off;
  const bool tfull = s.target.kind == LRDS_DISTR_GMM && s.target.gmm.layout == LRDS_GMM_FULL;  // lrds_distr_eval only
  if (!mix_tc && !tfull && s.target.kind == LRDS_DISTR_GMM && s.target.gmm.M > 1) off += (s.target.gmm.M + 3) / 4 * 4;
  L.rr = off;
  L.rh = off;
  if (ref_t_full(s) || tfull) {  // full-covariance reference: its score (rr) and the per-mode scratch h (rh), d_pad floats each
    L.rh = off + dp;
    off += 2 * dp;
    if (s.ref_0.layout != LRDS_GMM_FULL && s.ref_0.M > 1 && s.ref_0.M > 2 * dp) off += (s.ref_0.M + 3) / 4 * 4 - 2 * dp;
  } else if (!mix_tc) {
    int m = 0;
    if (s.has_ref_ctrl && s.ref_t.M > 1) m = s.ref_t.M;
    if (s.ref_0.layout != LRDS_GMM_FULL && s.ref_0.M > 1 && s.ref_0.M > m) m = s.ref_0.M;
    off += (m + 3) / 4 * 4;
  }
  L.g = off;
  if (s.target.kind == LRDS_DISTR_LOGREG) off += s.target.logreg.n_pad;
  L.us = off; L.tsd = off; L.db = off;
  if (s.kind == LRDS_ROLLOUT_CMCD || s.kind == LRDS_ROLLOUT_EUBO_CMCD) {
    L.us = off; off += dp;
    L.tsd = off; off += dp;
    L.db = off; off += dp;
  } else if (s.kind == LRDS_ROLLOUT_EUBO_LINEAR) {
    L.db = off; off += dp;
  }
  L.total = off;
  return L;
}

// x, rt, rr are float4-grouped columns (their layout offsets are multiples of 4); the rest are scalar columns
struct Particle {
  Col4 x, rt, rr, rh;
  Col g, us, tsd, db;
};

__device__ __forceinline__ Particle make_particle(float* smem, const ColLayout& L, int NT, int tid) {
  Particle P;
  P.x = Col4{smem + L.x * NT + 4 * tid, 4 * NT};
  P.rt = Col4{smem + L.rt * NT + 4 * tid, 4 * NT};
  P.rr = Col4{smem + L.rr * NT + 4 * tid, 4 * NT};
  P.rh = Col4{smem + L.rh * NT + 4 * tid, 4 * NT};
  P.g = Col{smem + L.g * NT + tid, NT};
  P.us = Col{smem + L.us * NT + tid, NT};
  P.tsd = Col{smem + L.tsd * NT + tid, NT};
  P.db = Col{smem + L.db * NT + tid, NT};
  return P;
}

// ---- per-step operand staging (LINEAR kind) ----------------------------------------------------------------
struct StageLayout {
  uint32_t tgt_logc_bytes, tgt_param_bytes, tgt_bytes;  // target mixture (static, M > 1): logc | sn
  uint32_t ref_logc_bytes, ref_param_bytes, row_bytes;  // one step: table row | logc | sn (M > 1)
  uint32_t tgt_mix_bytes, ref_mix_bytes;                // tensor-core images of the score contractions (mix_tc)
  uint32_t buf_bytes, off_tgt, off_buf, total;
};
// A block of lrds_gmm.mix_tc (include/lrds_b200.h):
//   [contraction image hi | lo][16 B: un-scale]  -  the score contraction (rows n = 16 c + i over 8-dim chunks)
//   [logit image hi | lo][c_m: Mp floats][16 B: un-scale, Wn, Cmax, shared]  -  the responsibilities' logits of a mixture
//   whose modes share their variances: logit_m = c_m + x . wc_m (+ a mode-independent term), wc_m = mu_m / var - mean_m
__host__ __device__ inline uint32_t gmm_mix_contr_bytes(int M, int d_pad) {
  return 2u * (uint32_t)((M + 15) / 16 * 2) * (uint32_t)(2 * d_pad) * 16u + 16u;
}
__host__ __device__ inline uint32_t gmm_mix_logit_part_bytes(int M, int d_pad) {  // one (hi | lo) part: Mp rows x Kin halves
  return (uint32_t)((M + 15) / 16 * 16) * (uint32_t)((d_pad + 15) / 16 * 16) * 2u;
}
__host__ __device__ inline uint32_t gmm_mix_tc_bytes(int M, int d_pad) {
  return gmm_mix_contr_bytes(M, d_pad) + 2u * gmm_mix_logit_part_bytes(M, d_pad) + (uint32_t)((M + 15) / 16 * 16) * 4u + 16u;
}

// level 1: table row + reference block per step; level 2: also the (static) target mixture
__host__ __device__ inline StageLayout stage_layout(const lrds_spec& s, int level, bool mix_tc = false) {
  StageLayout L{};
  const uint32_t dp = (uint32_t)s.mlp.d_pad;
  if (level >= 2 && s.target.kind == LRDS_DISTR_GMM && s.target.gmm.M > 1) {
    L.tgt_logc_bytes = (uint32_t)((s.target.gmm.M + 3) / 4 * 4) * 4u;
    L.tgt_param_bytes = (uint32_t)((s.target.gmm.M + 3) / 4) * dp * 32u;  // sn: 8 floats per mode (padded to 4) and dim
    if (mix_tc) L.tgt_mix_bytes = gmm_mix_tc_bytes(s.target.gmm.M, s.mlp.d_pad);
    L.tgt_bytes = L.tgt_logc_bytes + L.tgt_param_bytes + L.tgt_mix_bytes;
  }
  if (s.has_ref_ctrl && s.ref_t.M > 1 && !ref_t_full(s)) {  // single Gaussians (and full blocks) are read from global memory
    L.ref_logc_bytes = (uint32_t)((s.ref_t.M + 3) / 4 * 4) * 4u;
    L.ref_param_bytes = (uint32_t)((s.ref_t.M + 3) / 4) * dp * 32u;
    if (mix_tc) L.ref_mix_bytes = gmm_mix_tc_bytes(s.ref_t.M, s.mlp.d_pad);
  }
  L.row_bytes = LRDS_STEP_STRIDE * 4u;
  L.buf_bytes = L.row_bytes + L.ref_logc_bytes + L.ref_param_bytes + L.ref_mix_bytes;
  L.off_tgt = 16;  // two mbarriers in front
  L.off_buf = L.off_tgt + L.tgt_bytes;
  L.total = L.off_buf + 2u * L.buf_bytes;
  return L;
}

// issued by one thread; the caller has armed `bar` with the byte count
__device__ __forceinline__ void stage_gmm(uint8_t* dst, const GmmView& g, uint32_t logc_bytes, uint32_t param_bytes,
                                          uint64_t* bar) {
  ptx::bulk_g2s(dst, g.logc.p, logc_bytes, bar);
  ptx::bulk_g2s(dst + logc_bytes, g.sn.p, param_bytes, bar);
}
__device__ __forceinline__ void stage_step(uint8_t* dst, const lrds_spec& s, const StageLayout& L, int k, uint64_t* bar) {
  ptx::bulk_g2s(dst, s.steps + (int64_t)k * LRDS_STEP_STRIDE, L.row_bytes, bar);
  if (L.ref_param_bytes) stage_gmm(dst + L.row_bytes, gmm_at(s.ref_t, k), L.ref_logc_bytes, L.ref_param_bytes, bar);
}
// `g` = the same block in global memory (its single-Gaussian members stay valid in the staged view)
__device__ __forceinline__ GmmViewT<true> staged_view(const uint8_t* src, const GmmView& g, uint32_t logc_bytes,
                                                     uint32_t param_bytes) {
  GmmViewT<true> v;
  const uint32_t a = ptx::smem_u32(src);
  v.M = g.M;
  v.logc = PPtr<true>{a};
  v.sn = PPtr<true>{a + logc_bytes};
  v.glogc = g.glogc;
  v.mu = g.mu;
  v.ivar = g.ivar;
  return v;
}

// ---- compile-time specialisation of the LINEAR loop ----------------------------------------------------------
// The loop is driven by warp-uniform switches of the spec (update / Ito form, control kind, target kind, reference).
// Evaluated at run time they cost a branch sequence per 8-dim chunk each (~20% of the warp time in the ncu source
// view); a Traits type fixes them at compile time for the configurations the solvers actually build (-1 = run time).
template <int UPDATE = -1, int ITO = -1, int TARGET = -1, int SCORE = -1, int REF = -1, int MIX = 0>
struct LinearTraits {
  static constexpr bool kMix = MIX != 0;  // every mixture block on the path (target if GMM, reference) has M > 1
  static constexpr int kUpdate = UPDATE;  // lrds_update_form
  static constexpr int kIto = ITO;        // lrds_ito_form
  static constexpr int kTarget = TARGET;  // lrds_distr_kind
  static constexpr int kScore = SCORE;    // 1 = ScoreCtrl, 0 = ClippedCtrl
  static constexpr int kRef = REF;        // 0 = no reference control, 1 = Gaussian (M == 1), 2 = mixture (M > 1), 3 = full (ref_class)
};
using RuntimeTraits = LinearTraits<>;
// 3 = full-covariance reference (any M): only the run-time-switched kernels serve it
__host__ __device__ inline int ref_class(const lrds_spec& s) {
  return !s.has_ref_ctrl ? 0 : (ref_t_full(s) ? 3 : (s.ref_t.M > 1 ? 2 : 1));
}
template <class TR>
__host__ __device__ inline bool traits_match(const lrds_spec& s) {
  return (TR::kUpdate < 0 || TR::kUpdate == s.update_form) && (TR::kIto < 0 || TR::kIto == s.ito_form) &&
         (TR::kTarget < 0 || TR::kTarget == s.target.kind) &&
         (TR::kScore < 0 || (s.ctrl_kind <= LRDS_CTRL_SCORE && TR::kScore == (s.ctrl_kind == LRDS_CTRL_SCORE))) &&
         (TR::kRef < 0 || TR::kRef == ref_class(s)) && (TR::kRef < 0 || !gmm_full_on_path(s)) &&
         (!TR::kMix || ((s.target.kind != LRDS_DISTR_GMM || s.target.gmm.M > 1) && (!s.has_ref_ctrl || s.ref_t.M > 1)));
}

// fp32 FFMA drift network: hidden activations in 64 shared-memory columns per particle
struct SimtMlp {
  static constexpr bool kPipe = true;  // 128-thread CTAs: registers to spare for operand prefetch
  const lrds_mlp& w;
  Col act;
  template <bool BIAS_SH>
  __device__ __forceinline__ void hidden(const float* __restrict__ bias1, const Col4& x) {
    mlp_hidden<BIAS_SH>(w, bias1, x, act);
  }
  __device__ __forceinline__ void out_chunk(int j0, float (&out)[JC]) { mlp_out_chunk(w, act, j0, out); }
  __device__ __forceinline__ bool saturated() const { return false; }  // fp32 FFMA: no operand conversion
};

// ---- target helpers ---------------------------------------------------------------------------------
template <bool PIPE, bool MIX = false, bool SH>
__device__ __forceinline__ float target_pass1(const lrds_spec& s, int kind, const GmmViewT<SH>& tv, const Particle& P,
                                              bool want_logp) {
  const lrds_distr& t = s.target;
  if (kind == LRDS_DISTR_GMM) return gmm_pass1<PIPE, MIX>(tv, s.d, s.mlp.d_pad, P.x, P.rt);
  if (kind == LRDS_DISTR_LOGREG) return logreg_pass1(t.logreg, s.d, P.x, P.g, want_logp);
  if (kind == LRDS_DISTR_PHI4) return want_logp ? phi4_logp(t.phi4, s.d, P.x) : 0.f;
  return 0.f;
}

// raw target score for dims [j0, j0+JC); xm / xp are x_{j0-1} / x_{j0+JC} of the SAME state as xr
template <bool PIPE, bool MIX = false, bool SH>
__device__ __forceinline__ void target_score_chunk(const lrds_spec& s, int kind, const GmmViewT<SH>& tv, const Particle& P,
                                                   const float (&xr)[JC], float xm, float xp, int j0, float (&out)[JC]) {
  const lrds_distr& t = s.target;
  if (kind == LRDS_DISTR_GMM) {
    gmm_score_chunk<PIPE, MIX>(tv, s.d, s.mlp.d_pad, xr, P.rt, j0, out);
  } else if (kind == LRDS_DISTR_LOGREG) {
    logreg_score_chunk(t.logreg, s.d, s.mlp.d_pad, xr, P.g, j0, out);
  } else if (kind == LRDS_DISTR_PHI4) {
    const float coef = t.phi4.a * (float)s.d;
#pragma unroll
    for (int c = 0; c < JC; ++c) {
      const float left = (c == 0) ? xm : xr[c - 1];
      const float right = (c == JC - 1) ? xp : xr[c + 1];
      const int j = j0 + c;
      // Dirichlet-0: the neighbour beyond the last site is 0; xr is zero padded beyond d
      out[c] = (j < s.d) ? phi4_score_1(t.phi4, coef, left, xr[c], (j == s.d - 1) ? 0.f : right) : 0.f;
    }
  } else {
#pragma unroll
    for (int c = 0; c < JC; ++c) out[c] = 0.f;
  }
}

__device__ __forceinline__ void load_chunk(const Col& v, int j0, float (&out)[JC]) {
#pragma unroll
  for (int c = 0; c < JC; ++c) out[c] = v(j0 + c);
}
__device__ __forceinline__ void load_chunk(const Col4& v, int j0, float (&out)[JC]) {
  const float4 a = v.ld4(j0 >> 2), b = v.ld4((j0 >> 2) + 1);
  out[0] = a.x; out[1] = a.y; out[2] = a.z; out[3] = a.w; out[4] = b.x; out[5] = b.y; out[6] = b.z; out[7] = b.w;
}
__device__ __forceinline__ void store_chunk(const Col4& v, int j0, const float (&in)[JC]) {
  v.st4(j0 >> 2, make_float4(in[0], in[1], in[2], in[3]));
  v.st4((j0 >> 2) + 1, make_float4(in[4], in[5], in[6], in[7]));
}

// target score at P.x, chunk by chunk: consume(j0, xr, ts) gets dims [j0, j0 + JC) of x and of the score
template <bool PIPE, bool SH, class F>
__device__ __forceinline__ void target_score_loop(const lrds_spec& s, int kind, const GmmViewT<SH>& tv, const Particle& P,
                                                  F&& consume) {
  const int dp = s.mlp.d_pad;
  float xm = 0.f;
  for (int j0 = 0; j0 < dp; j0 += JC) {
    float xr[JC], ts[JC];
    load_chunk(P.x, j0, xr);
    const float xp = (j0 + JC < dp) ? P.x(j0 + JC) : 0.f;
    target_score_chunk<PIPE>(s, kind, tv, P, xr, xm, xp, j0, ts);
    xm = xr[JC - 1];
    consume(j0, xr, ts);
  }
}

// one thread per particle (the column-layout kernels of lrds_capi.cu): b is the thread's particle, clamped to the last
// one in the idle threads of the last CTA, whose results are not written (live = false)
struct ParticleThread {
  int b;
  bool live;
  Particle P;
};
__device__ __forceinline__ ParticleThread particle_thread(const lrds_spec& s, float* smem) {
  const int NT = blockDim.x, tid = threadIdx.x;
  const int b_raw = blockIdx.x * NT + tid;
  const bool live = b_raw < s.B;
  return ParticleThread{live ? b_raw : s.B - 1, live, make_particle(smem, col_layout(s), NT, tid)};
}

constexpr int MIX_MAX_M = 16;  // components of a mixture whose responsibilities live in registers (gmm_pass1_pair)

// Responsibilities r = softmax_m(logc_m - q_m / 2) of a mixture with M <= 16 components in registers (the arithmetic
// of gmm_pass1, lrds_device.cuh); returns the mixture log-density; modes beyond M get weight zero.  The quadratic forms
// are bound by the shared-memory pipe, not by the FMA pipe: every (1/sigma, -mu/sigma) pair is used once per particle and a warp-uniform LDS.128
// (one wavefront) feeds only two FFMA2.  Here the two half-warps split the mode blocks, and every thread evaluates
// its modes for TWO particles - its own and the one of lane ^ 16 - so that each operand vector feeds four FFMA2;
// the dims are the outer loop, so that a particle's coordinates are read once per call instead of once per mode
// block.  The halves swap their partner results with one SHFL per mode.
template <bool SH>
__device__ __forceinline__ float gmm_pass1_pair(const GmmViewT<SH>& g, int d, int dp, const Col4& x, float (&r)[MIX_MAX_M]) {
  const int lane = threadIdx.x & 31, h = lane >> 4;
  const int nq = (d + 3) >> 2;
  const int rowq = dp >> 2;
  const int M4 = (g.M + 3) >> 2;
  const int nb = (M4 + 1) >> 1;  // mode blocks per half-warp (warp-uniform): 1 or 2
  const int b0 = h * nb;
  const Col4 xo{x.p + ((lane ^ 16) - lane) * 4, x.stride};  // the partner's coordinates
  const int blk0 = min(b0, M4 - 1), blk1 = min(b0 + 1, M4 - 1);  // clamped: results of blocks >= M4 are discarded
  PPtr<SH> p0 = g.sn + blk0 * rowq * 32, p1 = g.sn + blk1 * rowq * 32;
  u64 qa[8] = {0, 0, 0, 0, 0, 0, 0, 0}, qb[8] = {0, 0, 0, 0, 0, 0, 0, 0};  // own / partner particle, (even, odd) dims
  auto block = [&](const PPtr<SH>& p, const ulonglong2& xa, const ulonglong2& xb, int o) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const ulonglong2 sv = p.ld2(2 * i), nv = p.ld2(2 * i + 1);
      const u64 a0 = f2::fma(xa.x, sv.x, nv.x), a1 = f2::fma(xa.y, sv.y, nv.y);
      const u64 c0 = f2::fma(xb.x, sv.x, nv.x), c1 = f2::fma(xb.y, sv.y, nv.y);
      qa[o + i] = f2::fma(a0, a0, qa[o + i]);
      qb[o + i] = f2::fma(c0, c0, qb[o + i]);
      qa[o + i] = f2::fma(a1, a1, qa[o + i]);
      qb[o + i] = f2::fma(c1, c1, qb[o + i]);
    }
  };
  if (nb > 1) {
    for (int c = 0; c < nq; ++c, p0 = p0 + 32, p1 = p1 + 32) {
      const ulonglong2 xa = x.ldu(c), xb = xo.ldu(c);
      block(p0, xa, xb, 0);
      block(p1, xa, xb, 4);
    }
  } else {
    for (int c = 0; c < nq; ++c, p0 = p0 + 32) {
      const ulonglong2 xa = x.ldu(c), xb = xo.ldu(c);
      block(p0, xa, xb, 0);
    }
  }
  float own[8], oth[8];
  {
    const float4 l0 = g.logc.ld4(blk0), l1 = g.logc.ld4(blk1);
    const float lc[8] = {l0.x, l0.y, l0.z, l0.w, l1.x, l1.y, l1.z, l1.w};
    const bool v0 = b0 < M4, v1 = nb > 1 && b0 + 1 < M4;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const bool v = k < 4 ? v0 : v1;
      float ax, ay, bx, by;
      f2::unpack(qa[k], ax, ay);
      f2::unpack(qb[k], bx, by);
      own[k] = v ? lc[k] - 0.5f * (ax + ay) : -INFINITY;
      oth[k] = v ? lc[k] - 0.5f * (bx + by) : -INFINITY;
    }
  }
#pragma unroll
  for (int k = 0; k < 8; ++k) oth[k] = __shfl_xor_sync(0xffffffffu, oth[k], 16);  // my particle, the other half's modes
  if (nb > 1) {
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      r[k] = h ? oth[k] : own[k];
      r[8 + k] = h ? own[k] : oth[k];
    }
  } else {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      r[k] = h ? oth[k] : own[k];
      r[4 + k] = h ? own[k] : oth[k];
    }
#pragma unroll
    for (int k = 8; k < MIX_MAX_M; ++k) r[k] = -INFINITY;
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
  return mx + __logf(s);
}

// control u = generative_ctrl(tau, x) for dims [j0, j0+JC) after mlp.hidden(), given the raw target score chunk
// `ts` (ScoreCtrl) and gamma = clip(score_model(tau)).   models/reparam.py:33-43, 112-117
struct CtrlConst {
  float bound_model, bound_score, scale_score;
  bool score;  // the control has a target-score term (every kind but ClippedCtrl)
  int d;
  int kind;    // lrds_ctrl_kind
};
__device__ __forceinline__ CtrlConst ctrl_const(const lrds_spec& s) {
  return CtrlConst{clip_bound(s.clip_model), clip_bound(s.clip_score), s.scale_score, s.ctrl_kind != LRDS_CTRL_CLIPPED, s.d,
                   s.ctrl_kind};
}
template <class MLP>
__device__ __forceinline__ void ctrl_chunk(const CtrlConst& cc, MLP& mlp, int j0, const float (&ts)[JC], float gamma,
                                           float (&u)[JC]) {
  mlp.out_chunk(j0, u);
#pragma unroll
  for (int c = 0; c < JC; ++c) {
    float v = clipb(u[c], cc.bound_model);
    if (cc.score) v = v + (cc.scale_score * clipb(ts[c], cc.bound_score)) * gamma;
    u[c] = (j0 + c < cc.d) ? v : 0.f;
  }
}

// The DIS parametrisations CancelDriftCtrl / LerpCtrl (models/reparam.py:131-147, 189-199): time-only coefficients of
// the table row, the state chunk `xr` and (LerpCtrl) the prior-score chunk `ps`.
struct CtrlStep {
  float gamma, cx, gscale, w;
};
__device__ __forceinline__ CtrlStep ctrl_step(const float* __restrict__ row) {
  return CtrlStep{__ldg(row + LRDS_STEP_GAMMA), __ldg(row + LRDS_STEP_CX), __ldg(row + LRDS_STEP_GSCALE), __ldg(row + LRDS_STEP_LERP)};
}
__device__ __forceinline__ float lerpf(float a, float b, float w) {  // torch.lerp's two-sided formula
  return w < 0.5f ? a + w * (b - a) : b - (b - a) * (1.0f - w);
}
template <class MLP>
__device__ __forceinline__ void ctrl_chunk_dis(const CtrlConst& cc, MLP& mlp, int j0, const float (&ts)[JC],
                                               const float (&xr)[JC], const float (&ps)[JC], const CtrlStep& st, float (&u)[JC]) {
  mlp.out_chunk(j0, u);
#pragma unroll
  for (int c = 0; c < JC; ++c) {
    float v = clipb(u[c], cc.bound_model);
    const float sc = cc.kind == LRDS_CTRL_LERP ? lerpf(ps[c], ts[c], st.w) : ts[c];
    const float t = (cc.scale_score * clipb(sc, cc.bound_score)) * st.gamma;
    if (cc.kind == LRDS_CTRL_CANCEL_DRIFT) v = v + st.cx * xr[c];
    v = v + st.gscale * t;
    u[c] = (j0 + c < cc.d) ? v : 0.f;
  }
}

__device__ __forceinline__ void noise_chunk(const RolloutArgs& a, int step, int b, int j0, float (&z)[JC]) {
  if (a.noise != nullptr) {
    const float* p = a.noise + ((int64_t)step * a.s.B + b) * a.s.d + j0;
#pragma unroll
    for (int c = 0; c < JC; ++c) z[c] = (j0 + c < a.s.d) ? __ldg(p + c) : 0.f;
  } else {
    float z4[4];
    const uint32_t pidx = (uint32_t)(a.particle_offset + (uint64_t)b);
    normals4(a.seed, pidx, (uint32_t)step, (uint32_t)(j0 >> 2), 0u, z4);
    z[0] = z4[0]; z[1] = z4[1]; z[2] = z4[2]; z[3] = z4[3];
    normals4(a.seed, pidx, (uint32_t)step, (uint32_t)(j0 >> 2) + 1u, 0u, z4);
    z[4] = z4[0]; z[5] = z4[1]; z[6] = z4[2]; z[7] = z4[3];
    if (j0 + JC > a.s.d) {  // only the last chunk holds padded dims
#pragma unroll
      for (int c = 0; c < JC; ++c)
        if (j0 + c >= a.s.d) z[c] = 0.f;
    }
  }
}

__device__ __forceinline__ void store_traj(const RolloutArgs& a, int row, int b, int j0, const float (&v)[JC]) {
  float* p = a.traj_out + ((int64_t)row * a.s.B + b) * a.s.d + j0;
#pragma unroll
  for (int c = 0; c < JC; ++c)
    if (j0 + c < a.s.d) p[c] = v[c];
}

// ControlledLangevinSDE.drift (eq/sdes.py:101-110) for one coordinate
__device__ __forceinline__ float langevin_drift(const lrds_spec& s, float ts, float ps, float frac) {
  float dr = ts * frac + ps * (1.0f - frac);
  dr *= 0.5f * s.cmcd_diff * s.cmcd_diff;
  return clipf(dr, s.cmcd_clip);
}

// reference_log_prob(x) of the terminal term: ref_0 in either layout (full: h is not stored, the score column untouched)
template <bool PIPE>
__device__ __forceinline__ float ref0_log_prob(const lrds_spec& s, const Particle& P) {
  if (s.ref_0.layout == LRDS_GMM_FULL) return gmm_full_pass<false>(gmm_full_at(s.ref_0, 0), s.d, s.mlp.d_pad, P.x, P.rr, P.rh);
  return gmm_pass1<PIPE>(gmm_at(s.ref_0, 0), s.d, s.mlp.d_pad, P.x, P.rr);
}

// `smem` = this CTA's column area (col_layout(s).total * blockDim.x floats); every thread of the CTA runs the body
// with uniform control flow (idle lanes shadow the last particle), which the tensor-core policy relies on.
// STAGE > 0 (LINEAR kind): `stage` is a stage_layout(s, STAGE).total-byte shared-memory area; the time-marginal
// reference block + table row of step k+1 are prefetched by the TMA engine (cp.async.bulk + mbarrier, double
// buffered) while step k computes, and with STAGE == 2 the target mixture is copied there once as well.
// One CTA barrier per step keeps the buffers safe.
template <int KIND, int STAGE, class TR = RuntimeTraits, class MLP>
__device__ __forceinline__ void rollout_body(const RolloutArgs& a, float* smem, uint8_t* stage, MLP& mlp) {
  constexpr bool PIPE = MLP::kPipe;
  const lrds_spec& s = a.s;
  const int NT = blockDim.x;
  const int tid = threadIdx.x;
  const int b_raw = blockIdx.x * NT + tid;
  const bool live = b_raw < s.B;
  const int b = live ? b_raw : s.B - 1;  // idle lanes shadow the last particle, results are not stored
  const int d = s.d, dp = s.mlp.d_pad, K = s.K;
  const ColLayout L = col_layout(s);
  const Particle P = make_particle(smem, L, NT, tid);

  for (int j = 0; j < dp; ++j) P.x(j) = (j < d) ? __ldg(a.x0 + (int64_t)b * d + j) : 0.f;
  if (a.traj_out != nullptr && live)
    for (int j = 0; j < d; ++j) a.traj_out[(int64_t)b * d + j] = P.x(j);

  const int tkind = TR::kTarget >= 0 ? TR::kTarget : s.target.kind;
  const bool score_ctrl = TR::kScore >= 0 ? TR::kScore != 0 : s.ctrl_kind != LRDS_CTRL_CLIPPED;
  const bool dis_ctrl = TR::kScore < 0 && s.ctrl_kind >= LRDS_CTRL_CANCEL_DRIFT;  // CancelDriftCtrl / LerpCtrl
  const bool has_ref = TR::kRef >= 0 ? TR::kRef != 0 : s.has_ref_ctrl != 0;
  const int update_form = TR::kUpdate >= 0 ? TR::kUpdate : s.update_form;
  const int ito_form = TR::kIto >= 0 ? TR::kIto : s.ito_form;
  const bool need_nbr = tkind == LRDS_DISTR_PHI4;  // lattice stencil reads x_{j0-1}, x_{j0+8}
  const bool rfull = TR::kRef < 0 && has_ref && s.ref_t.layout == LRDS_GMM_FULL;  // full reference: score column P.rr
  CtrlConst cc = ctrl_const(s);
  cc.score = score_ctrl;
  const GmmView tv0 = gmm_at(s.target.gmm, 0);  // target mixture in global memory (dereferenced for GMM targets only)
  float rnd = 0.f;

  if constexpr (KIND == LRDS_ROLLOUT_LINEAR) {
    constexpr bool STAGED = STAGE > 0;
    constexpr bool SH = STAGED, TSH = STAGE > 1;
    const StageLayout SL = stage_layout(s, STAGE);
    uint64_t* sbar = reinterpret_cast<uint64_t*>(stage);
    GmmViewT<TSH> tv{};
    if constexpr (!TSH) tv = tv0;
    if constexpr (STAGED) {
      if (tid == 0) {
        ptx::mbar_init(sbar, 1);
        ptx::mbar_init(sbar + 1, 1);
        ptx::fence_mbar_init();
      }
      __syncthreads();
      if (tid == 0) {
        ptx::mbar_expect_tx(sbar, SL.tgt_bytes + SL.buf_bytes);
        if (SL.tgt_bytes) stage_gmm(stage + SL.off_tgt, tv0, SL.tgt_logc_bytes, SL.tgt_param_bytes, sbar);
        stage_step(stage + SL.off_buf, s, SL, 0, sbar);
      }
      if constexpr (TSH) tv = staged_view(stage + SL.off_tgt, tv0, SL.tgt_logc_bytes, SL.tgt_param_bytes);
    }
    for (int k = 0; k < K; ++k) {
      const float* row = s.steps + (int64_t)k * LRDS_STEP_STRIDE;
      GmmViewT<SH> rv{};
      PPtr<SH> rowp{};
      if constexpr (STAGED) {
        __syncthreads();  // every warp has finished step k-1, whose buffer the prefetch below overwrites
        if (tid == 0 && k + 1 < K) {
          ptx::mbar_expect_tx(sbar + ((k + 1) & 1), SL.buf_bytes);
          stage_step(stage + SL.off_buf + ((k + 1) & 1) * SL.buf_bytes, s, SL, k + 1, sbar + ((k + 1) & 1));
        }
        ptx::mbar_wait(sbar + (k & 1), (uint32_t)(k >> 1) & 1u);
        const uint8_t* buf = stage + SL.off_buf + (k & 1) * SL.buf_bytes;
        row = reinterpret_cast<const float*>(buf);
        rowp = PPtr<true>{ptx::smem_u32(buf)};
        if (has_ref && !rfull) rv = staged_view(buf + SL.row_bytes, gmm_at(s.ref_t, k), SL.ref_logc_bytes, SL.ref_param_bytes);
      } else {
        rowp = PPtr<false>{row};
        if (has_ref && !rfull) rv = gmm_at(s.ref_t, k);
      }
      const float A = rowp.ld1(LRDS_STEP_A), Bc = rowp.ld1(LRDS_STEP_B), Cc = rowp.ld1(LRDS_STEP_C);
      const float dt = rowp.ld1(LRDS_STEP_DT), sqdt = rowp.ld1(LRDS_STEP_SQRT_DT);
      const float wcost = rowp.ld1(LRDS_STEP_W_COST), wito = rowp.ld1(LRDS_STEP_W_ITO);
      const float gamma = rowp.ld1(LRDS_STEP_GAMMA), sigu = rowp.ld1(LRDS_STEP_SIGU);
      if (score_ctrl) target_pass1<PIPE, TR::kMix>(s, tkind, tv, P, false);
      if (rfull) gmm_full_pass<true>(gmm_full_at(s.ref_t, k), d, dp, P.x, P.rr, P.rh);
      else if (has_ref && (TR::kRef == 2 || rv.M > 1)) gmm_pass1<PIPE, TR::kMix>(rv, d, dp, P.x, P.rr);
      mlp.template hidden<SH>(row + LRDS_STEP_BIAS1, P.x);
      float su2 = 0.f, sito = 0.f, xm = 0.f;
      for (int j0 = 0; j0 < dp; j0 += JC) {
        float xr[JC], ts[JC], u[JC], rs[JC], z[JC], xn[JC];
        load_chunk(P.x, j0, xr);
        const float xp = (need_nbr && j0 + JC < dp) ? P.x(j0 + JC) : 0.f;
        if (score_ctrl) target_score_chunk<PIPE, TR::kMix>(s, tkind, tv, P, xr, xm, xp, j0, ts);
        if (dis_ctrl) {
          float ps[JC] = {};
          if (cc.kind == LRDS_CTRL_LERP) gmm_score_chunk<false, false>(gmm_at(s.ref_0, 0), d, dp, xr, P.rr, j0, ps);
          ctrl_chunk_dis(cc, mlp, j0, ts, xr, ps, ctrl_step(s.steps + (int64_t)k * LRDS_STEP_STRIDE), u);
        } else {
          ctrl_chunk(cc, mlp, j0, ts, gamma, u);
        }
        if (rfull) load_chunk(P.rr, j0, rs);
        else if (has_ref) gmm_score_chunk<PIPE, TR::kMix>(rv, d, dp, xr, P.rr, j0, rs);
        noise_chunk(a, k, b, j0, z);
#pragma unroll
        for (int c = 0; c < JC; ++c) {
          const float r = has_ref ? rs[c] : 0.f;
          su2 = fmaf(u[c], u[c], su2);
          if (update_form == LRDS_UPDATE_AXPY) {
            xn[c] = (A * xr[c] + Bc * (r + u[c])) + Cc * z[c];
          } else {  // EM: A = f(tau), Bc = sigma, Cc = sigma^2
            float drift = -(A * xr[c]);
            if (has_ref) drift += Cc * r;
            xn[c] = xr[c] + (drift + Bc * u[c]) * dt + Bc * (z[c] * sqdt);
          }
          if (ito_form == LRDS_ITO_SCALED) sito = fmaf(u[c], z[c], sito);
          else if (ito_form == LRDS_ITO_EM) sito = fmaf(u[c], z[c] * sqdt, sito);
          else if (ito_form == LRDS_ITO_DDS) sito += ((sigu * u[c]) * z[c]) * wito;
          if (j0 + c >= d) xn[c] = 0.f;
        }
        xm = xr[JC - 1];
        store_chunk(P.x, j0, xn);
        if (a.traj_out != nullptr && live) store_traj(a, k + 1, b, j0, xn);
      }
      rnd += wcost * su2;
      if (ito_form == LRDS_ITO_SCALED) rnd += wito * sito;
      else if (ito_form != LRDS_ITO_NONE) rnd += sito;
    }
    // terminal cost: rnd += reference_log_prob(x) - terminal_unnorm_log_prob(x)   (oc.py:290, 505, 645, 1389);
    // init_cost (DIS): the initial cost initial_log_prob(x_0) + rnd_offset, written to rnd_out by lrds_rollout's pre-pass,
    // takes the place of the reference term (oc.py:1164-1168, 1230)
    const float lref = s.init_cost ? a.rnd_out[b] : ref0_log_prob<PIPE>(s, P);
    const float ltgt = clipf(target_pass1<PIPE>(s, tkind, tv, P, true), s.clip_target);
    rnd += lref - ltgt;
  }

  if constexpr (KIND == LRDS_ROLLOUT_EUBO_LINEAR) {
    {  // rnd = reference_log_prob(x) - terminal_unnorm_log_prob(x)   (oc.py:321, 536); init_cost (the discrete-time
       // DIS loss, oc.py:1000-1033): ref_0 is the prior and enters at the END of the noising rollout instead
      const float lref = s.init_cost ? 0.f : ref0_log_prob<PIPE>(s, P);
      const float ltgt = clipf(target_pass1<PIPE>(s, tkind, tv0, P, true), s.clip_target);
      rnd = lref - ltgt;
    }
    for (int k = 0; k < K; ++k) {  // rows are stored in loop order (reversed time)
      const float* row = s.steps + (int64_t)k * LRDS_STEP_STRIDE;
      const float mean = __ldg(row + LRDS_STEP_EU_A), stdf = __ldg(row + LRDS_STEP_EU_B);
      const float wx = __ldg(row + LRDS_STEP_EU_C), sig = __ldg(row + LRDS_STEP_B);
      const float wcost = __ldg(row + LRDS_STEP_W_COST), wito = __ldg(row + LRDS_STEP_W_ITO);
      const float gamma = __ldg(row + LRDS_STEP_GAMMA);
      for (int j0 = 0; j0 < dp; j0 += JC) {  // x <- mean x + std z   (oc.py:335-337, 550-552)
        float z[JC];
        noise_chunk(a, k, b, j0, z);
#pragma unroll
        for (int c = 0; c < JC; ++c) {
          P.db(j0 + c) = z[c];
          P.x(j0 + c) = (j0 + c < d) ? fmaf(stdf, z[c], P.x(j0 + c) * mean) : 0.f;
        }
      }
      if (score_ctrl) target_pass1<PIPE>(s, tkind, tv0, P, false);
      GmmView rv{};
      if (rfull) {
        gmm_full_pass<true>(gmm_full_at(s.ref_t, k), d, dp, P.x, P.rr, P.rh);
      } else if (has_ref) {
        rv = gmm_at(s.ref_t, k);
        if (rv.M > 1) gmm_pass1<PIPE>(rv, d, dp, P.x, P.rr);
      }
      mlp.template hidden<false>(row + LRDS_STEP_BIAS1, P.x);
      float cost = 0.f, gx = 0.f, gz = 0.f, xm = 0.f;
      for (int j0 = 0; j0 < dp; j0 += JC) {
        float xr[JC], ts[JC], u[JC], rs[JC];
        load_chunk(P.x, j0, xr);
        const float xp = (need_nbr && j0 + JC < dp) ? P.x(j0 + JC) : 0.f;
        if (score_ctrl) target_score_chunk<PIPE>(s, tkind, tv0, P, xr, xm, xp, j0, ts);
        ctrl_chunk(cc, mlp, j0, ts, gamma, u);
        if (rfull) {
          load_chunk(P.rr, j0, rs);
        } else if (has_ref) {
          gmm_score_chunk<PIPE>(rv, d, dp, xr, P.rr, j0, rs);
        } else {
#pragma unroll
          for (int c = 0; c < JC; ++c) rs[c] = 0.f;
        }
#pragma unroll
        for (int c = 0; c < JC; ++c) {
          const float g = (s.update_form == LRDS_UPDATE_EM) ? u[c] / sig : u[c];
          cost = fmaf(g, rs[c] + 0.5f * g, cost);
          gx = fmaf(g, xr[c], gx);
          gz = fmaf(g, P.db(j0 + c), gz);
        }
        xm = xr[JC - 1];
      }
      rnd -= cost * wcost;
      if (s.update_form == LRDS_UPDATE_EM) rnd += gx * wx;
      rnd -= gz * wito;
    }
    if (s.init_cost) rnd += gmm_pass1<PIPE>(gmm_at(s.ref_0, 0), d, dp, P.x, P.rr);  // + initial_log_prob(x), oc.py:1033
  }

  if constexpr (KIND == LRDS_ROLLOUT_CMCD || KIND == LRDS_ROLLOUT_EUBO_CMCD) {
    constexpr bool EUBO = (KIND == LRDS_ROLLOUT_EUBO_CMCD);
    const GmmView prior = gmm_at(s.ref_0, 0);
    const float sg = s.cmcd_diff;
    // control and raw target score at the starting point (row 0 forward, row K for the noising direction)
    auto eval_point = [&](int rowi, bool first, float dtk, float frac_for_drift, float& c2, float& cdb) {
      const float* row = s.steps + (int64_t)rowi * LRDS_STEP_STRIDE;
      const float gamma = __ldg(row + LRDS_STEP_GAMMA);
      target_pass1<PIPE>(s, tkind, tv0, P, false);
      mlp.template hidden<false>(row + LRDS_STEP_BIAS1, P.x);
      float xm = 0.f;
      for (int j0 = 0; j0 < dp; j0 += JC) {
        float xr[JC], ts[JC], u[JC];
        load_chunk(P.x, j0, xr);
        const float xp = (need_nbr && j0 + JC < dp) ? P.x(j0 + JC) : 0.f;
        target_score_chunk<PIPE>(s, tkind, tv0, P, xr, xm, xp, j0, ts);
        ctrl_chunk(cc, mlp, j0, ts, gamma, u);
#pragma unroll
        for (int c = 0; c < JC; ++c) {
          const int j = j0 + c;
          if (!first && j < d) {
            const float ps = -((xr[c] - prior.mu.ld1(j)) * prior.ivar.ld1(j));
            const float dnew = langevin_drift(s, ts[c], ps, frac_for_drift);
            // forward: cost = (drift_s + drift_t)/sig + u_s - u_t ; noising: (drift_s + drift_t)/sig + u_s - u_t
            // with (u_s, drift_s) the NEW point there (oc.py:737, 816)
            const float cst = EUBO ? ((dnew + P.tsd(j)) / sg + u[c] - P.us(j))
                                   : ((P.tsd(j) + dnew) / sg + P.us(j) - u[c]);
            c2 = fmaf(cst, cst, c2);
            cdb = fmaf(cst, P.db(j), cdb);
          }
          P.us(j) = u[c];
          P.tsd(j) = (j < d) ? ts[c] : 0.f;
        }
        xm = xr[JC - 1];
      }
      (void)dtk;
    };
    float c2 = 0.f, cdb = 0.f;
    if constexpr (!EUBO) {
      rnd = gmm_pass1<PIPE>(prior, d, dp, P.x, P.rr);  // initial_log_prob(x), oc.py:698
      eval_point(0, true, 0.f, 0.f, c2, cdb);
      for (int k = 0; k < K; ++k) {
        const float* row = s.steps + (int64_t)k * LRDS_STEP_STRIDE;
        const float dt = __ldg(row + LRDS_STEP_DT), sqdt = __ldg(row + LRDS_STEP_SQRT_DT);
        const float fs = __ldg(row + LRDS_STEP_FRAC), ft = __ldg(row + LRDS_STEP_STRIDE + LRDS_STEP_FRAC);
        for (int j0 = 0; j0 < dp; j0 += JC) {  // y = x + (drift_s + u_s sig) dt + sig db   (oc.py:722-724)
          float z[JC], xn[JC];
          noise_chunk(a, k, b, j0, z);
#pragma unroll
          for (int c = 0; c < JC; ++c) {
            const int j = j0 + c;
            float y = 0.f;
            if (j < d) {
              const float xj = P.x(j);
              const float ps = -((xj - prior.mu.ld1(j)) * prior.ivar.ld1(j));
              const float ds = langevin_drift(s, P.tsd(j), ps, fs);
              const float db = sqdt * z[c];
              y = xj + (ds + P.us(j) * sg) * dt + sg * db;
              P.tsd(j) = ds;
              P.db(j) = db;
            }
            xn[c] = y;
            P.x(j) = y;
          }
          if (a.traj_out != nullptr && live) store_traj(a, k + 1, b, j0, xn);
        }
        c2 = 0.f; cdb = 0.f;
        eval_point(k + 1, false, dt, ft, c2, cdb);
        rnd += 0.5f * c2 * dt;
        rnd += cdb;
      }
      rnd -= clipf(target_pass1<PIPE>(s, tkind, tv0, P, true), s.clip_target);  // oc.py:750
    } else {
      rnd = -clipf(target_pass1<PIPE>(s, tkind, tv0, P, true), s.clip_target);  // oc.py:782
      eval_point(K, true, 0.f, 0.f, c2, cdb);
      for (int i = 0; i < K; ++i) {
        const int kt = K - i, ks = K - 1 - i;  // t = ts[kt], s = ts[ks]
        const float* rows = s.steps + (int64_t)ks * LRDS_STEP_STRIDE;
        const float dt = __ldg(rows + LRDS_STEP_DT), sqdt = __ldg(rows + LRDS_STEP_SQRT_DT);
        const float ft = __ldg(s.steps + (int64_t)kt * LRDS_STEP_STRIDE + LRDS_STEP_FRAC);
        for (int j0 = 0; j0 < dp; j0 += JC) {  // y = x + (drift_t - u_t sig) dt + sig db   (oc.py:802-804)
          float z[JC];
          noise_chunk(a, i, b, j0, z);
#pragma unroll
          for (int c = 0; c < JC; ++c) {
            const int j = j0 + c;
            float y = 0.f;
            if (j < d) {
              const float xj = P.x(j);
              const float ps = -((xj - prior.mu.ld1(j)) * prior.ivar.ld1(j));
              const float dtt = langevin_drift(s, P.tsd(j), ps, ft);
              const float db = sqdt * z[c];
              y = xj + (dtt - P.us(j) * sg) * dt + sg * db;
              P.tsd(j) = dtt;
              P.db(j) = db;
            }
            P.x(j) = y;
          }
        }
        c2 = 0.f; cdb = 0.f;
        eval_point(ks, false, dt, ft, c2, cdb);  // drift_s uses time t (reference quirk, oc.py:807)
        rnd -= 0.5f * c2 * dt;
        rnd -= cdb;
      }
      rnd += gmm_pass1<PIPE>(prior, d, dp, P.x, P.rr);  // oc.py:825
    }
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

template <int KIND>
__global__ void __launch_bounds__(128) rollout_simt_kernel(const RolloutArgs a) {
  extern __shared__ float smem[];
  const ColLayout L = col_layout(a.s);
  SimtMlp mlp{a.s.mlp, Col{smem + L.act * blockDim.x + threadIdx.x, (int)blockDim.x}};
  rollout_body<KIND, 0, RuntimeTraits>(a, smem, nullptr, mlp);
}

}  // namespace lrds
