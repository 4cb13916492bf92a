// The benchmark loop (lrds_rollout_mix.cuh, configuration MixBench: RDS with a mixture reference, ScoreCtrl over a mixture
// target, exponential-integrator / DDPM-like update) for SMALL batches - the reference's own operating points: evaluation
// batches of 8192 and training batches of 512 .. 2048 particles (SURVEY Appendix A).  There a rollout is bound by the
// latency of one grid step, not by throughput: a CTA of the throughput kernel holds one or two warps and walks through
// ~6 k instructions and a dozen tensor-core round trips per step on its own.
//
// Here a CTA owns ONE tile of up to 128 particles and serves every particle with FOUR threads: warps w, w + 4, w + 8,
// w + 12 own the same TMEM lanes (thread <-> lane: 32 (w % 4) + lane) and split the work of a step
//   x -> A operand          16 dims each
//   responsibilities        thread 0: target mixture, thread 1: reference mixture (logit GEMM columns, softmax, error
//                           bound, exact quadratic forms as the fallback - exactly the arithmetic of the throughput kernel)
//   network epilogues       16 of the 64 hidden units each
//   contraction + update    the 8-dim chunks round robin; with one tile per SM the 512 TMEM columns hold ALL chunks
//                           (columns 128 + 32 c), so the whole contraction is ONE batch instead of one round trip per chunk
//   logits                  in their own columns, issued in ONE batch with the network's first GEMM (same A operand x)
//   noise                   the step's increments of a thread's chunks are drawn behind the hidden GEMMs
// and add their partial log-weights at the end.  Per step: 5 tensor-core round trips instead of 13, ~1.5 k instead of
// ~6 k instructions on the critical path.  The states are bit-identical to the throughput kernel's (same per-dim /
// per-mode arithmetic, same Philox counters); the log-weights agree to fp32 rounding (four partial sums instead of
// one running sum) - tests/test_edge_cases_gpu.py checks both.  LRDS_MIX_SMALL=0 in the environment switches the
// kernel off (tests and A/B timings).
#pragma once
#include "lrds_rollout_mix.cuh"

namespace lrds {

constexpr int MIXS_TP = 4;                  // threads per particle
constexpr int MIXS_THREADS = 128 * MIXS_TP;  // 16 warps
constexpr uint32_t MIXS_CHUNK_COL = 128;     // chunk c of the contractions: columns 128 + 32 c of the tile
constexpr uint32_t MIXS_LOGIT_COL = 480;     // the logits of the two mixtures: the tile's last 32 columns

__host__ __device__ inline bool mix_small_applicable(const lrds_spec& s, int sms) {
  return mix_tc_config(s) == 0 && s.B <= 128 * sms && s.mlp.d_pad <= 64 && s.mlp.num_hidden >= 1;
}

template <int PREC>
__global__ void __launch_bounds__(MIXS_THREADS, 1)
rollout_mix_small_kernel(const RolloutArgs a, const uint8_t* __restrict__ image) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  const lrds_spec& s = a.s;
  const TcLayout TL = tc_layout(s.d, s.mlp.num_hidden, PREC);
  const int tid = threadIdx.x;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int sub = warp >> 2;   // which of the particle's four threads
  const int ptid = tid & 127;  // particle within the tile = TMEM lane
  constexpr int NT = 128;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + TL.bytes);  // [0] image, [1] MMAs of the tile done, [2] the logits of a step, [3] the first contraction chunk of every thread
  uint32_t* cnts = reinterpret_cast<uint32_t*>(smem_raw + TL.bytes + TC_TAIL_BYTES);  // [0] hand-offs, [4 + i] step buffer i released
  uint8_t* stage = smem_raw + TL.bytes + TC_TAIL_BYTES + MIX_TAIL_BYTES;
  const StageLayout SL = stage_layout(s, 2, true);
  float* cols = reinterpret_cast<float*>(stage + ((SL.total + 15u) & ~15u));
  const int d = s.d, dp = s.mlp.d_pad, K = s.K;
  float* part = cols + (size_t)dp * NT;  // [4][128] partial log-weights
  uint64_t* sbar = reinterpret_cast<uint64_t*>(stage);
  const uint32_t mix_off_t = SL.tgt_logc_bytes + SL.tgt_param_bytes;
  const uint32_t mix_off_r = SL.row_bytes + SL.ref_logc_bytes + SL.ref_param_bytes;
  auto steps01 = [&]() {
    mix_load_step<true>(s, SL, stage, 0);
    if (K > 1) mix_load_step<true>(s, SL, stage, 1);
  };
  const uint32_t tmem =
      __shfl_sync(0xffffffffu, tc_cta_begin(smem_raw, TL, image, 512u, warp, 4, sbar, 2, cnts, 6, 0u, steps01), 0);
  MixTc<PREC> mlp;
  // hand-offs: the threads without a mixture to evaluate have slack
  mlp.init(TL, smem_raw, tmem, warp, bars + 1, cnts, 16u, (warp == 15 ? 1u : 0u) | (warp == 14 ? 2u : 0u), dp);
  const int Mt = s.target.gmm.M;
  const uint32_t contr_bytes = gmm_mix_contr_bytes(Mt, dp), lg_part = gmm_mix_logit_part_bytes(Mt, dp);
  const uint32_t lg_tail_off = contr_bytes + 2u * lg_part;
  mlp.lbo = (uint32_t)(2 * dp) * 16u;
  mlp.part_bytes = (contr_bytes - 16u) / 2u;
  mlp.lg_part = lg_part;

  const int b_raw = blockIdx.x * NT + ptid;
  const bool live = b_raw < s.B;
  const int b = live ? b_raw : s.B - 1;
  const Col4 X{cols + 4 * ptid, 4 * NT};
  for (int j = sub; j < dp; j += MIXS_TP) X(j) = (j < d) ? __ldg(a.x0 + (int64_t)b * d + j) : 0.f;
  if (a.traj_out != nullptr && live)
    for (int j = sub; j < d; j += MIXS_TP) a.traj_out[(int64_t)b * d + j] = __ldg(a.x0 + (int64_t)b * d + j);
  const CtrlConst cc = ctrl_const(s);
  const GmmView tv0 = gmm_at(s.target.gmm, 0);
  const GmmViewT<true> tv = staged_view(stage + SL.off_tgt, tv0, SL.tgt_logc_bytes, SL.tgt_param_bytes);
  const uint32_t tgt_img = ptx::smem_u32(stage + SL.off_tgt + mix_off_t);
  const int nchunk = dp / JC, nq = (d + 3) >> 2;
  float rnd = 0.f;
#ifdef LRDS_MIX_TIMING
  unsigned long long* tmw = reinterpret_cast<unsigned long long*>(part + MIXS_TP * NT) + warp * 16;
  if ((tid & 31) < 16) tmw[tid & 31] = 0;
  __syncwarp();
  mlp.tm.w = tmw;
#endif
  mlp.tm.start();

  uint32_t lphase = 0;  // parity of the logit barrier (waited for by the threads that own a mixture)
  uint32_t cphase = 0;  // parity of the first-chunks barrier
  for (int k = 0; k < K; ++k) {
    __syncthreads();  // the step's x is complete and visible to the four threads of every particle
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
    const float ust = *reinterpret_cast<const float*>(stage + SL.off_tgt + mix_off_t + contr_bytes - 16u);
    const float usr = *reinterpret_cast<const float*>(buf + mix_off_r + contr_bytes - 16u);
    if (16 * sub < TL.Kin) {
      float v[16];
#pragma unroll
      for (int h = 0; h < 4; ++h) {
        const int j0 = 16 * sub + 4 * h;
        const float4 q = j0 < dp ? X.ld4(j0 >> 2) : make_float4(0.f, 0.f, 0.f, 0.f);
        v[4 * h + 0] = q.x; v[4 * h + 1] = q.y; v[4 * h + 2] = q.z; v[4 * h + 3] = q.w;
      }
      mlp.store16_half(8 * sub, v);
    }
    mlp.tm.mark(1);
    // responsibilities: thread 0 the target mixture, thread 1 the reference mixture (lrds_rollout_mix.cuh)
    uint32_t r_p[16];
    bool need = sub < 2, ok = false;
    const PPtr<true> tail{(sub == 0 ? tgt_img : ref_img) + lg_tail_off};
    const PPtr<true> tail_t{tgt_img + lg_tail_off}, tail_r{ref_img + lg_tail_off};
    const bool lg_t = tail_t.ld1(MIX_MAX_M + 3) != 0.f, lg_r = tail_r.ld1(MIX_MAX_M + 3) != 0.f;  // CTA-uniform
    // ONE hand-off: the logits of both mixtures (own columns, committed to their own mbarrier: they complete first and
    // the softmax of the threads that own them overlaps the MMAs of the network's first GEMM), then that GEMM
    mlp.arrive_issue([&]() {
      if (lg_t) mlp.logit(0, tgt_img + contr_bytes, (int)MIXS_LOGIT_COL);
      if (lg_r) mlp.logit(1, ref_img + contr_bytes, (int)MIXS_LOGIT_COL);
      ptx::mma_commit(bars + 2);
      mlp.gemm(TL.off_in, TL.Kin, C);
    });
    mlp.tm.mark(2);
    float xnorm = 0.f;
    if (sub < 2) {
      u64 n2 = 0;
      for (int c = 0; c < nq; ++c) {
        const ulonglong2 xv = X.ldu(c);
        n2 = f2::fma(xv.x, xv.x, n2);
        n2 = f2::fma(xv.y, xv.y, n2);
      }
      xnorm = sqrtf(f2::hsum1(n2));
    }
    if (sub < 2) {  // warps 0 .. 7: one wait per step and commit, so the parity never runs ahead of a waiter
      ptx::mbar_wait(bars + 2, lphase);
      lphase ^= 1u;
      ptx::tc_fence_after();
    }
    mlp.tm.mark(3);
    if (sub < 2 && (sub == 0 ? lg_t : lg_r)) {
      uint32_t lg[16];
      ptx::tmem_ld16(mlp.tm_lane + MIXS_LOGIT_COL + (uint32_t)sub * MIX_MAX_M, lg);
      ptx::tmem_wait_ld();
      ok = mlp.softmax_logits(lg, tail, xnorm, r_p);
      need = __any_sync(0xffffffffu, !ok);
    }
    mlp.tm.mark(4);
    if (need) {  // warp-uniform: the exact quadratic forms of this thread's mixture
      float r[MIX_MAX_M];
      uint32_t p[16];
      if (sub == 0) gmm_pass1_pair(tv, d, dp, X, r);
      else gmm_pass1_pair(rv, d, dp, X, r);
      mlp.pack_r(r, p);
#pragma unroll
      for (int i = 0; i < 16; ++i) r_p[i] = ok ? r_p[i] : p[i];
    }
    mlp.tm.mark(6);
    const float* bh = reinterpret_cast<const float*>(smem_raw + TL.off_bhid);
    mlp.tm.mark(6);
    float z0[JC], z1[JC];  // the increments of this thread's first two chunks, drawn behind the hidden GEMMs
    const bool two = sub + MIXS_TP < nchunk;
    for (int l = 0; l <= TL.nh; ++l) {
      if (l > 0) {
        if (l == 1) noise_chunk(a, k, b, sub * JC, z0);
        else if (l == 2 && two) noise_chunk(a, k, b, (sub + MIXS_TP) * JC, z1);
      }
      mlp.wait();  // l == 0: the first GEMM, issued behind the logits
      mlp.tm.mark(7);
      if (l == 0) mlp.template epilogue_f16<false, 16>(row + LRDS_STEP_BIAS1, 0, 16 * sub, 16 * sub + 16);
      else mlp.template epilogue_f16<false, 16>(bh + (l - 1) * C, l, 16 * sub, 16 * sub + 16);
      if (l < TL.nh) mlp.issue(TL.off_hid + (uint32_t)(l * C * C * TL.es), C, C);
      else mlp.issue(TL.off_out, C, TL.Nout);
      mlp.tm.mark(8);
    }
    if (TL.nh < 1) noise_chunk(a, k, b, sub * JC, z0);  // (fewer hidden GEMMs than chunks per thread: draw what is left now)
    if (TL.nh < 2 && two) noise_chunk(a, k, b, (sub + MIXS_TP) * JC, z1);
    mlp.wait();
    mlp.tm.mark(9);
    if (sub < 2) mlp.store_r(sub, r_p);
    mlp.arrive_issue([&]() {  // the whole contraction in one hand-off: chunk c -> columns 128 + 32 c; the chunks the
      // threads take first are committed to their own mbarrier and are consumed while the others are still in the pipe
      for (int c = 0; c < nchunk; ++c) {
        if (c == MIXS_TP) ptx::mma_commit(bars + 3);
        mlp.template chunk<true, true>(c, tgt_img, ref_img, MIXS_CHUNK_COL + 32u * (uint32_t)c);
      }
      if (nchunk <= MIXS_TP) ptx::mma_commit(bars + 3);
    });
    const u64 A2 = f2::pk(A), B2 = f2::pk(Bc), C2 = f2::pk(Cc), usr2 = f2::pk(usr);
    const u64 gs2 = f2::pk((cc.scale_score * gamma) * ust);
    const float bts = cc.bound_score / ust;
    u64 su2 = 0, sito = 0;
    mlp.tm.mark(10);
    ptx::mbar_wait(bars + 3, cphase);
    cphase ^= 1u;
    ptx::tc_fence_after();
    mlp.tm.mark(11);
    bool waited = false;  // the hand-off's second commit (the tile barrier): once per step in every thread
    for (int c = sub, ci = 0; c < nchunk; c += MIXS_TP, ++ci) {
      if (ci == 1) {
        mlp.wait();
        waited = true;
      }
      const int j0 = c * JC;
      uint32_t m[32];
      ptx::tmem_ld32(mlp.tm_lane + MIXS_CHUNK_COL + 32u * (uint32_t)c, m);
      ptx::tmem_wait_ld();
      const ulonglong2 xa = X.ldu(2 * c), xb = X.ldu(2 * c + 1);
      const u64 XV[4] = {xa.x, xa.y, xb.x, xb.y};
      u64 U[4], XN[4];
      float z[JC];
      mlp.out_chunk2(j0, U);
      if (ci < 2) {
#pragma unroll
        for (int i = 0; i < JC; ++i) z[i] = ci == 0 ? z0[i] : z1[i];
      } else {
        noise_chunk(a, k, b, j0, z);
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const u64 ta = f2::pack(__uint_as_float(m[2 * q]), __uint_as_float(m[2 * q + 1]));
        const u64 tb = f2::pack(__uint_as_float(m[8 + 2 * q]), __uint_as_float(m[9 + 2 * q]));
        const u64 ra = f2::pack(__uint_as_float(m[16 + 2 * q]), __uint_as_float(m[17 + 2 * q]));
        const u64 rb = f2::pack(__uint_as_float(m[24 + 2 * q]), __uint_as_float(m[25 + 2 * q]));
        float t0, t1, u0, u1;
        f2::unpack(f2::fma(XV[q], ta, tb), t0, t1);
        f2::unpack(U[q], u0, u1);
        u64 v = f2::pack(clipb(u0, cc.bound_model), clipb(u1, cc.bound_model));
        v = f2::fma(f2::pack(clipb(t0, bts), clipb(t1, bts)), gs2, v);
        const u64 rraw = f2::fma(XV[q], ra, rb);
        const u64 z2 = f2::pack(z[2 * q], z[2 * q + 1]);
        su2 = f2::fma(v, v, su2);
        sito = f2::fma(v, z2, sito);
        const u64 rv2 = f2::fma(rraw, usr2, v);
        XN[q] = f2::fma(C2, z2, f2::fma(A2, XV[q], f2::mul(B2, rv2)));
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
    if (!waited) mlp.wait();  // threads with a single chunk (or none)
    rnd += wcost * f2::hsum1(su2);
    rnd += wito * f2::hsum1(sito);
    __syncwarp();
    if ((tid & 31) == 0) {  // the CTA's last warp to finish the step refills its buffer with the operands of step k + 2
      const uint32_t old = ptx::atom_add_acq_rel(cnts + 4 + (k & 1), 1u);
      if (old == (uint32_t)((k >> 1) * 16 + 15) && k + 2 < K) mix_load_step<true>(s, SL, stage, k + 2);
    }
    mlp.tm.mark(12);
  }
#ifdef LRDS_MIX_TIMING
  __syncwarp();
  if ((blockIdx.x == 0 || blockIdx.x == gridDim.x / 2) && (tid & 31) < 16)
    g_mix_timing[((blockIdx.x ? 1 : 0) * 16 + warp) * 16 + (tid & 31)] = tmw[tid & 31];
#endif
  __syncthreads();  // final state complete
  part[sub * NT + ptid] = rnd;
  __syncthreads();
  float xsum = 0.f;
  if (live && a.x_out != nullptr)
    for (int j = sub; j < d; j += MIXS_TP) {
      const float v = X(j);
      xsum += v;
      a.x_out[(int64_t)b * d + j] = v;
    }
  bool nonfinite = false;
  if (sub == 0) {  // terminal cost: rnd += reference_log_prob(x) - terminal_unnorm_log_prob(x)   (oc.py:505, 645)
    // the partial sums are added in the order the throughput kernel accumulates a particle's chunks within a step only
    // up to rounding: the log-weight agrees with it to fp32 rounding, not bit for bit
    rnd = ((part[ptid] + part[NT + ptid]) + part[2 * NT + ptid]) + part[3 * NT + ptid];
    const float lref = gmm_logp_any(gmm_at(s.ref_0, 0), d, dp, X);
    float rt[MIX_MAX_M];
    const float ltgt = gmm_pass1_pair(tv, d, dp, X, rt);
    rnd += lref - clipf(ltgt, s.clip_target);
    if (live) a.rnd_out[b] = rnd;
    nonfinite = !isfinite(rnd + xsum);  // (a non-finite coordinate reaches rnd through the terminal log-densities)
  }
  report_status(s, live, mlp.saturated(), nonfinite);
  tc_cta_end(warp, tmem, 512u);
}

// one CTA per tile of 128 particles; shared memory: [weight image | barriers | counters | operand stage | x columns | partial sums]
inline bool plan_rollout_mix_small(const lrds_spec& s, int smem_cap, int sms, TcPlan* out) {
  if (!mix_small_applicable(s, sms)) return false;
  const TcLayout TL = tc_layout(s.d, s.mlp.num_hidden, s.precision);
  if (TL.tile_cols != 128 || MIXS_CHUNK_COL + 32u * (uint32_t)(s.mlp.d_pad / JC) > MIXS_LOGIT_COL) return false;
  const size_t bytes = (size_t)TL.bytes + TC_TAIL_BYTES + MIX_TAIL_BYTES + ((stage_layout(s, 2, true).total + 15u) & ~15u) +
                       ((size_t)s.mlp.d_pad + MIXS_TP) * 128 * sizeof(float)
#ifdef LRDS_MIX_TIMING
                       + 16 * 16 * 8
#endif
      ;
  if (bytes > (size_t)smem_cap) return false;
  out->warps = MIXS_THREADS / 32;
  out->grid = (s.B + 127) / 128;
  out->staged = 2;
  out->tmem_cols = 512;
  out->smem = bytes;
  return true;
}

}  // namespace lrds
