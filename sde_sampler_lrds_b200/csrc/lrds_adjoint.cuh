// The adjoint of the LINEAR simulate loop under ClippedCtrl (lrds_adjoint, include/lrds_b200.h): one thread carries one
// particle's lambda_k = d loss / d x_k backwards through the K steps, reading the states x_k that lrds_rollout wrote and
// the same table fields, update form and Ito form as the rollout (so DIS needs nothing special).  Per step:
//
//   gbar_k   = w_b (2 W_COST g_k + e_k) + (dx_{k+1} / dg) lambda_{k+1}          e_k = Ito weight * z_k
//   lambda_k = a_k lambda_{k+1} + c_k J_r(x_k) lambda_{k+1} + J_net^T ([|net| <= clip_model] gbar_k)
//
// (a_k, c_k, dx_{k+1}/dg) = (A, B, B) for the AXPY update and (1 - A dt, C dt, B dt) for EM.  gbar_k goes to cot_out; the
// parameter gradient is lrds_mlp_grad / autograd with that cotangent (train.py).  The network is recomputed from x_k in
// fp32 with GELU' kept in shared-memory columns, the reference Jacobian J_r is the exact Hessian of the diagonal mixture
// log-density (quadratic forms as in gmm_pass1), and lambda_K uses the existing score device functions.
#pragma once
#include "lrds_rollout_simt.cuh"

namespace lrds {

struct AdjointArgs {
  RolloutArgs r;       // spec and the rollout's noise source (recorded increments or the Philox key); r.x0 unused
  const float* traj;   // [K+1][B][d]
  const float* row_w;  // [B] d loss / d rnd_b
  float* cot_out;      // [K][B][d]
};

// Shared-memory floats per particle.  One scratch area holds, at different times, the network tape (activations and
// GELU' of every layer), the target's per-particle scratch at x_K and the per-mode coefficients of J_r.
struct AdjLayout {
  ColLayout c;  // x, act (= scratch), rt / g (target, in the scratch), rr (reference responsibilities)
  int tape, cm, lam, lamn, total;
};
// net_cols: the network tape lives in shared memory (the SIMT kernel; the tensor-core kernel keeps it in TMEM)
__host__ __device__ inline AdjLayout adj_layout(const lrds_spec& s, bool net_cols = true) {
  AdjLayout L{};
  const int dp = s.mlp.d_pad;
  const bool tmix = s.target.kind == LRDS_DISTR_GMM && s.target.gmm.M > 1;
  const int trt = tmix ? (s.target.gmm.M + 3) / 4 * 4 : 0;
  const int tgt = trt + (s.target.kind == LRDS_DISTR_LOGREG ? s.target.logreg.n_pad : 0);
  const int mref = s.has_ref_ctrl && s.ref_t.M > 1 ? (s.ref_t.M + 3) / 4 * 4 : 0;
  const int mr = !s.init_cost && s.ref_0.M > 1 && s.ref_0.M > mref ? s.ref_0.M : mref;
  int scratch = net_cols ? (s.mlp.num_hidden + 2) * C : 0;
  if (tgt > scratch) scratch = tgt;
  if (mref > scratch) scratch = mref;
  int off = 0;
  L.c.x = off; off += dp;
  L.c.act = off; L.tape = off + C; L.c.rt = off; L.c.g = off + trt; L.cm = off;
  off += scratch;
  L.c.rr = L.c.rh = off; off += (mr + 3) / 4 * 4;
  L.lam = off; off += dp;
  L.lamn = off; off += dp;
  L.c.us = L.c.tsd = L.c.db = off;
  L.total = off;
  return L;
}

// out = J_r v for the diagonal mixture score r(x) = sum_m r_m h_m, h_m = -(x - mu_m) / var_m, with the responsibilities
// r_m in column r (gmm_pass1):  J_r v = sum_m r_m (-v / var_m + (h_m . v - s . v) h_m),  s . v = sum_m r_m (h_m . v).
// A single Gaussian: -v / var.  Padded dims (mu = ivar = 0) give 0.
__device__ __forceinline__ void gmm_score_jvp(const GmmView& g, int d, int dp, const Col4& x, const Col4& r, const Col4& v,
                                              const Col& cm, const Col4& out) {
  const int nq = (d + 3) >> 2;
  if (g.M == 1) {
    for (int c = 0; c < (dp >> 2); ++c) {
      const float4 vv = v.ld4(c), iv = g.ivar.ld4(c);
      out.st4(c, make_float4(-(vv.x * iv.x), -(vv.y * iv.y), -(vv.z * iv.z), -(vv.w * iv.w)));
    }
    return;
  }
  float sv = 0.f;
  for (int m = 0; m < g.M; ++m) {
    const PPtr<false> mu = g.mu + m * dp, iv = g.ivar + m * dp;
    float hv = 0.f;
    for (int c = 0; c < nq; ++c) {
      const float4 xv = x.ld4(c), vv = v.ld4(c), mv = mu.ld4(c), ivv = iv.ld4(c);
      hv = fmaf(-((xv.x - mv.x) * ivv.x), vv.x, hv);
      hv = fmaf(-((xv.y - mv.y) * ivv.y), vv.y, hv);
      hv = fmaf(-((xv.z - mv.z) * ivv.z), vv.z, hv);
      hv = fmaf(-((xv.w - mv.w) * ivv.w), vv.w, hv);
    }
    cm(m) = hv;
    sv = fmaf(r(m), hv, sv);
  }
  for (int c = 0; c < (dp >> 2); ++c) {
    const float4 xv = x.ld4(c), vv = v.ld4(c);
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int m = 0; m < g.M; ++m) {
      const float rm = r(m), cf = cm(m) - sv;
      const float4 mv = (g.mu + m * dp).ld4(c), ivv = (g.ivar + m * dp).ld4(c);
      acc.x = fmaf(rm, fmaf(cf, -((xv.x - mv.x) * ivv.x), -(vv.x * ivv.x)), acc.x);
      acc.y = fmaf(rm, fmaf(cf, -((xv.y - mv.y) * ivv.y), -(vv.y * ivv.y)), acc.y);
      acc.z = fmaf(rm, fmaf(cf, -((xv.z - mv.z) * ivv.z), -(vv.z * ivv.z)), acc.z);
      acc.w = fmaf(rm, fmaf(cf, -((xv.w - mv.w) * ivv.w), -(vv.w * ivv.w)), acc.w);
    }
    out.st4(c, acc);
  }
}

// w . v for a 64-float weight row (read-only path, warp-uniform) and a register vector
__device__ __forceinline__ float dot64(const float* __restrict__ wrow, const float (&v)[C]) {
  const float4* w4 = reinterpret_cast<const float4*>(wrow);
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
  for (int q = 0; q < C / 4; ++q) {
    const float4 t = __ldg(w4 + q);
    a0 = fmaf(t.x, v[4 * q], a0);
    a1 = fmaf(t.y, v[4 * q + 1], a1);
    a2 = fmaf(t.z, v[4 * q + 2], a2);
    a3 = fmaf(t.w, v[4 * q + 3], a3);
  }
  return (a0 + a1) + (a2 + a3);
}

// Per-step coefficients of the recursion, from the same table fields and forms as the rollout
struct AdjStep {
  float cg;   // d x_{k+1} / d g
  float ak;   // d x_{k+1} / d x_k (identity part)
  float ck;   // factor of J_r
  float wc2;  // 2 W_COST
  float ew;   // Ito weight of z_k
};
__device__ __forceinline__ AdjStep adj_step(const lrds_spec& s, const float* __restrict__ row) {
  const float A = __ldg(row + LRDS_STEP_A), Bc = __ldg(row + LRDS_STEP_B), Cc = __ldg(row + LRDS_STEP_C);
  const float dt = __ldg(row + LRDS_STEP_DT), sqdt = __ldg(row + LRDS_STEP_SQRT_DT);
  const float wito = __ldg(row + LRDS_STEP_W_ITO), sigu = __ldg(row + LRDS_STEP_SIGU);
  const bool em = s.update_form == LRDS_UPDATE_EM;
  AdjStep st;
  st.cg = em ? Bc * dt : Bc;
  st.ak = em ? 1.0f - A * dt : A;
  st.ck = em ? Cc * dt : Bc;
  st.wc2 = 2.0f * __ldg(row + LRDS_STEP_W_COST);
  st.ew = s.ito_form == LRDS_ITO_SCALED ? wito : s.ito_form == LRDS_ITO_EM ? sqdt : s.ito_form == LRDS_ITO_DDS ? sigu * wito : 0.f;
  return st;
}
// gbar = w (2 W_COST g + e) + (d x_{k+1} / d g) lambda_{k+1}
__device__ __forceinline__ float adj_gbar(const AdjStep& st, float w, float g, float z, float lam) {
  return fmaf(w, fmaf(st.wc2, g, st.ew * z), st.cg * lam);
}

// lambda_K = w (grad ref_0(x_K) - [|target(x_K)| <= clip_target] grad target(x_K)) into `lam` (x_K in P.x); init_cost
// (DIS): no ref_0 term
__device__ __forceinline__ void adj_terminal(const lrds_spec& s, const Particle& P, const Col4& lam, float w) {
  const int d = s.d, dp = s.mlp.d_pad, tkind = s.target.kind;
  const GmmView tv0 = gmm_at(s.target.gmm, 0), r0 = gmm_at(s.ref_0, 0);
  const float lt = target_pass1<false>(s, tkind, tv0, P, true);
  const float wt = (s.clip_target > 0.f && !(fabsf(lt) <= s.clip_target)) ? 0.f : w;
  const bool ref0 = !s.init_cost;
  if (ref0 && r0.M > 1) gmm_pass1<false>(r0, d, dp, P.x, P.rr);
  target_score_loop<false>(s, tkind, tv0, P, [&](int j0, const float(&xr)[JC], const float(&ts)[JC]) {
    float rs[JC] = {};
    if (ref0) gmm_score_chunk<false>(r0, d, dp, xr, P.rr, j0, rs);
#pragma unroll
    for (int c = 0; c < JC; ++c) lam(j0 + c) = (j0 + c < d) ? w * rs[c] - wt * ts[c] : 0.f;
  });
}

// out = J_r(x_k) lambda for the time-marginal reference of step k (x_k in P.x)
__device__ __forceinline__ void adj_jr(const lrds_spec& s, int k, const Particle& P, const Col4& lam, const Col& cm,
                                       const Col4& out) {
  const GmmView rv = gmm_at(s.ref_t, k);
  if (rv.M > 1) gmm_pass1<false>(rv, s.d, s.mlp.d_pad, P.x, P.rr);
  gmm_score_jvp(rv, s.d, s.mlp.d_pad, P.x, P.rr, lam, cm, out);
}

__device__ __forceinline__ void load_state(const AdjointArgs& a, int row, int b, const Col4& x) {
  const lrds_spec& s = a.r.s;
  const float* p = a.traj + ((int64_t)row * s.B + b) * s.d;
  for (int j = 0; j < s.mlp.d_pad; ++j) x(j) = (j < s.d) ? __ldg(p + j) : 0.f;
}

// The network policy is the fp32 FFMA one (SimtMlp's arithmetic); every precision the entry point accepts runs it.
__device__ __forceinline__ void adjoint_body(const AdjointArgs& a, float* smem) {
  const lrds_spec& s = a.r.s;
  const int NT = blockDim.x, tid = threadIdx.x;
  const int b = blockIdx.x * NT + tid;
  if (b >= s.B) return;  // no CTA-wide synchronisation below
  const int d = s.d, dp = s.mlp.d_pad, K = s.K, nh = s.mlp.num_hidden;
  const AdjLayout L = adj_layout(s);
  const Particle P = make_particle(smem, L.c, NT, tid);
  const Col act{smem + L.c.act * NT + tid, NT}, tape{smem + L.tape * NT + tid, NT}, cm{smem + L.cm * NT + tid, NT};
  Col4 lam{smem + L.lam * NT + 4 * tid, 4 * NT}, lamn{smem + L.lamn * NT + 4 * tid, 4 * NT};
  const lrds_mlp& w = s.mlp;
  const float bound = clip_bound(s.clip_model);
  const float wb = __ldg(a.row_w + b);
  const bool has_ref = s.has_ref_ctrl != 0;
  for (int j = 0; j < dp; ++j) lamn(j) = 0.f;

  load_state(a, K, b, P.x);
  adj_terminal(s, P, lam, wb);

  float chk = 0.f;
  for (int k = K - 1; k >= 0; --k) {
    const float* row = s.steps + (int64_t)k * LRDS_STEP_STRIDE;
    const AdjStep st = adj_step(s, row);
    const bool back = k > 0;  // lambda_0 is not needed: x_0 does not depend on the parameters
    load_state(a, k, b, P.x);
    if (back && has_ref) adj_jr(s, k, P, lam, cm, lamn);  // lamn = J_r(x_k) lambda_{k+1}
    mlp_hidden<false, true>(w, row + LRDS_STEP_BIAS1, P.x, act, tape);
    float da[C];  // d loss / d (last hidden activation), accumulated over the output chunks
#pragma unroll
    for (int n = 0; n < C; ++n) da[n] = 0.f;
    float* cot = a.cot_out + ((int64_t)k * s.B + b) * d;
    for (int j0 = 0; j0 < dp; j0 += JC) {
      float net[JC], z[JC], lr[JC], gm[JC];
      mlp_out_chunk(w, act, j0, net);
      noise_chunk(a.r, k, b, j0, z);
      load_chunk(lam, j0, lr);
#pragma unroll
      for (int c = 0; c < JC; ++c) {
        const float g = clipb(net[c], bound);
        float gb = adj_gbar(st, wb, g, z[c], lr[c]);
        if (j0 + c >= d) gb = 0.f;
        else cot[j0 + c] = gb;
        chk += gb;
        gm[c] = fabsf(net[c]) <= bound ? gb : 0.f;
      }
      if (back) {
#pragma unroll
        for (int n = 0; n < C; ++n) {
          const float4* wr = reinterpret_cast<const float4*>(w.w_out_t + (int64_t)n * dp + j0);
          const float4 p = __ldg(wr), q = __ldg(wr + 1);
          float t = da[n];
          t = fmaf(p.x, gm[0], t); t = fmaf(p.y, gm[1], t); t = fmaf(p.z, gm[2], t); t = fmaf(p.w, gm[3], t);
          t = fmaf(q.x, gm[4], t); t = fmaf(q.y, gm[5], t); t = fmaf(q.z, gm[6], t); t = fmaf(q.w, gm[7], t);
          da[n] = t;
        }
      }
    }
    if (!back) break;
    // back through the hidden layers: dh = d loss / d pre-activation, rows of w_hid_t are the inputs
#pragma unroll
    for (int n = 0; n < C; ++n) da[n] *= tape(nh * C + n);
    for (int l = nh - 1; l >= 0; --l) {
      const float* wl = w.w_hid_t + (int64_t)l * C * C;
      for (int i = 0; i < C; ++i) act(i) = dot64(wl + i * C, da) * tape(l * C + i);
#pragma unroll
      for (int n = 0; n < C; ++n) da[n] = act(n);
    }
    // input layer: lambda_k = a_k lambda_{k+1} + c_k J_r lambda_{k+1} + W_in^T dh, four dims at a time
    for (int c = 0; 4 * c < d; ++c) {
      const float4 l4 = lam.ld4(c), j4 = has_ref ? lamn.ld4(c) : make_float4(0.f, 0.f, 0.f, 0.f);
      const float lv[4] = {l4.x, l4.y, l4.z, l4.w}, jv[4] = {j4.x, j4.y, j4.z, j4.w};
      float o[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int j = 4 * c + e;
        o[e] = j < d ? fmaf(st.ak, lv[e], st.ck * jv[e]) + dot64(w.w_in_t + (int64_t)j * C, da) : 0.f;
      }
      lamn.st4(c, make_float4(o[0], o[1], o[2], o[3]));
    }
    const Col4 t = lam;
    lam = lamn;
    lamn = t;
  }
  report_status(s, true, false, !isfinite(chk));
}

}  // namespace lrds
