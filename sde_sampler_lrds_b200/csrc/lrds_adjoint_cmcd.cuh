// The adjoint of the CMCD simulate loop under ClippedCtrl (lrds_adjoint_cmcd, include/lrds_b200.h): one thread carries
// one particle's lambda_j = d loss / d x_j backwards over the K + 1 trajectory points that lrds_rollout wrote.  With
// u_j = clip(net(t_j, x_j)), D_j = clip(sig^2/2 (f_j score_pi(x_j) + (1 - f_j) score_0(x_j))) and
// e_k = w_b (c_k dt_k + sqrt(dt_k) z_k),  c_k = (D_k + D_{k+1}) / sig + u_k - u_{k+1}:
//
//   ubar_j   = [j<K] (e_j + sig dt_j lambda_{j+1}) - [j>=1] e_{j-1}                       -> cot_out[j]
//   Dbar_j   = [j<K] (e_j / sig + dt_j lambda_{j+1}) + [j>=1] e_{j-1} / sig
//   lambda_j = [j<K] lambda_{j+1} + J_net^T ([|net_j| <= clip_model] ubar_j)
//              + sig^2/2 (f_j H_pi(x_j) + (1 - f_j) H_0) ([|D_j^pre| <= cmcd_clip] Dbar_j)
//              + [j=K] (-w_b [|log pi(x_K)| <= clip_target] grad log pi(x_K))
//
// Point j needs e_{j-1}, i.e. u_{j-1} and D_{j-1}: every iteration first evaluates the control and the drift one point
// ahead (at x_{j-1}, without the GELU' tape) and carries q_{j-1} = D_{j-1} / sig - u_{j-1} into the next one, then
// recomputes the network at x_j with the tape for J_net^T.  H_pi is the exact Hessian of the diagonal mixture
// (gmm_score_jvp) or the PhiFour stencil, H_0 = -diag(1 / var_0) of the diagonal Gaussian prior in ref_0.
#pragma once
#include "lrds_adjoint.cuh"

namespace lrds {

// Shared-memory floats per particle.  The scratch area holds the network tape (activations and GELU' of every layer)
// and, after the backward pass through the network, the per-mode coefficients of the mixture Hessian-vector product.
struct AdjCmcdLayout {
  ColLayout c;  // x, act (= scratch), rt (target responsibilities)
  int tape, cm, lam, q, ea, eb, v, total;
};
__host__ __device__ inline AdjCmcdLayout adj_cmcd_layout(const lrds_spec& s) {
  AdjCmcdLayout L{};
  const int dp = s.mlp.d_pad;
  const int M = s.target.kind == LRDS_DISTR_GMM ? s.target.gmm.M : 0;
  const int trt = M > 1 ? (M + 3) / 4 * 4 : 0;
  int scratch = (s.mlp.num_hidden + 2) * C;
  if (M > scratch) scratch = (M + 3) / 4 * 4;
  int off = 0;
  L.c.x = off; off += dp;
  L.c.act = off; L.tape = off + C; L.cm = off;
  off += scratch;
  L.c.rt = off; off += trt;
  L.c.g = L.c.rr = L.c.rh = L.c.us = L.c.tsd = L.c.db = off;  // unused: logistic regression, reference, CMCD carry-over
  L.lam = off; off += dp;
  L.q = off; off += dp;
  L.ea = off; off += dp;
  L.eb = off; off += dp;
  L.v = off; off += dp;
  L.total = off;
  L.c.total = off;
  return L;
}

// v <- H_pi(x) v in place (x in P.x; GMM: responsibilities of x in P.rt from target_pass1)
__device__ __forceinline__ void target_hvp(const lrds_spec& s, const Particle& P, const Col4& v, const Col& cm) {
  const int d = s.d, dp = s.mlp.d_pad;
  if (s.target.kind == LRDS_DISTR_GMM) {
    gmm_score_jvp(gmm_at(s.target.gmm, 0), d, dp, P.x, P.rt, v, cm, v);
    return;
  }
  // PhiFour (Dirichlet-0): -beta [(3 x_i^2 - 1) / coef v_i + coef (2 v_i - v_{i-1} - v_{i+1})]
  const lrds_phi4& p = s.target.phi4;
  const float coef = p.a * (float)d;
  float vm = 0.f;
  for (int i = 0; i < d; ++i) {
    const float xi = P.x(i), vi = v(i), vp = i + 1 < d ? v(i + 1) : 0.f;
    v(i) = -p.beta * fmaf((3.0f * xi * xi - 1.0f) / coef, vi, coef * (2.0f * vi - vm - vp));
    vm = vi;
  }
}

__device__ __forceinline__ void adjoint_cmcd_body(const AdjointArgs& a, float* smem) {
  const lrds_spec& s = a.r.s;
  const int NT = blockDim.x, tid = threadIdx.x;
  const int b = blockIdx.x * NT + tid;
  if (b >= s.B) return;  // no CTA-wide synchronisation below
  const int d = s.d, dp = s.mlp.d_pad, K = s.K, nh = s.mlp.num_hidden, tkind = s.target.kind;
  const AdjCmcdLayout L = adj_cmcd_layout(s);
  const Particle P = make_particle(smem, L.c, NT, tid);
  // The scratch columns are rebuilt at every point with an opaque stride: that keeps the compiler from hoisting the
  // addresses of all their elements out of the loop (they do not fit in the registers)
  Col act, tape, cm;
  auto scratch_cols = [&]() {
    int nt = NT;
    asm volatile("" : "+r"(nt));
    act = Col{smem + L.c.act * nt + tid, nt};
    tape = Col{smem + L.tape * nt + tid, nt};
    cm = Col{smem + L.cm * nt + tid, nt};
  };
  auto col4 = [&](int off) { return Col4{smem + off * NT + 4 * tid, 4 * NT}; };
  const Col4 lam = col4(L.lam), q = col4(L.q), v = col4(L.v);
  Col4 ec = col4(L.ea), en = col4(L.eb);  // e_j, e_{j-1}
  const lrds_mlp& w = s.mlp;
  const GmmView tv0 = gmm_at(s.target.gmm, 0), prior = gmm_at(s.ref_0, 0);
  const float bound = clip_bound(s.clip_model), dbound = clip_bound(s.cmcd_clip);
  const float sg = s.cmcd_diff, isg = 1.0f / sg, h2 = 0.5f * sg * sg;
  const float wb = __ldg(a.row_w + b);
  auto row_of = [&](int j) { return s.steps + (int64_t)j * LRDS_STEP_STRIDE; };

  // control and drift at x_p (in P.x): q <- D_p / sig - u_p, and for p < K also e_p into en (q holding q_{p+1})
  auto ahead = [&](int p) {
    const float* row = row_of(p);
    const float f = __ldg(row + LRDS_STEP_FRAC), dt = __ldg(row + LRDS_STEP_DT), sqdt = __ldg(row + LRDS_STEP_SQRT_DT);
    target_pass1<false>(s, tkind, tv0, P, false);
    mlp_hidden<false>(w, row + LRDS_STEP_BIAS1, P.x, act);
    target_score_loop<false>(s, tkind, tv0, P, [&](int j0, const float(&xr)[JC], const float(&ts)[JC]) {
      float net[JC], z[JC];
      mlp_out_chunk(w, act, j0, net);
      if (p < K) noise_chunk(a.r, p, b, j0, z);
#pragma unroll
      for (int c = 0; c < JC; ++c) {
        const int j = j0 + c;
        float qn = 0.f, e = 0.f;
        if (j < d) {
          const float ps = -((xr[c] - prior.mu.ld1(j)) * prior.ivar.ld1(j));
          const float dr = langevin_drift(s, ts[c], ps, f), u = clipb(net[c], bound);
          qn = fmaf(dr, isg, -u);
          if (p < K) e = wb * fmaf(fmaf(dr, isg, u) + q(j), dt, sqdt * z[c]);
        }
        if (p < K) en(j) = e;
        q(j) = qn;
      }
    });
  };

  // lambda_K: the terminal term at x_K, then q_K
  load_state(a, K, b, P.x);
  {
    const float lt = target_pass1<false>(s, tkind, tv0, P, true);
    const float wt = (s.clip_target > 0.f && !(fabsf(lt) <= s.clip_target)) ? 0.f : wb;
    target_score_loop<false>(s, tkind, tv0, P, [&](int j0, const float(&xr)[JC], const float(&ts)[JC]) {
#pragma unroll
      for (int c = 0; c < JC; ++c) lam(j0 + c) = (j0 + c < d) ? -wt * ts[c] : 0.f;
    });
  }

  float chk = 0.f;
  for (int j = K + 1; j >= 0; --j) {  // j = K + 1 only evaluates q_K
    const bool last = j == K, first = j == 0;
    scratch_cols();
    if (!first) {  // e_{j-1} -> en, q_{j-1} -> q
      load_state(a, j - 1, b, P.x);
      ahead(j - 1);
    }
    if (j > K) continue;
    scratch_cols();
    const float* row = row_of(j);
    const float f = __ldg(row + LRDS_STEP_FRAC);
    const float dt = last ? 0.f : __ldg(row + LRDS_STEP_DT);
    load_state(a, j, b, P.x);
    mlp_hidden<false, true>(w, row + LRDS_STEP_BIAS1, P.x, act, tape);
    float da[C];  // d loss / d (last hidden activation), accumulated over the output chunks
#pragma unroll
    for (int n = 0; n < C; ++n) da[n] = 0.f;
    float* cot = a.cot_out + ((int64_t)j * s.B + b) * d;
    for (int j0 = 0; j0 < dp; j0 += JC) {
      float net[JC], gm[JC];
      mlp_out_chunk(w, act, j0, net);
#pragma unroll
      for (int c = 0; c < JC; ++c) {
        const int i = j0 + c;
        float ub = 0.f, db = 0.f;
        if (i < d) {
          if (!last) {
            const float e = ec(i), l = lam(i);
            ub = fmaf(sg * dt, l, e);
            db = fmaf(dt, l, e * isg);
          }
          if (!first) {
            const float e = en(i);
            ub -= e;
            db = fmaf(e, isg, db);
          }
          cot[i] = ub;
        }
        chk += ub;
        gm[c] = fabsf(net[c]) <= bound ? ub : 0.f;
        v(i) = db;
      }
      if (!first) {
#pragma unroll
        for (int n = 0; n < C; ++n) {
          const float4* wr = reinterpret_cast<const float4*>(w.w_out_t + (int64_t)n * dp + j0);
          const float4 p = __ldg(wr), r = __ldg(wr + 1);
          float t = da[n];
          t = fmaf(p.x, gm[0], t); t = fmaf(p.y, gm[1], t); t = fmaf(p.z, gm[2], t); t = fmaf(p.w, gm[3], t);
          t = fmaf(r.x, gm[4], t); t = fmaf(r.y, gm[5], t); t = fmaf(r.z, gm[6], t); t = fmaf(r.w, gm[7], t);
          da[n] = t;
        }
      }
    }
    if (first) break;  // lambda_0 is not needed: x_0 does not depend on the parameters
    // back through the hidden layers: dh = d loss / d pre-activation, rows of w_hid_t are the inputs
#pragma unroll
    for (int n = 0; n < C; ++n) da[n] *= tape(nh * C + n);
    for (int l = nh - 1; l >= 0; --l) {
      const float* wl = w.w_hid_t + (int64_t)l * C * C;
      for (int i = 0; i < C; ++i) act(i) = dot64(wl + i * C, da) * tape(l * C + i);
#pragma unroll
      for (int n = 0; n < C; ++n) da[n] = act(n);
    }
    // input layer (in place: lambda_{j+1}, resp. the terminal term at j = K, plus W_in^T dh)
    for (int i = 0; i < d; ++i) lam(i) += dot64(w.w_in_t + (int64_t)i * C, da);
    // the drift: mask of the clip at x_j, prior part sig^2/2 (1 - f) H_0, then the target part sig^2/2 f H_pi
    target_pass1<false>(s, tkind, tv0, P, false);
    const float hp = h2 * (1.0f - f), ht = h2 * f;
    target_score_loop<false>(s, tkind, tv0, P, [&](int j0, const float(&xr)[JC], const float(&ts)[JC]) {
#pragma unroll
      for (int c = 0; c < JC; ++c) {
        const int i = j0 + c;
        if (i < d) {
          const float iv = prior.ivar.ld1(i);
          const float ps = -((xr[c] - prior.mu.ld1(i)) * iv);
          const float pre = (ts[c] * f + ps * (1.0f - f)) * h2;  // langevin_drift before its clip
          const float m = fabsf(pre) <= dbound ? v(i) : 0.f;
          v(i) = m;
          lam(i) = fmaf(-hp * iv, m, lam(i));
        }
      }
    });
    target_hvp(s, P, v, cm);
    for (int i = 0; i < d; ++i) lam(i) = fmaf(ht, v(i), lam(i));
    const Col4 t = ec;
    ec = en;
    en = t;
  }
  report_status(s, true, false, !isfinite(chk));
}

}  // namespace lrds
