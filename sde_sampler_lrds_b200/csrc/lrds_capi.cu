// C ABI of liblrds_b200.so (declared in include/lrds_b200.h): argument validation, launch configuration, the error
// channel and launch counter shared by every translation unit, and the small auxiliary kernels (estimator partials,
// control / distribution evaluation, MALA chains, score cotangent sums, operand-image packers, axpy step, RNG dump).
#include <cuda_runtime.h>

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>

#include "lrds_adjoint.cuh"
#include "lrds_adjoint_cmcd.cuh"
#include "lrds_internal.h"
#include "lrds_rollout_simt.cuh"

namespace {
thread_local char g_err[512] = "";
std::atomic<int64_t> g_launches{0};
}  // namespace

namespace lrds {

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

int cuda_fail(cudaError_t e, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  const int n = vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  if (n >= 0 && (size_t)n < sizeof(g_err)) snprintf(g_err + n, sizeof(g_err) - n, ": %s", cudaGetErrorString(e));
  return LRDS_ERR_CUDA;
}

DeviceLimits device_limits() {
  int dev = 0;
  DeviceLimits l{0, 0};
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&l.smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  cudaDeviceGetAttribute(&l.sms, cudaDevAttrMultiProcessorCount, dev);
  if (l.sms <= 0) l.sms = 148;
  return l;
}

}  // namespace lrds

namespace {
using lrds::cuda_fail;
using lrds::fail;

// the kernel launch just issued: its error as "<what> launch: ...", else n more launches counted
int launched(const char* what, int n = 1) {
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "%s launch", what);
  g_launches.fetch_add(n);
  return LRDS_OK;
}

// threads per CTA for the column layout: as many as fit, preferring >= 2 CTAs per SM
int pick_threads(int floats_per_particle, int smem_cap) {
  const int per = floats_per_particle * (int)sizeof(float);
  if (128 * per <= smem_cap / 2) return 128;
  if (64 * per <= smem_cap / 3) return 64;
  for (int nt = 128; nt >= 32; nt -= 32)
    if (nt * per <= smem_cap) return nt;
  return 0;
}

// Launch of a kernel with one thread per particle and the spec's shared-memory columns (col_layout): `floats` more
// shared-memory floats per thread, `bytes` more per CTA, at most `max_nt` threads per CTA, `slices` CTA rows (grid.y);
// `launches` are counted when the launch succeeds; `layout` >= 0 replaces col_layout(s).total (a kernel with its own
// column layout).
struct ColExtra {
  int max_nt = 128, floats = 0;
  uint32_t bytes = 0;
  int slices = 1, launches = 1, layout = -1;
};
template <class K, class... A>
int launch_cols(K kernel, const char* what, const lrds_spec& s, const ColExtra& x, cudaStream_t st, A... args) {
  const int floats = (x.layout >= 0 ? x.layout : lrds::col_layout(s).total) + x.floats;
  int nt = pick_threads(floats, lrds::device_limits().smem_optin - (int)x.bytes);
  if (nt == 0) return fail(LRDS_ERR_RESOURCES, "per-particle state of %d floats does not fit in shared memory", floats);
  nt = nt < x.max_nt ? nt : x.max_nt;
  const size_t smem = (size_t)floats * nt * sizeof(float) + x.bytes;
  const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute");
  kernel<<<dim3((s.B + nt - 1) / nt, x.slices), nt, smem, st>>>(args...);
  return launched(what, x.launches);
}

int validate_gmm(const lrds_gmm& g, const char* name) {
  if (g.layout == LRDS_GMM_FULL) {  // logc, mu, sn = precision matrices; no ivar / tensor-core image
    if (g.M < 1 || !g.logc || !g.mu || !g.sn) return fail(LRDS_ERR_INVALID, "%s: incomplete full-covariance block", name);
    if (g.mix_tc) return fail(LRDS_ERR_INVALID, "%s: a full-covariance block has no mix_tc image", name);
    return LRDS_OK;
  }
  if (g.layout != LRDS_GMM_DIAG) return fail(LRDS_ERR_INVALID, "%s: unknown lrds_gmm layout", name);
  if (g.M < 1 || !g.logc || !g.mu || !g.ivar || !g.sn) return fail(LRDS_ERR_INVALID, "%s: incomplete mixture block", name);
  return LRDS_OK;
}
// the entry points that evaluate only diagonal blocks
int refuse_full(const lrds_gmm& g, const char* where) {
  if (g.layout == LRDS_GMM_FULL) return fail(LRDS_ERR_UNSUPPORTED, "%s: full-covariance blocks are built for the LINEAR / EUBO_LINEAR "
                                             "reference (ref_t, ref_0) and lrds_distr_eval only", where);
  return LRDS_OK;
}

int validate_spec(const lrds_spec* s, bool need_steps) {
  if (!s) return fail(LRDS_ERR_INVALID, "spec is NULL");
  if (s->abi_version != LRDS_ABI_VERSION) return fail(LRDS_ERR_INVALID, "abi_version mismatch (got %d)", s->abi_version);
  if (s->B < 1 || s->d < 1 || s->K < 0) return fail(LRDS_ERR_INVALID, "B, d must be positive and K non-negative");
  if (s->mlp.d != s->d || s->mlp.d_pad != ((s->d + 7) / 8) * 8) return fail(LRDS_ERR_INVALID, "mlp.d / d_pad inconsistent with d");
  if (!s->mlp.w_in_t || !s->mlp.w_out_t || !s->mlp.b_out || s->mlp.num_hidden < 0 ||
      (s->mlp.num_hidden > 0 && (!s->mlp.w_hid_t || !s->mlp.b_hid)))
    return fail(LRDS_ERR_INVALID, "mlp weight pointers missing");
  if (need_steps && !s->steps) return fail(LRDS_ERR_INVALID, "per-step table missing");
  if (s->ctrl_kind < LRDS_CTRL_CLIPPED || s->ctrl_kind > LRDS_CTRL_LERP) return fail(LRDS_ERR_INVALID, "unknown ctrl_kind");
  if (s->ctrl_kind == LRDS_CTRL_LERP && (s->ref_0.M != 1 || s->ref_0.layout != LRDS_GMM_DIAG || !s->ref_0.mu || !s->ref_0.ivar))
    return fail(LRDS_ERR_INVALID, "LerpCtrl needs the diagonal Gaussian prior in ref_0");
  switch (s->target.kind) {
    case LRDS_DISTR_GMM:
      if (int r = validate_gmm(s->target.gmm, "target")) return r;
      if (int r = refuse_full(s->target.gmm, "target")) return r;
      break;
    case LRDS_DISTR_PHI4:
      break;
    case LRDS_DISTR_LOGREG:
      if (s->target.logreg.p + 1 != s->d || !s->target.logreg.X || !s->target.logreg.Xt || !s->target.logreg.y ||
          s->target.logreg.n_pad % 4 != 0 || s->target.logreg.n_pad < s->target.logreg.N)
        return fail(LRDS_ERR_INVALID, "logistic-regression block inconsistent");
      break;
    case LRDS_DISTR_NONE:
      if (s->ctrl_kind != LRDS_CTRL_CLIPPED) return fail(LRDS_ERR_INVALID, "ScoreCtrl needs a target");
      break;
    default:
      return fail(LRDS_ERR_UNSUPPORTED, "unknown target kind");
  }
  return LRDS_OK;
}

// the fp32 adjoint (lrds_adjoint.cuh): the parity anchor, and every spec outside the tensor-core kernel's envelope
__global__ void __launch_bounds__(128) adjoint_simt_kernel(const lrds::AdjointArgs a) {
  extern __shared__ __align__(16) float smem[];
  lrds::adjoint_body(a, smem);
}
// the fp32 adjoint of the CMCD loop (lrds_adjoint_cmcd.cuh)
__global__ void __launch_bounds__(128) adjoint_cmcd_simt_kernel(const lrds::AdjointArgs a) {
  extern __shared__ __align__(16) float smem[];
  lrds::adjoint_cmcd_body(a, smem);
}

// ---- estimator partials -----------------------------------------------------------------------------
constexpr int EST_THREADS = 256;
constexpr int EST_PER_BLOCK = 8192;

// merge of two partial records (max-shifted sums), associative and commutative
__device__ void merge8(double* acc, const double* p) {
  if (p[5] == 0.0) return;
  if (acc[5] == 0.0) {
    for (int i = 0; i < 8; ++i) acc[i] = p[i];
    return;
  }
  const double m = fmax(acc[0], p[0]);
  const double ea = exp(acc[0] - m), eb = exp(p[0] - m);
  acc[1] = acc[1] * ea + p[1] * eb;
  acc[2] = acc[2] * ea * ea + p[2] * eb * eb;
  acc[0] = m;
  acc[3] += p[3]; acc[4] += p[4]; acc[5] += p[5];
  const double m2 = fmax(acc[6], p[6]);
  acc[7] = acc[7] * exp(acc[6] - m2) + p[7] * exp(p[6] - m2);
  acc[6] = m2;
}

__global__ void __launch_bounds__(EST_THREADS) estimator_kernel(const float* __restrict__ rnd, int B,
                                                                double* __restrict__ out, double* scratch,
                                                                unsigned int* counter) {
  using lrds::block_reduce;
  const lrds::MaxOp mx_op{};
  const lrds::SumOp sum{};
  __shared__ double sh[EST_THREADS / 32];
  __shared__ bool is_last;
  const int lo = blockIdx.x * EST_PER_BLOCK, hi = min(B, lo + EST_PER_BLOCK);
  double mx = -INFINITY, mn = -INFINITY;
  for (int i = lo + threadIdx.x; i < hi; i += EST_THREADS) {
    const double v = (double)rnd[i];
    mx = fmax(mx, -v);
    mn = fmax(mn, v);
  }
  mx = block_reduce(mx, mx_op, -HUGE_VAL, sh);
  mn = block_reduce(mn, mx_op, -HUGE_VAL, sh);
  double s1 = 0, s2 = 0, sr = 0, sr2 = 0, sf = 0;
  for (int i = lo + threadIdx.x; i < hi; i += EST_THREADS) {
    const double v = (double)rnd[i];
    const double e = exp(-v - mx);
    s1 += e; s2 += e * e; sr += v; sr2 += v * v; sf += exp(v - mn);
  }
  s1 = block_reduce(s1, sum, 0.0, sh);
  s2 = block_reduce(s2, sum, 0.0, sh);
  sr = block_reduce(sr, sum, 0.0, sh);
  sr2 = block_reduce(sr2, sum, 0.0, sh);
  sf = block_reduce(sf, sum, 0.0, sh);
  if (threadIdx.x == 0) {
    double* p = scratch + 8 * blockIdx.x;
    p[0] = mx; p[1] = s1; p[2] = s2; p[3] = sr; p[4] = sr2; p[5] = (double)(hi - lo); p[6] = mn; p[7] = sf;
    __threadfence();
    const unsigned int t = atomicAdd(counter, 1u);
    is_last = (t == gridDim.x - 1);
  }
  __syncthreads();
  if (is_last && threadIdx.x == 0) {
    __threadfence();
    double acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (unsigned int k = 0; k < gridDim.x; ++k) merge8(acc, scratch + 8 * k);
    for (int i = 0; i < 8; ++i) out[i] = acc[i];
    *counter = 0u;
  }
}

// merge of n partial records (one per rank, gathered by the caller) on the device: the result stays on the GPU, so the
// multi-GPU estimator needs no host round trip between the collective and whatever consumes the scalars
__global__ void estimator_merge_kernel(const double* __restrict__ parts, int n, double* __restrict__ out) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  double acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (int k = 0; k < n; ++k) merge8(acc, parts + 8 * k);
  for (int i = 0; i < 8; ++i) out[i] = acc[i];
}

// ---- packers of the tensor-core operand images (layouts in include/lrds_b200.h) --------------------------------------
// one block per step
__global__ void __launch_bounds__(256) pack_gmm_mix_kernel(const lrds_gmm g, int d, int d_pad, uint8_t* __restrict__ out) {
  using namespace lrds;
  __shared__ float red[8];
  __shared__ float wbar[LRDS_MAX_DIM_PAD];
  __shared__ double cm[64];
  __shared__ float wn[64];
  const int Mp = (g.M + 15) / 16 * 16, N2 = 2 * d_pad;
  const uint32_t part_bytes = (uint32_t)(Mp / 8) * (uint32_t)N2 * 16u;
  const float* mu = g.mu + (int64_t)blockIdx.x * g.step_stride_param;
  const float* iv = g.ivar + (int64_t)blockIdx.x * g.step_stride_param;
  const float* logc = g.logc + (int64_t)blockIdx.x * g.step_stride_logc;
  uint8_t* o = out + (int64_t)blockIdx.x * lrds::gmm_mix_tc_bytes(g.M, d_pad);
  auto value = [&](int m, int n) -> float {
    if (m >= g.M) return 0.f;
    const int c = n >> 4, i = n & 15, j = 8 * c + (i & 7);
    const float a = iv[(int64_t)m * d_pad + j];
    return i < 8 ? -a : mu[(int64_t)m * d_pad + j] * a;
  };
  float amax = 0.f;
  for (int idx = threadIdx.x; idx < Mp * N2; idx += blockDim.x) amax = fmaxf(amax, fabsf(value(idx / N2, idx % N2)));
  amax = block_reduce(amax, MaxOp{}, 0.f, red);
  const int k = pow2_exponent_for(amax);
  const float sc = ldexpf(1.0f, k);
  for (int idx = threadIdx.x; idx < Mp * N2; idx += blockDim.x) {
    const int m = idx / N2, n = idx % N2;
    put_hi_lo(o, part_bytes, (uint32_t)(m >> 3) * (uint32_t)N2 * 16u + (uint32_t)n * 16u + (uint32_t)(m & 7) * 2u, value(m, n) * sc);
  }
  if (threadIdx.x < 4) reinterpret_cast<float*>(o + 2 * part_bytes)[threadIdx.x] = threadIdx.x == 0 ? ldexpf(1.0f, -k) : 0.f;

  // ---- logit image: rows = modes, K = dims; wc_mj = mu_mj / var_mj - mean over the modes
  uint8_t* ol = o + lrds::gmm_mix_contr_bytes(g.M, d_pad);
  const uint32_t lpart = lrds::gmm_mix_logit_part_bytes(g.M, d_pad);
  const int Kin = (d_pad + 15) / 16 * 16;
  float shared_dev = 0.f;  // largest relative deviation of a mode's 1/var from mode 0's
  for (int j = threadIdx.x; j < d_pad; j += blockDim.x) {
    double acc = 0.0;
    for (int m = 0; m < g.M; ++m) acc += (double)mu[(int64_t)m * d_pad + j] * (double)iv[(int64_t)m * d_pad + j];
    wbar[j] = j < d ? (float)(acc / g.M) : 0.f;
    if (j < d)
      for (int m = 1; m < g.M; ++m)
        shared_dev = fmaxf(shared_dev, fabsf(iv[(int64_t)m * d_pad + j] - iv[j]) / fabsf(iv[j]));
  }
  shared_dev = block_reduce(shared_dev, MaxOp{}, 0.f, red);  // (contains the __syncthreads that publishes wbar)
  auto wc = [&](int m, int j) -> float {
    if (m >= g.M || j >= d) return 0.f;
    return (float)((double)mu[(int64_t)m * d_pad + j] * (double)iv[(int64_t)m * d_pad + j] - (double)wbar[j]);
  };
  float lmax = 0.f;
  for (int idx = threadIdx.x; idx < Mp * Kin; idx += blockDim.x) lmax = fmaxf(lmax, fabsf(wc(idx / Kin, idx % Kin)));
  lmax = block_reduce(lmax, MaxOp{}, 0.f, red);
  const int kl = pow2_exponent_for(lmax);
  const float scl = ldexpf(1.0f, kl);
  for (int idx = threadIdx.x; idx < Mp * Kin; idx += blockDim.x) {
    const int m = idx / Kin, j = idx % Kin;
    put_hi_lo(ol, lpart, (uint32_t)(j >> 3) * (uint32_t)Mp * 16u + (uint32_t)m * 16u + (uint32_t)(j & 7) * 2u, wc(m, j) * scl);
  }
  // c_m = logc_m - sum_j mu^2 / var / 2 and |wc_m|_2, one warp per mode at a time
  for (int m = threadIdx.x >> 5; m < Mp; m += blockDim.x >> 5) {
    double q = 0.0, w2 = 0.0;
    if (m < g.M)
      for (int j = threadIdx.x & 31; j < d; j += 32) {
        const double mm = mu[(int64_t)m * d_pad + j], a = iv[(int64_t)m * d_pad + j];
        q += mm * mm * a;
        const double w = wc(m, j);
        w2 += w * w;
      }
    for (int off = 16; off > 0; off >>= 1) {
      q += __shfl_xor_sync(0xffffffffu, q, off);
      w2 += __shfl_xor_sync(0xffffffffu, w2, off);
    }
    if ((threadIdx.x & 31) == 0) {
      cm[m] = m < g.M ? (double)logc[m] - 0.5 * q : -INFINITY;
      wn[m] = (float)sqrt(w2);
    }
  }
  __syncthreads();
  float* cdst = reinterpret_cast<float*>(ol + 2 * lpart);
  double ctop = -INFINITY;  // softmax-invariant shift: c_m - max_m c_m (the error bound scales with max |c_m|)
  for (int m = 0; m < g.M; ++m) ctop = fmax(ctop, cm[m]);
  for (int m = threadIdx.x; m < Mp; m += blockDim.x) cdst[m] = (float)(cm[m] - ctop);
  if (threadIdx.x == 0) {
    float wnmax = 0.f, cmax = 0.f;
    for (int m = 0; m < g.M; ++m) {
      wnmax = fmaxf(wnmax, wn[m]);
      if (isfinite(cm[m])) cmax = fmaxf(cmax, fabsf((float)(cm[m] - ctop)));
    }
    float* t2 = cdst + Mp;
    t2[0] = ldexpf(1.0f, -kl);
    t2[1] = wnmax;
    t2[2] = cmax;
    t2[3] = shared_dev <= 1e-6f ? 1.0f : 0.f;
  }
}

__global__ void __launch_bounds__(256) pack_logreg_kernel(const lrds_logreg L, int d_pad, uint8_t* __restrict__ out) {
  using namespace lrds;
  __shared__ float red[8];
  const int N16 = (L.N + 15) / 16 * 16, K16 = (L.p + 1 + 15) / 16 * 16;
  const uint32_t part_bytes = (uint32_t)N16 * (uint32_t)K16 * 2u;
  auto value = [&](int n, int k) -> float {
    if (n >= L.N || k > L.p) return 0.f;
    return k == L.p ? 1.0f : L.X[(int64_t)n * d_pad + k];
  };
  float amax = 0.f;
  for (int idx = threadIdx.x; idx < N16 * K16; idx += blockDim.x) amax = fmaxf(amax, fabsf(value(idx / K16, idx % K16)));
  amax = block_reduce(amax, MaxOp{}, 0.f, red);
  const int e = pow2_exponent_for(amax);
  const float sc = ldexpf(1.0f, e);
  for (int idx = threadIdx.x; idx < N16 * K16; idx += blockDim.x) {
    const int n = idx / K16, k = idx % K16;
    put_hi_lo(out, part_bytes, (uint32_t)(k >> 3) * (uint32_t)N16 * 16u + (uint32_t)n * 16u + (uint32_t)(k & 7) * 2u, value(n, k) * sc);
  }
  float* tail = reinterpret_cast<float*>(out + 2 * part_bytes);
  if (threadIdx.x < 4) tail[threadIdx.x] = threadIdx.x == 0 ? ldexpf(1.0f, -e) : 0.f;
  for (int n = threadIdx.x; n < N16; n += blockDim.x) tail[4 + n] = n < L.N ? L.y[n] : 0.f;
}

// ---- evaluation kernels for the small public interfaces -------------------------------------------------
__global__ void __launch_bounds__(128) ctrl_forward_kernel(const lrds_spec s, int rowi, const float* __restrict__ x,
                                                           float* __restrict__ out) {
  using namespace lrds;
  extern __shared__ float smem[];
  const ParticleThread t = particle_thread(s, smem);
  const int b = t.b;
  const bool live = t.live;
  const Particle& P = t.P;
  const GmmView tv0 = gmm_at(s.target.gmm, 0);
  const int NT = blockDim.x;
  SimtMlp mlp{s.mlp, Col{smem + col_layout(s).act * NT + (int)threadIdx.x, NT}};
  const int d = s.d, dp = s.mlp.d_pad;
  for (int j = 0; j < dp; ++j) P.x(j) = (j < d) ? __ldg(x + (int64_t)b * d + j) : 0.f;
  const float* row = s.steps + (int64_t)rowi * LRDS_STEP_STRIDE;
  const bool score_ctrl = s.ctrl_kind != LRDS_CTRL_CLIPPED;
  const CtrlConst cc = ctrl_const(s);
  if (score_ctrl) target_pass1<false>(s, s.target.kind, tv0, P, false);
  mlp.template hidden<false>(row + LRDS_STEP_BIAS1, P.x);
  const int kind = score_ctrl ? s.target.kind : LRDS_DISTR_NONE;  // ClippedCtrl reads no score (NONE: zeros)
  target_score_loop<false>(s, kind, tv0, P, [&](int j0, const float(&xr)[JC], const float(&ts)[JC]) {
    float u[JC];
    if (s.ctrl_kind >= LRDS_CTRL_CANCEL_DRIFT) {
      float ps[JC] = {};
      if (s.ctrl_kind == LRDS_CTRL_LERP) gmm_score_chunk<false, false>(gmm_at(s.ref_0, 0), d, dp, xr, P.rr, j0, ps);
      ctrl_chunk_dis(cc, mlp, j0, ts, xr, ps, ctrl_step(row), u);
    } else {
      ctrl_chunk(cc, mlp, j0, ts, __ldg(row + LRDS_STEP_GAMMA), u);
    }
    if (live)
#pragma unroll
      for (int c = 0; c < JC; ++c)
        if (j0 + c < d) out[(int64_t)b * d + j0 + c] = u[c];
  });
}

__global__ void __launch_bounds__(128) distr_eval_kernel(const lrds_spec s, const float* __restrict__ x,
                                                         float* __restrict__ logp_out, float* __restrict__ score_out) {
  using namespace lrds;
  extern __shared__ float smem[];
  const ParticleThread t = particle_thread(s, smem);
  const int b = t.b;
  const bool live = t.live;
  const Particle& P = t.P;
  const GmmView tv0 = gmm_at(s.target.gmm, 0);
  const int d = s.d, dp = s.mlp.d_pad;
  for (int j = 0; j < dp; ++j) P.x(j) = (j < d) ? __ldg(x + (int64_t)b * d + j) : 0.f;
  if (s.target.kind == LRDS_DISTR_GMM && s.target.gmm.layout == LRDS_GMM_FULL) {  // score column P.rr, scratch P.rh
    const GmmFullView g = gmm_full_at(s.target.gmm, 0);
    const float lp = score_out ? gmm_full_pass<true>(g, d, dp, P.x, P.rr, P.rh) : gmm_full_pass<false>(g, d, dp, P.x, P.rr, P.rh);
    if (live && logp_out) logp_out[b] = lp + s.rnd_offset;
    if (live && score_out)
      for (int j = 0; j < d; ++j) score_out[(int64_t)b * d + j] = P.rr(j);
    return;
  }
  const float lp = target_pass1<false>(s, s.target.kind, tv0, P, logp_out != nullptr);
  if (live && logp_out) logp_out[b] = lp + s.rnd_offset;
  if (!score_out) return;
  float xm = 0.f;  // target_score_loop written out: through the helper this kernel's register allocation changes
  for (int j0 = 0; j0 < dp; j0 += JC) {
    float xr[JC], ts[JC];
    load_chunk(P.x, j0, xr);
    const float xp = (j0 + JC < dp) ? P.x(j0 + JC) : 0.f;
    target_score_chunk<false>(s, s.target.kind, tv0, P, xr, xm, xp, j0, ts);
    xm = xr[JC - 1];
    if (live)
#pragma unroll
      for (int c = 0; c < JC; ++c)
        if (j0 + c < d) score_out[(int64_t)b * d + j0 + c] = ts[c];
  }
}

// ---- sum_b w_sb cot_sb (x) clip(score(x_sb)) per time slice s: the cotangent of the time-only factor of ScoreCtrl
// (models/reparam.py:112-117: ctrl = clip(net) + scale * clip(score) * clip(TimeEmbed_score(t))) in the batched gradient
// pass of train.py.  One thread per stored state; the products replace the staged cotangents in shared memory and the
// block's columns are summed from there; every block writes its partial row (part[s][block][dp]) and score_cot_reduce_kernel adds them in a fixed order.
// bytes of a mixture target staged in shared memory behind the particle columns (0: read from global memory)
inline uint32_t score_cot_stage_bytes(const lrds_spec& s) { return lrds::stage_layout(s, 2).tgt_bytes; }

template <bool SH>
__device__ __forceinline__ void score_cot_body(const lrds_spec& s, const lrds::GmmViewT<SH>& tv, const lrds::Particle& P,
                                               float* __restrict__ rows, int ld, float w, float clip,
                                               float* __restrict__ dst) {
  using namespace lrds;
  const int tid = threadIdx.x, NT = blockDim.x;
  const int d = s.d, dp = s.mlp.d_pad;
  float* mine = rows + tid * ld;  // this thread's row of the staged cotangents; the products replace them in place
  if (SH && s.target.kind == LRDS_DISTR_GMM && s.target.gmm.M <= MIX_MAX_M) {
    // the responsibilities with every (1/sigma, -mu/sigma) vector serving two particles (lrds_rollout_simt.cuh): this
    // kernel is bound by the shared-memory data pipe, not by the FMA pipe
    float r[MIX_MAX_M];
    gmm_pass1_pair(tv, d, dp, P.x, r);
    const int M4 = (s.target.gmm.M + 3) / 4;
#pragma unroll
    for (int mb = 0; mb < MIX_MAX_M / 4; ++mb)
      if (mb < M4) P.rt.st4(mb, make_float4(r[4 * mb], r[4 * mb + 1], r[4 * mb + 2], r[4 * mb + 3]));
  } else {
    target_pass1<SH>(s, s.target.kind, tv, P, false);
  }
  float xm = 0.f;  // target_score_loop written out (particle_thread too): through the helpers this kernel runs longer code
  for (int j0 = 0; j0 < dp; j0 += JC) {
    float xr[JC], ts[JC];
    load_chunk(P.x, j0, xr);
    const float xp = (j0 + JC < dp) ? P.x(j0 + JC) : 0.f;
    target_score_chunk<SH>(s, s.target.kind, tv, P, xr, xm, xp, j0, ts);
    xm = xr[JC - 1];
#pragma unroll
    for (int c = 0; c < JC; ++c) {
      if (j0 + c < d) {
        float v = ts[c];
        if (clip > 0.f) v = fminf(fmaxf(v, -clip), clip);
        mine[j0 + c] = v * mine[j0 + c] * w;
      }
    }
  }
  __syncthreads();
  for (int j = tid; j < d; j += NT) {  // column sums over the block's rows, in row order
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;  // four chains (NT is a multiple of 32)
    for (int p = 0; p < NT; p += 4) {
      a0 += rows[p * ld + j];
      a1 += rows[(p + 1) * ld + j];
      a2 += rows[(p + 2) * ld + j];
      a3 += rows[(p + 3) * ld + j];
    }
    dst[j] = (a0 + a1) + (a2 + a3);
  }
}

__global__ void __launch_bounds__(128) score_cot_kernel(const lrds_spec s, const float* __restrict__ x,
                                                        const float* __restrict__ cot, const float* __restrict__ step_w,
                                                        const float* __restrict__ row_w, const float clip,
                                                        float* __restrict__ part) {
  using namespace lrds;
  extern __shared__ __align__(16) float smem[];
  const int NT = blockDim.x, tid = threadIdx.x;
  const int slice = blockIdx.y;
  const int b_raw = blockIdx.x * NT + tid;
  const bool live = b_raw < s.B;
  const int b = live ? b_raw : s.B - 1;
  const ColLayout L = col_layout(s);
  const Particle P = make_particle(smem, L, NT, tid);
  const GmmView tv0 = gmm_at(s.target.gmm, 0);
  const int d = s.d, dp = s.mlp.d_pad;
  const int warp = tid >> 5, lane = tid & 31, nw = NT >> 5;
  const StageLayout SL = stage_layout(s, 2);
  const uint32_t stage_bytes = SL.tgt_bytes, logc_bytes = SL.tgt_logc_bytes;
  // The block's rows are contiguous in global memory: the warps read them row by row (coalesced) into a padded
  // row-major staging area and every thread then takes its own row from there (per-thread global reads of rows
  // 4 d bytes apart cost 32 wavefronts per load).
  float* rows = smem + (size_t)L.total * NT + stage_bytes / 4u;  // [NT][d + 1]
  const int ld = d + 1;
  auto stage_rows = [&](const float* __restrict__ src) {
    for (int p0 = warp; p0 < NT; p0 += 8 * nw) {  // eight rows in flight per warp
      float va[8], vb[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int p = p0 + i * nw;
        const int bp = min(blockIdx.x * NT + (p < NT ? p : 0), s.B - 1);
        const float* g = src + ((int64_t)slice * s.B + bp) * d;
        va[i] = lane < d ? __ldg(g + lane) : 0.f;
        vb[i] = lane + 32 < d ? __ldg(g + lane + 32) : 0.f;
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int p = p0 + i * nw;
        if (p < NT) {
          if (lane < d) rows[p * ld + lane] = va[i];
          if (lane + 32 < d) rows[p * ld + lane + 32] = vb[i];
        }
      }
      for (int j = lane + 64; j < d; j += 32)  // d > 64: the rest of the eight rows
        for (int i = 0; i < 8; ++i) {
          const int p = p0 + i * nw;
          if (p < NT) rows[p * ld + j] = __ldg(src + ((int64_t)slice * s.B + min(blockIdx.x * NT + p, s.B - 1)) * d + j);
        }
    }
  };
  stage_rows(x);
  __syncthreads();
  for (int j = 0; j < dp; ++j) P.x(j) = (j < d) ? rows[tid * ld + j] : 0.f;
  __syncthreads();
  stage_rows(cot);
  float w = live ? 1.f : 0.f;
  if (step_w) w *= __ldg(step_w + slice);
  if (row_w) w *= __ldg(row_w + b);
  float* dst = part + ((int64_t)slice * gridDim.x + blockIdx.x) * dp;
  if (stage_bytes) {  // mixture target: its (logc, sn) blocks go to shared memory once per block
    float4* stg = reinterpret_cast<float4*>(smem + (size_t)L.total * NT);
    const float4* g_logc = reinterpret_cast<const float4*>(tv0.logc.p);
    const float4* g_sn = reinterpret_cast<const float4*>(tv0.sn.p);
    const int n_logc = (int)(logc_bytes / 16u), n_all = (int)(stage_bytes / 16u);
    for (int i = tid; i < n_all; i += NT) stg[i] = i < n_logc ? __ldg(g_logc + i) : __ldg(g_sn + (i - n_logc));
    __syncthreads();
    const GmmViewT<true> tv = staged_view(reinterpret_cast<const uint8_t*>(stg), tv0, logc_bytes, stage_bytes - logc_bytes);
    score_cot_body<true>(s, tv, P, rows, ld, w, clip, dst);
  } else {
    __syncthreads();
    score_cot_body<false>(s, tv0, P, rows, ld, w, clip, dst);
  }
}

__global__ void score_cot_reduce_kernel(const float* __restrict__ part, int nblk, int dp, int d, float* __restrict__ out) {
  const int slice = blockIdx.x, j = threadIdx.x;
  if (j >= d) return;
  const float* src = part + (int64_t)slice * nblk * dp + j;
  float acc = 0.f;
  for (int i = 0; i < nblk; ++i) acc += src[(int64_t)i * dp];
  out[(int64_t)slice * d + j] = acc;
}

// ---- MALA chains: the whole loop of mcmc_sample(mcmc_type='mala') (experiments/benchmark_utils.py:268-333) around
// mala_step and heuristics_step_size (sde_sampler/additions/mcmc.py:75-134, 54-72) in one launch, one thread per chain.
// Columns: x = proposal, us = current state, tsd = score at the current state, db = score at the proposal.
struct MalaArgs {
  const float* y0;      // [C][d]
  float* step_size;     // [C] in / out
  const float* noise;   // [S][C][d] standard normals or NULL (Philox stream 0)
  const float* unif;    // [S][C] uniforms in (0, 1] or NULL (Philox stream 2)
  uint64_t seed;
  float* ys;            // [n_steps][C][d] states after the warm-up
  float* log_acc;       // [S][C] or NULL
  int n_warmup, n_steps, adapt, sampler;
  float log_target, up_thr, down_thr, factor;  // log(0.75), log1p(tol), -log1p(-tol), 1.01
};

__global__ void __launch_bounds__(128) mala_kernel(const lrds_spec s, const MalaArgs m) {
  using namespace lrds;
  extern __shared__ float smem[];
  const ParticleThread t = particle_thread(s, smem);
  const int b = t.b;
  const bool live = t.live;
  const Particle& P = t.P;
  const GmmView tv0 = gmm_at(s.target.gmm, 0);
  const int d = s.d, dp = s.mlp.d_pad, kind = s.target.kind;
  const RolloutArgs na{s, nullptr, m.noise, m.seed, 0, nullptr, nullptr, nullptr};
  // log-density and score at P.x; the score goes to column `out`
  auto eval = [&](const Col& out) -> float {
    const float lp = target_pass1<false>(s, kind, tv0, P, true);
    target_score_loop<false>(s, kind, tv0, P, [&](int j0, const float(&)[JC], const float(&ts)[JC]) {
#pragma unroll
      for (int c = 0; c < JC; ++c) out(j0 + c) = (j0 + c < d) ? ts[c] : 0.f;
    });
    return lp;
  };
  for (int j = 0; j < dp; ++j) {
    const float v = (j < d) ? __ldg(m.y0 + (int64_t)b * d + j) : 0.f;
    P.x(j) = v;
    P.us(j) = v;
  }
  const bool rwmh = m.sampler == LRDS_MCMC_RWMH;
  float logp = rwmh ? target_pass1<false>(s, kind, tv0, P, true) : eval(P.tsd);
  float h = __ldg(m.step_size + b);
  const int S = m.n_warmup + m.n_steps;
  for (int step = 0; step < S; ++step) {
    // proposal: MALA y' = sqrt(2 h) z + (y + h grad) (mcmc.py:8-14, 98-102);  RWMH y' = y + h z (mcmc.py:275-277)
    const float var = 2.0f * h, sq = sqrtf(var);
    float fwd = 0.f;
    for (int j0 = 0; j0 < dp; j0 += JC) {
      float z[JC];
      noise_chunk(na, step, b, j0, z);
#pragma unroll
      for (int c = 0; c < JC; ++c) {
        const int j = j0 + c;
        if (rwmh) {
          P.x(j) = (j < d) ? P.us(j) + h * z[c] : 0.f;
        } else {
          const float mean = P.us(j) + h * P.tsd(j);
          const float yp = (j < d) ? sq * z[c] + mean : 0.f;
          P.x(j) = yp;
          const float df = yp - mean;
          fwd += df * df;
        }
      }
    }
    float logp_p, log_acc;
    if (rwmh) {  // the Metropolis ratio of a symmetric proposal (mcmc.py:279-281); no score
      logp_p = target_pass1<false>(s, kind, tv0, P, true);
      log_acc = logp_p - logp;
    } else {
      logp_p = eval(P.db);
      float bwd = 0.f;
      for (int j = 0; j < d; ++j) {
        const float df = P.us(j) - (P.x(j) + h * P.db(j));
        bwd += df * df;
      }
      // joint_prop - joint_orig with the unnormalised Gaussian log-densities of mcmc.py:17-31
      log_acc = (logp_p - (-0.5f * fwd) / var) - (logp - (-0.5f * bwd) / var);
    }
    float u;
    if (m.unif != nullptr) {
      u = __ldg(m.unif + (int64_t)step * s.B + b);
    } else {
      uint32_t r[4];
      philox4x32_10((uint32_t)b, (uint32_t)step, 0u, 2u, (uint32_t)m.seed, (uint32_t)(m.seed >> 32), r);
      u = (float)((r[0] >> 8) + 1u) * 5.9604644775390625e-08f;
    }
    if (logf(u) < log_acc) {  // mcmc.py:121-124
      for (int j = 0; j < dp; ++j) {
        P.us(j) = P.x(j);
        P.tsd(j) = P.db(j);
      }
      logp = logp_p;
    }
    if (m.adapt) {  // heuristics_step_size, mcmc.py:54-72 (both tests read the same log_acc)
      const float h0 = h;
      if (log_acc - m.log_target > m.up_thr) h = h0 * m.factor;
      if (m.log_target - log_acc > m.down_thr) h = h / m.factor;
    }
    if (live && m.log_acc != nullptr) m.log_acc[(int64_t)step * s.B + b] = log_acc;
    if (live && step >= m.n_warmup) {
      float* out = m.ys + ((int64_t)(step - m.n_warmup) * s.B + b) * d;
      for (int j = 0; j < d; ++j) out[j] = P.us(j);
    }
  }
  if (live) m.step_size[b] = h;
}

__global__ void axpy_step_kernel(const float* __restrict__ x, const float* __restrict__ s, const float* __restrict__ z,
                                 float a, float b, float c, float* __restrict__ out, int64_t n) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    float v = a * x[i];
    if (s) v += b * s[i];
    if (z) v += c * z[i];
    out[i] = v;
  }
}

__global__ void normals_kernel(uint64_t seed, uint64_t offset, int stream_id, int K, int B, int d, float* __restrict__ out) {
  const int nblk = (d + 3) / 4;
  const int64_t total = (int64_t)K * B * nblk;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    const int blk = (int)(i % nblk);
    const int b = (int)((i / nblk) % B);
    const int k = (int)(i / ((int64_t)nblk * B));
    float z[4];
    lrds::normals4(seed, (uint32_t)(offset + (uint64_t)b), (uint32_t)k, (uint32_t)blk, (uint32_t)stream_id, z);
    float* p = out + ((int64_t)k * B + b) * d + 4 * blk;
    for (int c = 0; c < 4; ++c)
      if (4 * blk + c < d) p[c] = z[c];
  }
}

// Spec of a bare distribution evaluation (lrds_distr_eval, lrds_score_cot_sums, lrds_mala); `who` names the entry
// point in the messages; full-covariance mixtures are evaluated by lrds_distr_eval only (full_ok).  The caller sets the
// spec kind / precision that select its column layout.
int distr_spec(const lrds_distr* distr, int32_t d, int32_t B, const char* who, bool full_ok, lrds_spec* out) {
  lrds_spec& s = *out;
  memset(&s, 0, sizeof(s));
  s.abi_version = LRDS_ABI_VERSION;
  s.B = B;
  s.d = d;
  s.mlp.d = d;
  s.mlp.d_pad = ((d + 7) / 8) * 8;
  s.target = *distr;
  s.ctrl_kind = LRDS_CTRL_CLIPPED;
  if (distr->kind == LRDS_DISTR_GMM) {
    if (int r = validate_gmm(distr->gmm, who)) return r;
    if (!full_ok)
      if (int r = refuse_full(distr->gmm, who)) return r;
  } else if (distr->kind == LRDS_DISTR_LOGREG) {
    if (distr->logreg.p + 1 != d) return fail(LRDS_ERR_INVALID, "%s: logreg: d must be p + 1", who);
  } else if (distr->kind != LRDS_DISTR_PHI4) {
    return fail(LRDS_ERR_UNSUPPORTED, "%s: unknown distribution kind", who);
  }
  return LRDS_OK;
}

// shared by lrds_distr_eval and the initial-cost pre-pass of lrds_rollout: logp_out = log-density + offset
int distr_eval_launch(const lrds_distr* distr, int32_t d, const float* x, int32_t B, float* logp_out, float* score_out,
                      float offset, cudaStream_t st) {
  if (!distr || !x || B < 1 || d < 1 || (!logp_out && !score_out)) return fail(LRDS_ERR_INVALID, "distr_eval: bad arguments");
  lrds_spec s;
  if (int r = distr_spec(distr, d, B, "distr_eval", true, &s)) return r;
  s.rnd_offset = offset;
  return launch_cols(distr_eval_kernel, "distr_eval", s, {}, st, s, x, logp_out, score_out);
}

int score_cot_spec(const lrds_distr* distr, int32_t d, int32_t B, lrds_spec* s) {
  if (int r = distr_spec(distr, d, B, "score_cot_sums", false, s)) return r;
  s->precision = LRDS_PRECISION_F16X3;  // column layout without the fp32 network's activation columns (no network here)
  return LRDS_OK;
}

int score_cot_threads(const lrds_spec& s) {  // the columns + one padded row of the staging area per thread
  return pick_threads(lrds::col_layout(s).total + s.d + 1, lrds::device_limits().smem_optin - (int)score_cot_stage_bytes(s));
}

}  // namespace

extern "C" {

int64_t lrds_score_cot_scratch_floats(const lrds_distr* distr, int32_t d, int32_t S, int32_t B) {
  lrds_spec s;
  if (!distr || d < 1 || S < 1 || B < 1) return fail(LRDS_ERR_INVALID, "score_cot_sums: bad arguments");
  if (int r = score_cot_spec(distr, d, B, &s)) return r;
  const int nt = score_cot_threads(s);
  if (nt == 0) return fail(LRDS_ERR_RESOURCES, "score_cot_sums: per-particle state does not fit in shared memory");
  return (int64_t)S * ((B + nt - 1) / nt) * s.mlp.d_pad;
}

int lrds_score_cot_sums(const lrds_distr* distr, int32_t d, const float* x, const float* cot, const float* step_w,
                        const float* row_w, float clip, int32_t S, int32_t B, float* out, float* scratch, void* stream) {
  if (!distr || !x || !cot || !out || !scratch || d < 1 || S < 1 || B < 1)
    return fail(LRDS_ERR_INVALID, "score_cot_sums: bad arguments");
  if (S > 65535) return fail(LRDS_ERR_UNSUPPORTED, "score_cot_sums: at most 65535 time slices per call");
  lrds_spec s;
  if (int r = score_cot_spec(distr, d, B, &s)) return r;
  cudaStream_t st = (cudaStream_t)stream;
  const int nt = score_cot_threads(s);
  if (nt == 0) return fail(LRDS_ERR_RESOURCES, "score_cot_sums: per-particle state does not fit in shared memory");
  // both kernels are counted once the second is issued
  const ColExtra rows{128, d + 1, score_cot_stage_bytes(s), S, 0};
  if (int r = launch_cols(score_cot_kernel, "score_cot_sums", s, rows, st, s, x, cot, step_w, row_w, clip, scratch)) return r;
  score_cot_reduce_kernel<<<S, ((d + 31) / 32) * 32, 0, st>>>(scratch, (B + nt - 1) / nt, s.mlp.d_pad, d, out);
  return launched("score_cot_sums", 2);
}

const char* lrds_last_error(void) { return g_err; }
int lrds_abi_version(void) { return LRDS_ABI_VERSION; }
int64_t lrds_launch_count(void) { return g_launches.load(); }

int lrds_rollout(const lrds_spec* spec, const float* x0, const float* noise, uint64_t seed, uint64_t particle_offset,
                 float* x_out, float* rnd_out, float* traj_out, void* stream) {
  if (int r = validate_spec(spec, true)) return r;
  if (!x0 || !rnd_out) return fail(LRDS_ERR_INVALID, "x0 and rnd_out are required");
  const lrds_spec& s = *spec;
  if (s.K < 1) return fail(LRDS_ERR_INVALID, "K must be >= 1");
  if (int r = validate_gmm(s.ref_0, "ref_0")) return r;
  const bool linear = s.kind == LRDS_ROLLOUT_LINEAR || s.kind == LRDS_ROLLOUT_EUBO_LINEAR;
  if (s.kind == LRDS_ROLLOUT_EUBO_LINEAR && !s.has_ref_ctrl && !s.init_cost)
    return fail(LRDS_ERR_INVALID, "compute_eubo needs a reference control (or init_cost: the discrete-time DIS loss)");
  if (s.ctrl_kind >= LRDS_CTRL_CANCEL_DRIFT && s.kind != LRDS_ROLLOUT_LINEAR)
    return fail(LRDS_ERR_UNSUPPORTED, "CancelDriftCtrl / LerpCtrl are built for the LINEAR simulate loop (DIS) only");
  if (linear && s.has_ref_ctrl)
    if (int r = validate_gmm(s.ref_t, "ref_t")) return r;
  if (!linear && (s.ref_0.M != 1 || s.ref_0.layout != LRDS_GMM_DIAG))
    return fail(LRDS_ERR_UNSUPPORTED, "CMCD needs a diagonal Gaussian prior");
  if (s.init_cost)
    if (int r = refuse_full(s.ref_0, "the DIS prior (init_cost)")) return r;
  if (!linear && s.target.kind == LRDS_DISTR_NONE) return fail(LRDS_ERR_INVALID, "CMCD needs a target");
  cudaStream_t st = (cudaStream_t)stream;
  lrds::RolloutArgs a{s, x0, noise, seed, particle_offset, x_out, rnd_out, traj_out};
  if (s.init_cost && !linear) return fail(LRDS_ERR_INVALID, "init_cost is defined for the LINEAR loops only");
  if (s.init_cost && s.kind == LRDS_ROLLOUT_EUBO_LINEAR && (s.has_ref_ctrl || s.update_form != LRDS_UPDATE_AXPY))
    return fail(LRDS_ERR_UNSUPPORTED, "init_cost compute_eubo is the discrete-time DIS loss: no reference control, axpy update");
  if (s.init_cost && s.kind == LRDS_ROLLOUT_LINEAR) {  // DIS (oc.py:929, 1164-1168): rnd_out = initial_log_prob(x_0) + rnd_offset
    lrds_distr prior;
    memset(&prior, 0, sizeof(prior));
    prior.kind = LRDS_DISTR_GMM;
    prior.gmm = s.ref_0;
    if (int r = distr_eval_launch(&prior, s.d, x0, s.B, rnd_out, nullptr, s.rnd_offset, st)) return r;
  }

  if (s.precision != LRDS_PRECISION_FP32_SIMT) {
    const int r = lrds::launch_rollout_tc(a, st);
    if (r == LRDS_OK) g_launches.fetch_add(1);
    return r;
  }

  using lrds::rollout_simt_kernel;
  switch (s.kind) {
    case LRDS_ROLLOUT_LINEAR: return launch_cols(rollout_simt_kernel<LRDS_ROLLOUT_LINEAR>, "rollout", s, {}, st, a);
    case LRDS_ROLLOUT_CMCD: return launch_cols(rollout_simt_kernel<LRDS_ROLLOUT_CMCD>, "rollout", s, {}, st, a);
    case LRDS_ROLLOUT_EUBO_LINEAR: return launch_cols(rollout_simt_kernel<LRDS_ROLLOUT_EUBO_LINEAR>, "rollout", s, {}, st, a);
    case LRDS_ROLLOUT_EUBO_CMCD: return launch_cols(rollout_simt_kernel<LRDS_ROLLOUT_EUBO_CMCD>, "rollout", s, {}, st, a);
    default: return fail(LRDS_ERR_INVALID, "unknown rollout kind");
  }
}

int lrds_adjoint(const lrds_spec* spec, const float* traj, const float* noise, uint64_t seed, uint64_t particle_offset,
                 const float* row_w, float* cot_out, void* stream) {
  if (int r = validate_spec(spec, true)) return r;
  if (!traj || !row_w || !cot_out) return fail(LRDS_ERR_INVALID, "adjoint: traj, row_w and cot_out are required");
  const lrds_spec& s = *spec;
  if (s.K < 1) return fail(LRDS_ERR_INVALID, "adjoint: K must be >= 1");
  if (s.kind != LRDS_ROLLOUT_LINEAR)
    return fail(LRDS_ERR_UNSUPPORTED, "adjoint: built for the LINEAR simulate loop (CMCD evaluates the control at both ends of a "
                                      "step: lrds_adjoint_cmcd; the EUBO kinds are not trained through it)");
  if (s.ctrl_kind != LRDS_CTRL_CLIPPED)
    return fail(LRDS_ERR_UNSUPPORTED, "adjoint: built for ClippedCtrl; the score-family controls also need the target's "
                                      "Hessian-vector product");
  if (s.precision == LRDS_PRECISION_BF16 || s.precision == LRDS_PRECISION_TF32)
    return fail(LRDS_ERR_UNSUPPORTED, "adjoint: the reduced-precision network moved the particles, the adjoint would linearise a "
                                      "different one (use f16x3, tf32x3 or fp32)");
  if (s.precision != LRDS_PRECISION_FP32_SIMT && s.precision != LRDS_PRECISION_TF32X3 && s.precision != LRDS_PRECISION_F16X3)
    return fail(LRDS_ERR_INVALID, "adjoint: unknown precision");
  if (int r = validate_gmm(s.ref_0, "ref_0")) return r;
  if (s.has_ref_ctrl)
    if (int r = validate_gmm(s.ref_t, "ref_t")) return r;
  if (lrds::ref_t_full(s) || s.ref_0.layout == LRDS_GMM_FULL)
    return fail(LRDS_ERR_UNSUPPORTED, "adjoint: built for diagonal references (full-covariance ref_t / ref_0 are not)");
  const lrds::AdjointArgs a{lrds::RolloutArgs{s, nullptr, noise, seed, particle_offset, nullptr, nullptr, nullptr}, traj, row_w,
                            cot_out};
  if (lrds::adjoint_tc_applicable(s)) {
    const int r = lrds::launch_adjoint_tc(a, (cudaStream_t)stream);
    if (r == LRDS_OK) g_launches.fetch_add(1);
    return r;
  }
  ColExtra cols;
  cols.layout = lrds::adj_layout(s).total;
  return launch_cols(adjoint_simt_kernel, "adjoint", s, cols, (cudaStream_t)stream, a);
}

int lrds_adjoint_cmcd(const lrds_spec* spec, const float* traj, const float* noise, uint64_t seed, uint64_t particle_offset,
                      const float* row_w, float* cot_out, void* stream) {
  if (int r = validate_spec(spec, true)) return r;
  if (!traj || !row_w || !cot_out) return fail(LRDS_ERR_INVALID, "adjoint_cmcd: traj, row_w and cot_out are required");
  const lrds_spec& s = *spec;
  if (s.K < 1) return fail(LRDS_ERR_INVALID, "adjoint_cmcd: K must be >= 1");
  if (s.kind != LRDS_ROLLOUT_CMCD)
    return fail(LRDS_ERR_UNSUPPORTED, "adjoint_cmcd: built for the CMCD simulate loop (LINEAR: lrds_adjoint; the EUBO kinds are "
                                      "not trained through it)");
  if (s.ctrl_kind != LRDS_CTRL_CLIPPED)
    return fail(LRDS_ERR_UNSUPPORTED, "adjoint_cmcd: built for ClippedCtrl; the score-family controls also need the Hessian-vector "
                                      "product inside the control");
  if (s.precision == LRDS_PRECISION_BF16 || s.precision == LRDS_PRECISION_TF32)
    return fail(LRDS_ERR_UNSUPPORTED, "adjoint_cmcd: the reduced-precision network moved the particles, the adjoint would "
                                      "linearise a different one (use f16x3, tf32x3 or fp32)");
  if (s.precision != LRDS_PRECISION_FP32_SIMT && s.precision != LRDS_PRECISION_TF32X3 && s.precision != LRDS_PRECISION_F16X3)
    return fail(LRDS_ERR_INVALID, "adjoint_cmcd: unknown precision");
  if (s.target.kind == LRDS_DISTR_NONE) return fail(LRDS_ERR_INVALID, "adjoint_cmcd: CMCD needs a target");
  if (s.target.kind != LRDS_DISTR_GMM && s.target.kind != LRDS_DISTR_PHI4)
    return fail(LRDS_ERR_UNSUPPORTED, "adjoint_cmcd: built for mixture and PhiFour targets (the logistic-regression target has "
                                      "no Hessian-vector product here)");
  if (int r = validate_gmm(s.ref_0, "ref_0")) return r;
  if (s.ref_0.layout == LRDS_GMM_FULL || s.ref_0.M != 1)
    return fail(LRDS_ERR_UNSUPPORTED, "adjoint_cmcd: built for a diagonal Gaussian prior in ref_0 (full-covariance priors are not)");
  const lrds::AdjointArgs a{lrds::RolloutArgs{s, nullptr, noise, seed, particle_offset, nullptr, nullptr, nullptr}, traj, row_w,
                            cot_out};
  if (lrds::adjoint_cmcd_tc_applicable(s)) {
    const int r = lrds::launch_adjoint_cmcd_tc(a, (cudaStream_t)stream);
    if (r == LRDS_OK) g_launches.fetch_add(1);
    return r;
  }
  ColExtra cols;
  cols.layout = lrds::adj_cmcd_layout(s).total;
  return launch_cols(adjoint_cmcd_simt_kernel, "adjoint_cmcd", s, cols, (cudaStream_t)stream, a);
}

int64_t lrds_tc_image_bytes(int32_t d, int32_t num_hidden, int32_t precision) {
  if (d < 1 || num_hidden < 0 || precision == LRDS_PRECISION_FP32_SIMT || precision < 0 || precision > LRDS_PRECISION_F16X3)
    return fail(LRDS_ERR_INVALID, "tc_image_bytes: bad arguments");
  return (int64_t)lrds::tc_image_bytes(d, num_hidden, precision);
}

int64_t lrds_gmm_mix_tc_bytes(int32_t M, int32_t d_pad) {
  if (M < 2 || d_pad < 8 || d_pad % 8 != 0) return fail(LRDS_ERR_INVALID, "gmm_mix_tc_bytes: bad arguments");
  return (int64_t)lrds::gmm_mix_tc_bytes(M, d_pad);
}

int lrds_pack_gmm_mix_tc(const lrds_gmm* gmm, int32_t d, int32_t d_pad, int32_t steps, void* image_out, void* stream) {
  if (gmm && gmm->layout != LRDS_GMM_DIAG) return fail(LRDS_ERR_UNSUPPORTED, "pack_gmm_mix_tc: diagonal blocks only");
  if (!gmm || !image_out || !gmm->mu || !gmm->ivar || !gmm->logc || gmm->M < 2 || gmm->M > 64 || d < 1 || d > d_pad || d_pad < 8 ||
      d_pad % 8 != 0 || d_pad > LRDS_MAX_DIM_PAD || steps < 1)
    return fail(LRDS_ERR_INVALID, "pack_gmm_mix_tc: bad arguments");
  pack_gmm_mix_kernel<<<steps, 256, 0, (cudaStream_t)stream>>>(*gmm, d, d_pad, static_cast<uint8_t*>(image_out));
  return launched("pack_gmm_mix_tc");
}

int64_t lrds_logreg_tc_bytes(int32_t N, int32_t p) {
  if (N < 1 || p < 1) return fail(LRDS_ERR_INVALID, "logreg_tc_bytes: bad arguments");
  const int64_t N16 = (N + 15) / 16 * 16, K16 = (p + 1 + 15) / 16 * 16;
  return 4 * N16 * K16 + 16 + 4 * N16;
}

int lrds_pack_logreg_tc(const lrds_logreg* logreg, int32_t d_pad, void* image_out, void* stream) {
  if (!logreg || !image_out || !logreg->X || !logreg->y || logreg->N < 1 || logreg->p < 1 || d_pad < logreg->p + 1)
    return fail(LRDS_ERR_INVALID, "pack_logreg_tc: bad arguments");
  pack_logreg_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(*logreg, d_pad, static_cast<uint8_t*>(image_out));
  return launched("pack_logreg_tc");
}

int lrds_pack_mlp_tc(const lrds_mlp* mlp, int32_t precision, void* image_out, void* stream) {
  if (!mlp || !image_out || !mlp->w_in_t || !mlp->w_out_t || !mlp->b_out || mlp->d < 1 ||
      mlp->d_pad != ((mlp->d + 7) / 8) * 8 || (mlp->num_hidden > 0 && (!mlp->w_hid_t || !mlp->b_hid)))
    return fail(LRDS_ERR_INVALID, "pack_mlp_tc: incomplete mlp block");
  if (precision != LRDS_PRECISION_TF32X3 && precision != LRDS_PRECISION_BF16 && precision != LRDS_PRECISION_TF32 &&
      precision != LRDS_PRECISION_F16X3)
    return fail(LRDS_ERR_INVALID, "pack_mlp_tc: not a tensor-core precision");
  const int r = lrds::pack_tc_image(*mlp, precision, image_out, (cudaStream_t)stream);
  if (r == LRDS_OK) g_launches.fetch_add(1);  // one, also for the two kernels of F16X3
  return r;
}

int lrds_estimator_blocks(int32_t B) { return B < 1 ? 0 : (B + EST_PER_BLOCK - 1) / EST_PER_BLOCK; }

int lrds_estimator_partials(const float* rnd, int32_t B, double* partials, double* scratch, void* stream) {
  if (!rnd || !partials || !scratch || B < 1) return fail(LRDS_ERR_INVALID, "estimator: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  const int blocks = lrds_estimator_blocks(B);
  unsigned int* counter = reinterpret_cast<unsigned int*>(scratch + 8 * (size_t)blocks);
  cudaError_t e = cudaMemsetAsync(counter, 0, sizeof(double), st);
  if (e != cudaSuccess) return cuda_fail(e, "estimator memset");
  estimator_kernel<<<blocks, EST_THREADS, 0, st>>>(rnd, B, partials, scratch, counter);
  return launched("estimator");
}

int lrds_estimator_merge(const double* parts, int32_t n, double* out, void* stream) {
  if (!parts || !out || n < 1) return fail(LRDS_ERR_INVALID, "estimator_merge: bad arguments");
  estimator_merge_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(parts, n, out);
  return launched("estimator_merge");
}

int lrds_ctrl_forward(const lrds_spec* spec, int32_t row, const float* x, int32_t B, float* u_out, void* stream) {
  if (int r = validate_spec(spec, true)) return r;
  if (!x || !u_out || B < 1 || row < 0) return fail(LRDS_ERR_INVALID, "ctrl_forward: bad arguments");
  lrds_spec s = *spec;
  s.B = B;
  s.kind = LRDS_ROLLOUT_LINEAR;
  s.precision = LRDS_PRECISION_FP32_SIMT;  // this entry point evaluates the network with fp32 FFMA
  s.has_ref_ctrl = 0;
  if (s.ctrl_kind != LRDS_CTRL_LERP) s.ref_0.M = 0;  // LerpCtrl reads the prior from ref_0
  return launch_cols(ctrl_forward_kernel, "ctrl_forward", s, {}, (cudaStream_t)stream, s, row, x, u_out);
}

int64_t lrds_mlp_grad_floats(int32_t d, int32_t num_hidden) {
  return lrds::mlp_grad_applicable(d, num_hidden) ? lrds::mlp_grad_params(d, num_hidden) : (int64_t)LRDS_ERR_UNSUPPORTED;
}
int64_t lrds_mlp_grad_scratch_floats(int32_t d, int32_t num_hidden, int32_t S, int32_t B) {
  if (!lrds::mlp_grad_applicable(d, num_hidden) || S < 1 || B < 1) return (int64_t)LRDS_ERR_UNSUPPORTED;
  return lrds::mlp_grad_scratch_floats(d, num_hidden, S, B);
}
int lrds_mlp_grad(const lrds_mlp* mlp, const float* bias1, const float* x, const float* cot, const float* step_w,
                  const float* row_w, float clip, float cot_scale, const float* cot_scale_dev, int32_t S, int32_t B,
                  float* grads_out, float* dbias1_out, float* scratch, void* stream) {
  if (!mlp || !bias1 || !x || !cot || !grads_out || !dbias1_out || !scratch || S < 1 || B < 1 ||
      (!cot_scale_dev && !(cot_scale > 0.f)))
    return fail(LRDS_ERR_INVALID, "mlp_grad: bad arguments");
  const int r = lrds::launch_mlp_grad(*mlp, bias1, x, cot, step_w, row_w, clip, cot_scale, cot_scale_dev, S, B, grads_out, dbias1_out,
                                      scratch, (cudaStream_t)stream);
  if (r == LRDS_OK) g_launches.fetch_add(2);
  return r;
}

int lrds_distr_eval(const lrds_distr* distr, int32_t d, const float* x, int32_t B, float* logp_out, float* score_out,
                    void* stream) {
  return distr_eval_launch(distr, d, x, B, logp_out, score_out, 0.f, (cudaStream_t)stream);
}

int lrds_mala(const lrds_distr* target, int32_t d, int32_t C, int32_t n_warmup, int32_t n_steps, int32_t adapt,
              int32_t sampler, const float* y0, float* step_size, const float* noise, const float* unif, uint64_t seed,
              float* ys_out, float* log_acc_out, void* stream) {
  if (!target || !y0 || !step_size || !ys_out || d < 1 || C < 1 || n_warmup < 0 || n_steps < 1 ||
      (sampler != LRDS_MCMC_MALA && sampler != LRDS_MCMC_RWMH))
    return fail(LRDS_ERR_INVALID, "mala: bad arguments");
  lrds_spec s;
  if (int r = distr_spec(target, d, C, "mala", false, &s)) return r;
  s.kind = LRDS_ROLLOUT_CMCD;  // column layout with the three extra per-chain vectors (current state, two scores)
  const float tol = 0.05f, target_acc = 0.75f;
  MalaArgs m{y0, step_size, noise, unif, seed, ys_out, log_acc_out, n_warmup, n_steps, adapt, sampler,
             logf(target_acc), log1pf(tol), -log1pf(-tol), 1.01f};
  // few chains, long loops: at most one warp per CTA spreads the chains over the SMs
  return launch_cols(mala_kernel, "mala", s, {32}, (cudaStream_t)stream, s, m);
}

int lrds_axpy_step(const float* x, const float* s, const float* z, float a, float b, float c, float* out, int64_t n,
                   void* stream) {
  if (!x || !out || n < 1) return fail(LRDS_ERR_INVALID, "axpy_step: bad arguments");
  const int threads = 256;
  const int64_t want = (n + threads - 1) / threads;
  const int grid = (int)(want < 148 * 8 ? want : 148 * 8);
  axpy_step_kernel<<<grid, threads, 0, (cudaStream_t)stream>>>(x, s, z, a, b, c, out, n);
  return launched("axpy_step");
}

int lrds_normals(uint64_t seed, uint64_t particle_offset, int32_t stream_id, int32_t K, int32_t B, int32_t d, float* out,
                 void* stream) {
  if (!out || K < 1 || B < 1 || d < 1) return fail(LRDS_ERR_INVALID, "normals: bad arguments");
  const int64_t total = (int64_t)K * B * ((d + 3) / 4);
  const int threads = 256;
  const int64_t want = (total + threads - 1) / threads;
  const int grid = (int)(want < 148 * 16 ? want : 148 * 16);
  normals_kernel<<<grid, threads, 0, (cudaStream_t)stream>>>(seed, particle_offset, stream_id, K, B, d, out);
  return launched("normals");
}

}  // extern "C"
