// Device-side building blocks shared by the rollout kernels (fp32 SIMT path and the epilogues of the
// tcgen05 path): per-particle column views of shared memory, exact GELU, Philox4x32-10 normals, the
// distribution scores / log-densities and the FourierMLP layers in thread-per-particle form.
//
// Arithmetic follows the reference (file:line relative to /root/reference/sde_sampler/):
//   GELU (exact erf)          conf/model/base/fouriermlp.yaml:5-6, models/mlp.py:141-143
//   diag-GMM logits / score   distr/gauss.py:67-73, 97-107, 124-126, 202-221
//   PhiFour U / grad_U        distr/phi_four.py:45-96
//   logistic regression       distr/logistic_regression.py:41-61 (+ autograd score, distr/base.py:146-154)
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/lrds_b200.h"

namespace lrds {

constexpr int C = LRDS_CHANNELS;  // hidden width
constexpr int JC = 8;             // dimension chunk processed per inner iteration

// A particle's private vector living in shared memory as a column: element j of thread t is at
// base[j * stride + t]; with stride = blockDim.x (a multiple of 32) a warp touches 32 consecutive banks.
struct Col {
  float* p;
  int stride;
  __device__ __forceinline__ float& operator()(int j) const { return p[j * stride]; }
};

// The same for vectors that the hot loops read four dims at a time (x, mixture responsibilities): dims
// [4c, 4c+4) of thread t are the float4 at base[(c * blockDim.x + t) * 4], so one conflict-free LDS.128 feeds
// four lanes of arithmetic.  Scalar access stays available (4-way bank conflict: keep it off the hot paths).
struct Col4 {
  float* p;    // base + 4 * threadIdx.x
  int stride;  // 4 * blockDim.x floats between consecutive groups
  __device__ __forceinline__ float& operator()(int j) const { return p[(j >> 2) * stride + (j & 3)]; }
  __device__ __forceinline__ float4 ld4(int c) const { return *reinterpret_cast<const float4*>(p + c * stride); }
  __device__ __forceinline__ ulonglong2 ldu(int c) const { return *reinterpret_cast<const ulonglong2*>(p + c * stride); }
  __device__ __forceinline__ void st4(int c, const float4& v) const { *reinterpret_cast<float4*>(p + c * stride) = v; }
  __device__ __forceinline__ void stu(int c, const ulonglong2& v) const { *reinterpret_cast<ulonglong2*>(p + c * stride) = v; }
};

// clip bounds arrive as "<= 0: no clip"; kernels turn that into +inf once so that a clip is two FMNMX
__device__ __forceinline__ float clip_bound(float c) { return c > 0.f ? c : INFINITY; }
// clip(v, -bound, bound) for bound >= 0 (possibly +inf) as ONE instruction: min(|v|, bound) with v's sign (the bound's
// sign bit is 0); NaN propagates like torch.clip
__device__ __forceinline__ float clipb(float v, float bound) {
  float r;
  asm("min.NaN.xorsign.abs.f32 %0, %1, %2;" : "=f"(r) : "f"(v), "f"(bound));
  return r;
}
__device__ __forceinline__ float clipf(float v, float c) { return c > 0.f ? fminf(fmaxf(v, -c), c) : v; }

// Packed fp32x2 arithmetic (FFMA2 / FMUL2 on sm_100): one issue slot for two lanes of work.
typedef unsigned long long u64;
namespace f2 {
__device__ __forceinline__ u64 pack(float a, float b) {
  u64 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ void unpack(u64 v, float& a, float& b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); }
__device__ __forceinline__ u64 fma(u64 a, u64 b, u64 c) {
  u64 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ u64 mul(u64 a, u64 b) {
  u64 d;
  asm("mul.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ u64 pk(float a) { return pack(a, a); }
__device__ __forceinline__ float hsum1(u64 a) {
  float x, y;
  unpack(a, x, y);
  return x + y;
}
// (hi, lo) of a pair for the 3-pass operand splits: hi = the top 11 significand bits of each lane, lo = v - hi (exact)
__device__ __forceinline__ void split(u64 v, u64& hi, u64& lo) {
  hi = v & 0xFFFFE000FFFFE000ull;
  lo = fma(hi, pk(-1.0f), v);
}
__device__ __forceinline__ float hsum(u64 a, u64 b) {  // (a.x + a.y) + (b.x + b.y)
  float x, y, z, w;
  unpack(a, x, y);
  unpack(b, z, w);
  return (x + y) + (z + w);
}
}  // namespace f2

// three-input max (FMNMX3 on sm_100) for the saturation trackers of the fp16 tensor-core operands
__device__ __forceinline__ float max3(float a, float b, float c) {
  float d;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}
__device__ __forceinline__ float max3abs(float a, float b, float c) {  // max(|a|, |b|, |c|)
  float d;
  asm("max.abs.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}
constexpr float F16X3_MAX_COORD = 65504.f;  // largest coordinate the fp16 (hi, lo) A operand holds
constexpr float F16X3_MAX_PREACT = 1023.f;  // hidden activations enter as 64 GELU(v): v beyond this saturates

// GELU with the exact (erf) definition, conf/model/base/fouriermlp.yaml:5-6:  v/2 (1 + erf(v / sqrt 2)).
// erf(|x|) = 1 - 2^(|x| Q(|x|)) with a degree-6 minimax Q on [0, 4] (saturated beyond): absolute error of erf
// 7.7e-8, of the GELU 1.6e-7 max(1, |v|) - the same as evaluating the erf formula in fp32 (tools/fit_erf.py).
// One MUFU.EX2 and 9 FMA-pipe instructions instead of erff's ~25.
__device__ __forceinline__ float gelu_exact(float v) {
  const float t = fminf(fabsf(v), 5.656854249f);
  float q = 8.857967404e-06f;
  q = fmaf(q, t, -5.769414971e-05f);
  q = fmaf(q, t, -4.069866499e-04f);
  q = fmaf(q, t, 7.363130652e-03f);
  q = fmaf(q, t, -5.266660834e-02f);
  q = fmaf(q, t, -4.591643231e-01f);
  q = fmaf(q, t, -1.151108839e+00f);
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(q * t));
  const float r = copysignf(1.0f - e, v);
  const float h = 0.5f * v;
  return fmaf(h, r, h);
}

// The same for two values at once on packed fp32x2 arithmetic (one issue slot per pair for the polynomial).
// `half_scale` = 0.5 * s returns s * GELU (s a power of two: the fp16 tensor-core operands are pre-scaled).
__device__ __forceinline__ void gelu_exact2(float va, float vb, float& ga, float& gb, float half_scale = 0.5f) {
  const u64 t = f2::pack(fminf(fabsf(va), 5.656854249f), fminf(fabsf(vb), 5.656854249f));
  u64 q = f2::pack(8.857967404e-06f, 8.857967404e-06f);
  q = f2::fma(q, t, f2::pack(-5.769414971e-05f, -5.769414971e-05f));
  q = f2::fma(q, t, f2::pack(-4.069866499e-04f, -4.069866499e-04f));
  q = f2::fma(q, t, f2::pack(7.363130652e-03f, 7.363130652e-03f));
  q = f2::fma(q, t, f2::pack(-5.266660834e-02f, -5.266660834e-02f));
  q = f2::fma(q, t, f2::pack(-4.591643231e-01f, -4.591643231e-01f));
  q = f2::fma(q, t, f2::pack(-1.151108839e+00f, -1.151108839e+00f));
  float pa, pb, ea, eb;
  f2::unpack(f2::mul(q, t), pa, pb);
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(ea) : "f"(pa));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(eb) : "f"(pb));
  const u64 r = f2::pack(copysignf(1.0f - ea, va), copysignf(1.0f - eb, vb));
  const u64 h = f2::mul(f2::pack(half_scale, half_scale), f2::pack(va, vb));
  f2::unpack(f2::fma(h, r, h), ga, gb);
}

// The same GELU for a pair in the form  s GELU(v) = s relu(v) + nt (s/2) 2^(t Q(t)),  nt = -t = -min(|v|, 4 sqrt 2):
// no sign transfer and no 1 - e; the polynomial runs in nt (P(nt) = -Q(-nt)) and s/2 = 2^k2 enters through the
// exponent.  `s` is a power of two (1, or the fp16 operand scale of the tensor-core path).
__device__ __forceinline__ u64 gelu_pair(u64 v2, float k2, float s) {
  float va, vb;
  f2::unpack(v2, va, vb);
  const u64 nt = f2::pack(fmaxf(-fabsf(va), -5.656854249f), fmaxf(-fabsf(vb), -5.656854249f));
  u64 q = f2::pk(-8.857967404e-06f);
  q = f2::fma(q, nt, f2::pk(-5.769414971e-05f));
  q = f2::fma(q, nt, f2::pk(4.069866499e-04f));
  q = f2::fma(q, nt, f2::pk(7.363130652e-03f));
  q = f2::fma(q, nt, f2::pk(5.266660834e-02f));
  q = f2::fma(q, nt, f2::pk(-4.591643231e-01f));
  q = f2::fma(q, nt, f2::pk(1.151108839e+00f));
  float pa, pb, ea, eb;
  f2::unpack(f2::fma(q, nt, f2::pk(k2)), pa, pb);
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(ea) : "f"(pa));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(eb) : "f"(pb));
  u64 r = f2::pack(fmaxf(va, 0.f), fmaxf(vb, 0.f));
  if (s != 1.0f) r = f2::mul(r, f2::pk(s));
  return f2::fma(nt, f2::pack(ea, eb), r);
}

// ---------------------------------------------------------------------------------------------------
// Philox4x32-10 + Box-Muller; spec in oracle/philox_ref.py (the numpy statement the tests compare with)
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mulwide(uint32_t a, uint32_t m, uint32_t& hi, uint32_t& lo) {  // one IMAD.WIDE.U32
  asm("{\n\t.reg .b64 t;\n\tmul.wide.u32 t, %2, %3;\n\tmov.b64 {%0, %1}, t;\n\t}" : "=r"(lo), "=r"(hi) : "r"(a), "r"(m));
}
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                               uint32_t k1, uint32_t (&out)[4]) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0, lo0, hi1, lo1;
    mulwide(c0, 0xD2511F53u, hi0, lo0);
    mulwide(c2, 0xCD9E8D57u, hi1, lo1);
    c0 = hi1 ^ c1 ^ k0;
    c1 = lo1;
    c2 = hi0 ^ c3 ^ k1;
    c3 = lo0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

__device__ __forceinline__ void box_muller(uint32_t ra, uint32_t rb, float& z0, float& z1) {
  const float u1 = (float)((ra >> 8) + 1u) * 5.9604644775390625e-08f;  // (0, 1]
  const float u2 = (float)(rb >> 8) * 5.9604644775390625e-08f;         // [0, 1)
  float l2, rad;  // sqrt(-2 ln u1) = sqrt(-2 ln2 * lg2 u1): two MUFU ops
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l2) : "f"(u1));
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rad) : "f"(l2 * -1.3862943611198906f));
  float s, c;
  __sincosf(fmaf(u2, 6.283185307179586f, -3.141592653589793f), &s, &c);
  z0 = rad * c;
  z1 = rad * s;
}

// four normals for dims [4*blk, 4*blk+4) of particle `pidx` at step `step`
__device__ __forceinline__ void normals4(uint64_t seed, uint32_t pidx, uint32_t step, uint32_t blk,
                                         uint32_t stream_id, float (&z)[4]) {
  uint32_t r[4];
  philox4x32_10(pidx, step, blk, stream_id, (uint32_t)seed, (uint32_t)(seed >> 32), r);
  box_muller(r[0], r[1], z[0], z[1]);
  box_muller(r[2], r[3], z[2], z[3]);
}

// ---------------------------------------------------------------------------------------------------
// diagonal Gaussian mixture
// ---------------------------------------------------------------------------------------------------
// Warp-uniform operand pointer.  SH = the operand block sits in shared memory (staged per step by the TMA engine:
// one wavefront per warp-uniform LDS.128, 32-bit address arithmetic) instead of global memory (read-only path:
// four wavefronts per warp-uniform LDG.128).
template <bool SH>
struct PPtr;
template <>
struct PPtr<false> {
  const float* p;
  __device__ __forceinline__ PPtr operator+(int floats) const { return PPtr{p + floats}; }
  __device__ __forceinline__ float4 ld4(int i) const { return __ldg(reinterpret_cast<const float4*>(p) + i); }
  __device__ __forceinline__ float ld1(int i) const { return __ldg(p + i); }
  __device__ __forceinline__ ulonglong2 ld2(int i) const { return __ldg(reinterpret_cast<const ulonglong2*>(p) + i); }
};
template <>
struct PPtr<true> {
  uint32_t a;  // shared-window byte address
  __device__ __forceinline__ PPtr operator+(int floats) const { return PPtr{a + 4u * (uint32_t)floats}; }
  __device__ __forceinline__ float4 ld4(int i) const {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a + 16u * (uint32_t)i));
    return v;
  }
  __device__ __forceinline__ float ld1(int i) const {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a + 4u * (uint32_t)i));
    return v;
  }
  __device__ __forceinline__ ulonglong2 ld2(int i) const {  // the same 16 bytes as two packed fp32 pairs
    ulonglong2 v;
    asm volatile("ld.shared.v2.b64 {%0,%1}, [%2];" : "=l"(v.x), "=l"(v.y) : "r"(a + 16u * (uint32_t)i));
    return v;
  }
};

template <bool SH>
__device__ __forceinline__ float4 gld4(const float4* p) {  // plain pointers: shared is inferred by the compiler
  if constexpr (SH) return *p;
  else return __ldg(p);
}

// A mixture block.  Mixtures (M > 1) are evaluated from (logc, sn = interleaved 1/sigma and -mu/sigma, see
// lrds_gmm), possibly staged in shared memory; single Gaussians (M == 1) from (glogc, mu, ivar) in global memory in
// the reference's operation order.
template <bool SH>
struct GmmViewT {
  int M;
  PPtr<SH> logc, sn;
  PPtr<false> glogc, mu, ivar;
};
using GmmView = GmmViewT<false>;

__device__ __forceinline__ GmmView gmm_at(const lrds_gmm& g, int step) {
  GmmView v;
  const int64_t o = (int64_t)step * g.step_stride_param;
  v.M = g.M;
  v.logc = v.glogc = PPtr<false>{g.logc + (int64_t)step * g.step_stride_logc};
  v.mu = PPtr<false>{g.mu + o};
  v.ivar = PPtr<false>{g.ivar + o};
  v.sn = PPtr<false>{g.sn + (int64_t)step * g.step_stride_sn};
  return v;
}

// Mixture parameters are rows of dp = d_pad floats (zero padded), read as warp-uniform 16-byte vectors.
__device__ __forceinline__ void quad4(float& q, const float4& xv, const float4& mu, const float4& iv) {
  float t;
  t = xv.x - mu.x; q = fmaf(t * t, iv.x, q);
  t = xv.y - mu.y; q = fmaf(t * t, iv.y, q);
  t = xv.z - mu.z; q = fmaf(t * t, iv.z, q);
  t = xv.w - mu.w; q = fmaf(t * t, iv.w, q);
}

// Operands of one pass-1 block: four dims of x and of four modes' (1/sigma, -mu/sigma) = 8 consecutive 16-byte
// vectors of `sn`.  PIPE keeps two of these in registers and loads block c+1 while block c computes (ptxas does not
// pipeline loads across loop iterations on its own, and with <= 2 warps per scheduler nothing else hides the latency).
template <bool SH>
struct Pass1Ops {
  ulonglong2 xv, s[4], n[4];
  __device__ __forceinline__ void load(const Col4& x, int c, const PPtr<SH>& p) {  // p = sn + (block * rowq + c) * 32
    xv = x.ldu(c);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      s[i] = p.ld2(2 * i);
      n[i] = p.ld2(2 * i + 1);
    }
  }
  // w = x / sigma - mu / sigma (one FFMA2 per pair of dims), q += w^2 (one FFMA2 per pair)
  __device__ __forceinline__ void accumulate(u64 (&qa)[4], u64 (&qb)[4]) const {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const u64 w0 = f2::fma(xv.x, s[i].x, n[i].x), w1 = f2::fma(xv.y, s[i].y, n[i].y);
      qa[i] = f2::fma(w0, w0, qa[i]);
      qb[i] = f2::fma(w1, w1, qb[i]);
    }
  }
};

// Pass 1: responsibilities r(m) = softmax_m(logc_m - q_m / 2), q_m = sum_j (x_j - mu_mj)^2 / var_mj.
// Returns log sum_m exp(logit_m) (= the mixture log-density).  For M == 1, r is not touched.
// r holds 4 * ceil(M / 4) entries; padded modes carry logc = -inf, i.e. weight zero.
// PIPE: software-pipelined operand loads (needs ~40 more registers; used by the kernels compiled for <= 256 threads)
// MIX: the caller knows M > 1 (skips the single-Gaussian branch)
template <bool PIPE, bool MIX = false, bool SH>
__device__ __forceinline__ float gmm_pass1(const GmmViewT<SH>& g, int d, int dp, const Col4& x, const Col4& r) {
  const int nq = (d + 3) >> 2;  // 16-byte groups that hold real dims
  const int rowq = dp >> 2;     // groups per mode block in `sn`
  if (!MIX && g.M == 1) {
    float q = 0.f;
    for (int c = 0; c < nq; ++c) quad4(q, x.ld4(c), g.mu.ld4(c), g.ivar.ld4(c));
    return g.glogc.ld1(0) - 0.5f * q;
  }
  float mx = -INFINITY;
  const int M4 = (g.M + 3) >> 2;
  for (int mb = 0; mb < M4; ++mb) {  // 4 modes at a time so that one x load feeds 4 quadratic forms
    u64 qa[4] = {0, 0, 0, 0}, qb[4] = {0, 0, 0, 0};  // (even, odd) dim partial sums per mode
    PPtr<SH> p = g.sn + mb * rowq * 32;
    if constexpr (PIPE) {
      Pass1Ops<SH> A, B;
      A.load(x, 0, p);
      int c = 0;
      for (; c + 1 < nq; c += 2, p = p + 64) {
        B.load(x, c + 1, p + 32);
        A.accumulate(qa, qb);
        if (c + 2 < nq) A.load(x, c + 2, p + 64);
        B.accumulate(qa, qb);
      }
      if (c < nq) A.accumulate(qa, qb);
    } else {
#pragma unroll 2
      for (int c = 0; c < nq; ++c, p = p + 32) {
        Pass1Ops<SH> A;
        A.load(x, c, p);
        A.accumulate(qa, qb);
      }
    }
    const float4 lc = g.logc.ld4(mb);
    const float4 l = make_float4(lc.x - 0.5f * f2::hsum(qa[0], qb[0]), lc.y - 0.5f * f2::hsum(qa[1], qb[1]),
                                 lc.z - 0.5f * f2::hsum(qa[2], qb[2]), lc.w - 0.5f * f2::hsum(qa[3], qb[3]));
    r.st4(mb, l);
    mx = fmaxf(fmaxf(mx, fmaxf(l.x, l.y)), fmaxf(l.z, l.w));
  }
  float s = 0.f;
  for (int mb = 0; mb < M4; ++mb) {
    float4 l = r.ld4(mb);
    l.x = __expf(l.x - mx); l.y = __expf(l.y - mx); l.z = __expf(l.z - mx); l.w = __expf(l.w - mx);
    s += (l.x + l.y) + (l.z + l.w);
    r.st4(mb, l);
  }
  const float inv = 1.0f / s;
  for (int mb = 0; mb < M4; ++mb) {
    float4 l = r.ld4(mb);
    l.x *= inv; l.y *= inv; l.z *= inv; l.w *= inv;
    r.st4(mb, l);
  }
  return mx + __logf(s);
}

// Operands of one mode for an 8-dim chunk of pass 2: mode i of the block at p = sn + (block * rowq + j0 / 4) * 32
template <bool SH>
struct Pass2Ops {
  ulonglong2 s0, n0, s1, n1;
  __device__ __forceinline__ void load(const PPtr<SH>& p, int i, bool two) {
    s0 = p.ld2(2 * i);
    n0 = p.ld2(2 * i + 1);
    if (two) {
      s1 = p.ld2(8 + 2 * i);
      n1 = p.ld2(9 + 2 * i);
    }
  }
  // c = r / sigma;  a += c / sigma;  b += c (-mu / sigma)
  __device__ __forceinline__ void accumulate(float rm, bool two, u64 (&a)[4], u64 (&b)[4]) const {
    const u64 rm2 = f2::pack(rm, rm);
    const u64 c0 = f2::mul(rm2, s0.x), c1 = f2::mul(rm2, s0.y);
    a[0] = f2::fma(c0, s0.x, a[0]); b[0] = f2::fma(c0, n0.x, b[0]);
    a[1] = f2::fma(c1, s0.y, a[1]); b[1] = f2::fma(c1, n0.y, b[1]);
    if (two) {
      const u64 c2 = f2::mul(rm2, s1.x), c3 = f2::mul(rm2, s1.y);
      a[2] = f2::fma(c2, s1.x, a[2]); b[2] = f2::fma(c2, n1.x, b[2]);
      a[3] = f2::fma(c3, s1.y, a[3]); b[3] = f2::fma(c3, n1.y, b[3]);
    }
  }
};

// Pass 2 for dims [j0, j0+JC):  score_j = -sum_m r_m (x_j - mu_mj) / var_mj.  With c_mj = r_m / sigma_mj:
//   score_j = -( x_j sum_m c_mj / sigma_mj  +  sum_m c_mj (-mu_mj / sigma_mj) )
// i.e. one FMUL2 + two FFMA2 per mode and pair of dims (zero for the padded dims and modes).
template <bool PIPE, bool MIX = false, bool SH>
__device__ __forceinline__ void gmm_score_chunk(const GmmViewT<SH>& g, int d, int dp, const float (&xr)[JC], const Col4& r,
                                                int j0, float (&out)[JC]) {
  if (!MIX && g.M == 1) {  // -((x - mu) * ivar), the operation order of score_gauss (distr/gauss.py:124-126)
    const PPtr<false> mu = g.mu + j0, iv = g.ivar + j0;
    const float4 m0 = mu.ld4(0), m1 = mu.ld4(1), i0 = iv.ld4(0), i1 = iv.ld4(1);
    out[0] = -((xr[0] - m0.x) * i0.x); out[1] = -((xr[1] - m0.y) * i0.y);
    out[2] = -((xr[2] - m0.z) * i0.z); out[3] = -((xr[3] - m0.w) * i0.w);
    out[4] = -((xr[4] - m1.x) * i1.x); out[5] = -((xr[5] - m1.y) * i1.y);
    out[6] = -((xr[6] - m1.z) * i1.z); out[7] = -((xr[7] - m1.w) * i1.w);
    return;
  }
  const int blk = (dp >> 2) * 32;  // floats per mode block of `sn`
  const bool two = j0 + 4 < d;     // the second 16-byte group of the chunk holds real dims
  u64 a[4] = {0, 0, 0, 0}, b[4] = {0, 0, 0, 0};
  const int M4 = (g.M + 3) >> 2;
  PPtr<SH> p = g.sn + (j0 >> 2) * 32;
  if constexpr (PIPE) {  // operands of mode m+1 are loaded while mode m accumulates
    Pass2Ops<SH> A, B;
    A.load(p, 0, two);
    for (int mb = 0; mb < M4; ++mb, p = p + blk) {
      const float4 rm = r.ld4(mb);
      B.load(p, 1, two);
      A.accumulate(rm.x, two, a, b);
      A.load(p, 2, two);
      B.accumulate(rm.y, two, a, b);
      B.load(p, 3, two);
      A.accumulate(rm.z, two, a, b);
      if (mb + 1 < M4) A.load(p + blk, 0, two);
      B.accumulate(rm.w, two, a, b);
    }
  } else {
    for (int mb = 0; mb < M4; ++mb, p = p + blk) {
      const float4 rm = r.ld4(mb);
      const float rms[4] = {rm.x, rm.y, rm.z, rm.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        Pass2Ops<SH> T;
        T.load(p, i, two);
        T.accumulate(rms[i], two, a, b);
      }
    }
  }
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    float ax, ay, bx, by;
    f2::unpack(a[q], ax, ay);
    f2::unpack(b[q], bx, by);
    out[2 * q] = -fmaf(xr[2 * q], ax, bx);
    out[2 * q + 1] = -fmaf(xr[2 * q + 1], ay, by);
  }
}

// ---------------------------------------------------------------------------------------------------
// full-covariance Gaussian mixture (lrds_gmm.layout == LRDS_GMM_FULL), distr/gauss.py:76-121
// ---------------------------------------------------------------------------------------------------
// Per mode m: h_m = prec_m (x - mu_m), q_m = (x - mu_m) . h_m, logit_m = logc_m - q_m / 2.  The precision rows are
// warp-uniform 16-byte loads through L1 (one broadcast load feeds 32 particles); a per-step block is M d_pad^2 floats,
// far beyond the TMA step stage at the sizes this layout is for, so nothing is staged.  The arithmetic is fp32 in
// every network precision.
struct GmmFullView {
  int M;
  const float* logc;
  const float* mu;    // [M][dp]
  const float* prec;  // [M][dp][dp]
};
__device__ __forceinline__ GmmFullView gmm_full_at(const lrds_gmm& g, int step) {
  return GmmFullView{g.M, g.logc + (int64_t)step * g.step_stride_logc, g.mu + (int64_t)step * g.step_stride_param,
                     g.sn + (int64_t)step * g.step_stride_sn};
}

// q_m of mode m; with STORE, h_m goes to column h (zero in the padded dims: the padded precision rows are zero).
// Eight rows of prec at a time, so that one read of (x - mu) from the particle column feeds 32 FMA.
template <bool STORE>
__device__ __forceinline__ float gmm_full_mode(const GmmFullView& g, int m, int d, int dp, const Col4& x, const Col4& h) {
  const float* P = g.prec + (int64_t)m * dp * dp;
  const float4* mu4 = reinterpret_cast<const float4*>(g.mu + (int64_t)m * dp);
  const int nq = (d + 3) >> 2;
  float q = 0.f;
  for (int i0 = 0; i0 < d; i0 += JC) {
    float acc[JC];
#pragma unroll
    for (int r = 0; r < JC; ++r) acc[r] = 0.f;
    const float4* row = reinterpret_cast<const float4*>(P + (int64_t)i0 * dp);
    const int rq = dp >> 2;  // float4 per row
#pragma unroll 2
    for (int c = 0; c < nq; ++c) {
      const float4 xv = x.ld4(c), mv = __ldg(mu4 + c);
      const float y0 = xv.x - mv.x, y1 = xv.y - mv.y, y2 = xv.z - mv.z, y3 = xv.w - mv.w;
#pragma unroll
      for (int r = 0; r < JC; ++r) {
        const float4 p = __ldg(row + r * rq + c);
        acc[r] = fmaf(p.x, y0, acc[r]);
        acc[r] = fmaf(p.y, y1, acc[r]);
        acc[r] = fmaf(p.z, y2, acc[r]);
        acc[r] = fmaf(p.w, y3, acc[r]);
      }
    }
    const float4 xa = x.ld4(i0 >> 2), xb = x.ld4((i0 >> 2) + 1);
    const float4 ma = __ldg(mu4 + (i0 >> 2)), mb = __ldg(mu4 + (i0 >> 2) + 1);
    q = fmaf(xa.x - ma.x, acc[0], q); q = fmaf(xa.y - ma.y, acc[1], q);
    q = fmaf(xa.z - ma.z, acc[2], q); q = fmaf(xa.w - ma.w, acc[3], q);
    q = fmaf(xb.x - mb.x, acc[4], q); q = fmaf(xb.y - mb.y, acc[5], q);
    q = fmaf(xb.z - mb.z, acc[6], q); q = fmaf(xb.w - mb.w, acc[7], q);
    if constexpr (STORE) {
      h.st4(i0 >> 2, make_float4(acc[0], acc[1], acc[2], acc[3]));
      h.st4((i0 >> 2) + 1, make_float4(acc[4], acc[5], acc[6], acc[7]));
    }
  }
  return q;
}

// log sum_m exp(logit_m) (the mixture log-density) in one pass over the modes with a running maximum.  With a score
// column `sc` (SCORE), also sc = -sum_m r_m h_m, r = softmax_m(logit_m), accumulated online: sc holds
// sum_m exp(logit_m - running max) h_m and is rescaled whenever the maximum moves; `h` is the per-mode scratch column.
template <bool SCORE>
__device__ __forceinline__ float gmm_full_pass(const GmmFullView& g, int d, int dp, const Col4& x, const Col4& sc,
                                               const Col4& h) {
  float mx = -INFINITY, s = 0.f;
  const int nq = dp >> 2;
  for (int m = 0; m < g.M; ++m) {
    const float l = __ldg(g.logc + m) - 0.5f * gmm_full_mode<SCORE>(g, m, d, dp, x, h);
    float w, scale;
    if (l > mx) {
      scale = __expf(mx - l);  // 0 for the first mode
      w = 1.f;
      mx = l;
    } else {
      scale = 1.f;
      w = __expf(l - mx);
    }
    s = fmaf(s, scale, w);
    if constexpr (SCORE) {
      if (m == 0) {
        for (int c = 0; c < nq; ++c) sc.st4(c, h.ld4(c));
      } else {
        for (int c = 0; c < nq; ++c) {
          const float4 a = sc.ld4(c), b = h.ld4(c);
          sc.st4(c, make_float4(fmaf(a.x, scale, w * b.x), fmaf(a.y, scale, w * b.y), fmaf(a.z, scale, w * b.z),
                                fmaf(a.w, scale, w * b.w)));
        }
      }
    }
  }
  if constexpr (SCORE) {
    const float inv = -1.0f / s;
    for (int c = 0; c < nq; ++c) {
      const float4 a = sc.ld4(c);
      sc.st4(c, make_float4(a.x * inv, a.y * inv, a.z * inv, a.w * inv));
    }
  }
  return mx + __logf(s);
}

// ---------------------------------------------------------------------------------------------------
// PhiFour (1-D lattice, Dirichlet-0)
// ---------------------------------------------------------------------------------------------------
// score_j = -beta * [ (b - x_j (1 - x_j^2)) / coef + coef (2 x_j - x_{j+1} - x_{j-1}) ]
__device__ __forceinline__ float phi4_score_1(const lrds_phi4& p, float coef, float xm, float x0, float xp) {
  const float ret = (p.b - x0 * (1.0f - x0 * x0)) / coef + coef * (2.0f * x0 - xp - xm);
  return -p.beta * ret;
}

// log-density -beta * U(x), U = coef * sum_{i=0..d} (x_{i+1}-x_i)^2/2 + sum((1-x^2)^2/4 + b x)/coef
__device__ __forceinline__ float phi4_logp(const lrds_phi4& p, int d, const Col4& x) {
  const float coef = p.a * (float)d;
  float grad = 0.f, v = 0.f, prev = 0.f;
  for (int c = 0; 4 * c < d; ++c) {
    const float4 q = x.ld4(c);
    const float xs[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      if (4 * c + e < d) {
        const float xj = xs[e];
        const float df = xj - prev;
        grad += df * df * 0.5f;
        const float w = 1.0f - xj * xj;
        v += w * w * 0.25f + p.b * xj;
        prev = xj;
      }
    }
  }
  grad += prev * prev * 0.5f;
  return -p.beta * (grad * coef + v / coef);
}

// ---------------------------------------------------------------------------------------------------
// Bayesian logistic regression
// ---------------------------------------------------------------------------------------------------
// Pass 1: g(n) = m_n (y_n - sigma(z_n)), z_n = X_n . w + intercept, m_n = [eps <= sigma(z_n) <= 1 - eps].
// With want_logp the log-posterior (likelihood + Normal priors) is returned.
__device__ __forceinline__ float logreg_pass1(const lrds_logreg& L, int d, const Col4& x, const Col& g, bool want_logp) {
  const float icpt = x(d - 1);
  const float hi = 1.0f - L.eps;
  float ll = 0.f;
  for (int n = 0; n < L.N; n += 4) {
    float z0 = 0.f, z1 = 0.f, z2 = 0.f, z3 = 0.f;
    const float* xt = L.Xt + n;
    for (int jq = 0; 4 * jq < L.p; ++jq) {
      const float4 xq = x.ld4(jq);
      const float xs[4] = {xq.x, xq.y, xq.z, xq.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int j = 4 * jq + e;
        if (j < L.p) {
          const float4 v = __ldg(reinterpret_cast<const float4*>(xt + (int64_t)j * L.n_pad));
          z0 = fmaf(v.x, xs[e], z0); z1 = fmaf(v.y, xs[e], z1); z2 = fmaf(v.z, xs[e], z2); z3 = fmaf(v.w, xs[e], z3);
        }
      }
    }
    const float zz[4] = {z0 + icpt, z1 + icpt, z2 + icpt, z3 + icpt};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (n + i < L.N) {
        const float yn = __ldg(L.y + n + i);
        const float sig = 1.0f / (1.0f + expf(-zz[i]));
        const bool inside = (sig >= L.threshold) && (sig >= L.eps) && (sig <= hi);
        g(n + i) = inside ? (yn - sig) : 0.f;
        if (want_logp) {
          const float ps = fminf(fmaxf(fmaxf(sig, L.threshold), L.eps), hi);
          ll += yn * logf(ps) + (1.0f - yn) * log1pf(-ps);
        }
      }
    }
  }
  if (!want_logp) return 0.f;
  // Normal priors, logistic_regression.py:27-39, 51-53
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

// Pass 2 for dims [j0, j0+JC): score_j = sum_n g_n X_nj - w_j / s_w^2 ; intercept: sum_n g_n - (b - m)/s_b^2
__device__ __forceinline__ void logreg_score_chunk(const lrds_logreg& L, int d, int d_pad, const float (&xr)[JC],
                                                   const Col& g, int j0, float (&out)[JC]) {
  float acc[JC];
  float gs = 0.f;
#pragma unroll
  for (int c = 0; c < JC; ++c) acc[c] = 0.f;
  for (int n = 0; n < L.N; ++n) {
    const float gn = g(n);
    const float4* row = reinterpret_cast<const float4*>(L.X + (int64_t)n * d_pad + j0);
    const float4 a = __ldg(row), b = __ldg(row + 1);
    acc[0] = fmaf(gn, a.x, acc[0]); acc[1] = fmaf(gn, a.y, acc[1]); acc[2] = fmaf(gn, a.z, acc[2]);
    acc[3] = fmaf(gn, a.w, acc[3]); acc[4] = fmaf(gn, b.x, acc[4]); acc[5] = fmaf(gn, b.y, acc[5]);
    acc[6] = fmaf(gn, b.z, acc[6]); acc[7] = fmaf(gn, b.w, acc[7]);
    gs += gn;
  }
  const float iw = 1.0f / (L.weight_scale * L.weight_scale);
#pragma unroll
  for (int c = 0; c < JC; ++c) {
    const int j = j0 + c;
    if (j < L.p) out[c] = acc[c] - xr[c] * iw;
    else if (j == L.p) out[c] = gs - (xr[c] - L.intercept_mean) / (L.intercept_scale * L.intercept_scale);
    else out[c] = 0.f;
  }
}

// ---------------------------------------------------------------------------------------------------
// FourierMLP, thread-per-particle (fp32 SIMT).  Weights are read through the read-only path: every lane
// of a warp reads the same address, so each 16-byte load is one broadcast transaction.
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void fma_row64(float (&acc)[C], const float* __restrict__ wrow, float a) {
  const float4* w4 = reinterpret_cast<const float4*>(wrow);
#pragma unroll
  for (int q = 0; q < C / 4; ++q) {
    const float4 v = __ldg(w4 + q);
    acc[4 * q + 0] = fmaf(v.x, a, acc[4 * q + 0]);
    acc[4 * q + 1] = fmaf(v.y, a, acc[4 * q + 1]);
    acc[4 * q + 2] = fmaf(v.z, a, acc[4 * q + 2]);
    acc[4 * q + 3] = fmaf(v.w, a, acc[4 * q + 3]);
  }
}

// GELU'(v) = Phi(v) + v phi(v) of the exact GELU
__device__ __forceinline__ float gelu_grad(float v) {
  return fmaf(v * 0.3989422804014327f, __expf(-0.5f * v * v), normcdff(v));
}

// hidden activations GELU(h_L) of the particle -> act(0..63)   (models/mlp.py:136-142)
// TAPE (the adjoint's forward recompute): also GELU'(h_l) of every layer l -> tape(64 l + n)
template <bool BIAS_SH, bool TAPE = false>
__device__ __forceinline__ void mlp_hidden(const lrds_mlp& w, const float* __restrict__ bias1, const Col4& x,
                                           const Col& act, const Col& tape = Col{nullptr, 0}) {
  float acc[C];
#pragma unroll
  for (int q = 0; q < C / 4; ++q) {
    const float4 b = gld4<BIAS_SH>(reinterpret_cast<const float4*>(bias1) + q);
    acc[4 * q] = b.x; acc[4 * q + 1] = b.y; acc[4 * q + 2] = b.z; acc[4 * q + 3] = b.w;
  }
  for (int kq = 0; 4 * kq < w.d; ++kq) {
    const float4 xq = x.ld4(kq);
    const float xs[4] = {xq.x, xq.y, xq.z, xq.w};
#pragma unroll
    for (int e = 0; e < 4; ++e)
      if (4 * kq + e < w.d) fma_row64(acc, w.w_in_t + (int64_t)(4 * kq + e) * C, xs[e]);
  }
#pragma unroll
  for (int n = 0; n < C; ++n) {
    act(n) = gelu_exact(acc[n]);
    if constexpr (TAPE) tape(n) = gelu_grad(acc[n]);
  }
  for (int l = 0; l < w.num_hidden; ++l) {
    const float* wl = w.w_hid_t + (int64_t)l * C * C;
#pragma unroll
    for (int n = 0; n < C; ++n) acc[n] = __ldg(w.b_hid + l * C + n);
#pragma unroll 2
    for (int k = 0; k < C; ++k) fma_row64(acc, wl + k * C, act(k));
#pragma unroll
    for (int n = 0; n < C; ++n) {
      act(n) = gelu_exact(acc[n]);
      if constexpr (TAPE) tape((l + 1) * C + n) = gelu_grad(acc[n]);
    }
  }
}

// out_layer for dims [j0, j0+JC)   (models/mlp.py:143)
__device__ __forceinline__ void mlp_out_chunk(const lrds_mlp& w, const Col& act, int j0, float (&out)[JC]) {
  {
    const float4* b4 = reinterpret_cast<const float4*>(w.b_out + j0);
    const float4 a = __ldg(b4), b = __ldg(b4 + 1);
    out[0] = a.x; out[1] = a.y; out[2] = a.z; out[3] = a.w; out[4] = b.x; out[5] = b.y; out[6] = b.z; out[7] = b.w;
  }
#pragma unroll 4
  for (int k = 0; k < C; ++k) {
    const float ak = act(k);
    const float4* row = reinterpret_cast<const float4*>(w.w_out_t + (int64_t)k * w.d_pad + j0);
    const float4 a = __ldg(row), b = __ldg(row + 1);
    out[0] = fmaf(a.x, ak, out[0]); out[1] = fmaf(a.y, ak, out[1]); out[2] = fmaf(a.z, ak, out[2]);
    out[3] = fmaf(a.w, ak, out[3]); out[4] = fmaf(b.x, ak, out[4]); out[5] = fmaf(b.y, ak, out[5]);
    out[6] = fmaf(b.z, ak, out[6]); out[7] = fmaf(b.w, ak, out[7]);
  }
}

// ---- block-wide helpers of the operand-image packers and the estimator ---------------------------------------------
struct MaxOp {
  template <class T>
  __device__ __forceinline__ T operator()(T a, T b) const { return fmax(a, b); }
};
struct SumOp {
  template <class T>
  __device__ __forceinline__ T operator()(T a, T b) const { return a + b; }
};
// op over the block's v (blockDim.x a multiple of 32): shuffles within the warps, then identity op the warp results in
// warp order 0, 1, ... (so sums are reproducible); `red` holds blockDim.x / 32 values; every thread gets the result
template <class T, class Op>
__device__ __forceinline__ T block_reduce(T v, Op op, T identity, T* red) {
  for (int o = 16; o > 0; o >>= 1) v = op(v, __shfl_xor_sync(0xffffffffu, v, o));
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  T r = identity;
  for (int w = 0; w < (int)(blockDim.x >> 5); ++w) r = op(r, red[w]);
  return r;
}
// k with amax * 2^k in [2^14, 2^15) (0 for amax = 0 or inf / NaN), clamped to [-100, 100]: the fp16 operand scale
__device__ __forceinline__ int pow2_exponent_for(float amax) {
  int k = 0;
  if (amax > 0.f && amax < INFINITY) k = 14 - ilogbf(amax);
  return k > 100 ? 100 : (k < -100 ? -100 : k);
}
// fp16 hi | lo split of vs: hi at out + byte, the rounding remainder at out + part_bytes + byte
__device__ __forceinline__ void put_hi_lo(uint8_t* out, uint32_t part_bytes, uint32_t byte, float vs) {
  const __half hi = __float2half_rn(vs);
  *reinterpret_cast<__half*>(out + byte) = hi;
  *reinterpret_cast<__half*>(out + part_bytes + byte) = __float2half_rn(vs - __half2float(hi));
}

}  // namespace lrds
