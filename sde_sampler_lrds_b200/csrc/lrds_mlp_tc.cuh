// Building blocks of the drift network's backward pass on tcgen05, shared by the weight-gradient kernel
// (lrds_mlp_grad.cu) and the tensor-core adjoint (lrds_adjoint.cuh): a tile of 128 rows, four threads per row (TMEM lane
// = row, the threads split the columns in quarters), the A operand as fp16 (hi, lo) parts in TMEM, the rollout's F16X3
// weight image as B.  Forward GEMMs read the image K-major; the backward-data GEMMs read the SAME image MN-major (the
// contraction runs over the image's rows).  GELU' of every layer is kept in TMEM as 16-bit fixed point.
#pragma once
#include <cuda_fp16.h>

#include "lrds_rollout_tc.cuh"

namespace lrds {

constexpr int MG_THREADS = 512;  // 16 warps: four threads per row of the tile, 16 columns each
constexpr uint32_t MG_A_HI = 0, MG_A_LO = 32, MG_D = 64, MG_GP = 128, MG_ACC = 256, MG_TMEM_COLS = 512;
constexpr uint32_t MG_GROUP = 2048;  // 8 features x 128 rows x fp16: [row][8] with 16 bytes per row

// 64 GELU(v) and GELU'(v) = Phi(v) + v phi(v) for a pair (same erfc polynomial as gelu_pair, lrds_device.cuh)
__device__ __forceinline__ void gelu_grad_pair(u64 v2, u64& g64, float& da, float& db) {
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
  float pa, pb, ea, eb, wa, wb;
  f2::unpack(f2::mul(q, nt), pa, pb);
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(ea) : "f"(pa));  // erfc(|v| / sqrt 2) = 2 Phi(-|v|)
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(eb) : "f"(pb));
  const u64 r = f2::mul(f2::pack(fmaxf(va, 0.f), fmaxf(vb, 0.f)), f2::pk(TC_ACT_SCALE));
  g64 = f2::fma(f2::mul(nt, f2::pk(0.5f * TC_ACT_SCALE)), f2::pack(ea, eb), r);
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(wa) : "f"(-0.72134752f * va * va));  // exp(-v^2 / 2)
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(wb) : "f"(-0.72134752f * vb * vb));
  da = fmaf(va * 0.3989422804f, wa, va > 0.f ? fmaf(-0.5f, ea, 1.0f) : 0.5f * ea);
  db = fmaf(vb * 0.3989422804f, wb, vb > 0.f ? fmaf(-0.5f, eb, 1.0f) : 0.5f * eb);
}

__device__ __forceinline__ void split_pack(float a, float b, uint32_t& hi, uint32_t& lo) {
  u64 h2, l2;
  f2::split(f2::pack(a, b), h2, l2);
  float h0, h1, l0, l1;
  f2::unpack(h2, h0, h1);
  f2::unpack(l2, l0, l1);
  hi = ptx::pack_f16x2(h0, h1);
  lo = ptx::pack_f16x2(l0, l1);
}

// GELU' lies in (-0.13, 1.13): two values per TMEM column as 16-bit fixed point (step 2^-15, absolute error 1.5e-5; an
// fp16 pair would carry a RELATIVE 2.4e-4, which enters every delta upstream of the layer).  v + 256.25 has the 16 bits
// round((v + 0.25) 2^15) at the bottom of its significand: one FADD and half a byte permute per value either way.
__device__ __forceinline__ uint32_t pack_gp(float a, float b) {
  return __byte_perm(__float_as_uint(a + 256.25f), __float_as_uint(b + 256.25f), 0x5410);
}
__device__ __forceinline__ float2 unpack_gp(uint32_t p) {
  return make_float2(__uint_as_float(0x43800000u | (p & 0xFFFFu)) - 256.25f, __uint_as_float(0x43800000u | (p >> 16)) - 256.25f);
}

// D[128][N] = A[128][K] W^T with W the image's layer [N][K] (K-major), 3-pass (lo.hi, hi.lo, hi.hi); one elected thread
__device__ __forceinline__ void mg_mma_fwd(uint32_t tmem, uint32_t img_s, const TcLayout& TL, uint32_t b_off, int K, int N) {
  const uint32_t idesc = ptx::make_idesc_f16(128, N);
  const int ksteps = K / 16;
  const uint32_t kbytes = 2u * (uint32_t)N * 16u;
  uint32_t acc = 0;
  auto pass = [&](uint32_t acol, int b_part) {
    const uint32_t bbase = img_s + (uint32_t)b_part * TL.part_bytes + b_off;
    for (int ks = 0; ks < ksteps; ++ks) {
      const uint64_t bd = ptx::make_smem_desc(bbase + (uint32_t)ks * kbytes, (uint32_t)N * 16u, 128u);
      ptx::mma_bf16_ts(tmem + MG_D, tmem + acol + ks * 8, bd, idesc, acc);
      acc = 1;
    }
  };
  pass(MG_A_LO, 0);
  pass(MG_A_HI, 1);
  pass(MG_A_HI, 0);
}
// D[128][Nres] = A[128][Nimg] W: the image's rows (Nimg of them) are the contraction index, its K the Nres result
// columns (64 for the hidden / output layers, Kin for the input layer)
__device__ __forceinline__ void mg_mma_bwd(uint32_t tmem, uint32_t img_s, const TcLayout& TL, uint32_t b_off, int Nimg, int Nres) {
  const uint32_t idesc = ptx::make_idesc_f16(128, Nres) | ptx::IDESC_B_MN;
  const int ksteps = Nimg / 16;
  uint32_t acc = 0;
  auto pass = [&](uint32_t acol, int b_part) {
    const uint32_t bbase = img_s + (uint32_t)b_part * TL.part_bytes + b_off;
    for (int ks = 0; ks < ksteps; ++ks) {
      const uint64_t bd = ptx::make_smem_desc(bbase + (uint32_t)ks * 256u, 128u, (uint32_t)Nimg * 16u);
      ptx::mma_bf16_ts(tmem + MG_D, tmem + acol + ks * 8, bd, idesc, acc);
      acc = 1;
    }
  };
  pass(MG_A_LO, 0);
  pass(MG_A_HI, 1);
  pass(MG_A_HI, 0);
}

// Epilogue of forward layer l for this thread's 16 columns (block h): v = D un-scaled by `us` + bias (b4: layer 0 reads
// the per-time bias rows from global memory, the hidden layers the image's biases), 64 GELU(v) to TMEM as the next A
// operand (hi, lo), GELU'(v) to TMEM columns MG_GP + 32 l; pg = the activations' single fp16 rounding (the weight-gradient
// operand).  TRACK: vmax = max(vmax, |v|) (the F16X3 saturation check of the hidden pre-activations).
template <bool TRACK>
__device__ __forceinline__ void mg_forward_layer(uint32_t tm_lane, int h, int l, float us, const float4* b4, uint32_t (&pg)[8],
                                                 float& vmax) {
  const u64 us2 = f2::pk(us);
  uint32_t rr[16];
  ptx::tmem_ld16(tm_lane + MG_D + 16 * h, rr);
  ptx::tmem_wait_ld();
  uint32_t ph[8], pl[8], pp[8];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float4 bb = l == 0 ? __ldg(b4 + i) : b4[i];
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const u64 acc = f2::pack(__uint_as_float(rr[4 * i + 2 * e]), __uint_as_float(rr[4 * i + 2 * e + 1]));
      const u64 v = f2::fma(acc, us2, e ? f2::pack(bb.z, bb.w) : f2::pack(bb.x, bb.y));
      if constexpr (TRACK) {
        float va, vb;
        f2::unpack(v, va, vb);
        vmax = max3abs(vmax, va, vb);
      }
      u64 g;
      float da, db, ga, gb;
      gelu_grad_pair(v, g, da, db);
      f2::unpack(g, ga, gb);
      split_pack(ga, gb, ph[2 * i + e], pl[2 * i + e]);
      pg[2 * i + e] = ptx::pack_f16x2(ga, gb);
      pp[2 * i + e] = pack_gp(da, db);
    }
  }
  ptx::tmem_st8(tm_lane + MG_A_HI + 8 * h, ph);
  ptx::tmem_st8(tm_lane + MG_A_LO + 8 * h, pl);
  ptx::tmem_st8(tm_lane + MG_GP + 32 * l + 8 * h, pp);
}

}  // namespace lrds
