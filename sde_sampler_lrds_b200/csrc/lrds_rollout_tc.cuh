// tcgen05 tensor-core drift network (LRDS_PRECISION_TF32 / TF32X3 / BF16) and the kernel wrapper that runs the
// shared rollout body (lrds_rollout_simt.cuh) with it.
//
// Mapping.  A CTA holds W <= 16 warps = up to four 128-particle tiles; warp w integrates particles
// [32 w, 32 w + 32) of the CTA and owns TMEM lanes 32 (w % 4) .. +31 of tile w / 4, i.e. thread <-> particle <->
// TMEM lane <-> row of every GEMM.  Per grid step and tile the FourierMLP (models/mlp.py:135-143) is four GEMMs
//     [128 x Kin] . W_in^T -> GELU -> [128 x 64] . W_h^T -> GELU -> ... -> [128 x 64] . W_out^T
// issued by the tile's first thread as tcgen05.mma with the A operand in TMEM (written by the particles' own
// threads with tcgen05.st), B = the weight image in shared memory (K-major, no swizzle; staged ONCE per CTA by a
// bulk TMA copy) and the fp32 accumulator in TMEM (read back with tcgen05.ld for bias + GELU).  Activations never
// touch shared or global memory.  Tiles of one CTA run out of phase, so one tile's MMA latency is covered by the
// other tiles' SIMT work (scores, noise, integrator).
//
// Precisions: TF32X3 splits both operands into tf32 (hi, lo) and accumulates lo*hi + hi*lo + hi*hi (fp32-grade
// products, the parity mode); F16X3 does the same with fp16 (hi, lo) pairs of power-of-two scaled operands (weights
// scaled per layer so that max |W| lands in [2^14, 2^15), hidden activations by 64; the accumulator is scaled back by
// the bias FFMA of the epilogue): the same 22 mantissa bits per operand at half the shared-memory image, half the
// TMEM columns (=> twice the resident tiles) and twice the tensor rate.  TF32 and BF16 are single-pass
// reduced-precision modes reported separately.
#pragma once
#include <cuda_fp16.h>

#include "lrds_internal.h"
#include "lrds_rollout_simt.cuh"
#include "lrds_tc_ptx.cuh"

namespace lrds {

constexpr int TC_MAX_WARPS = 16;
// The tf32 3-pass split needs 192 TMEM columns per tile, i.e. at most two tiles = 8 warps per CTA: compile it for 256
// threads so that ptxas may use 255 registers and keep more operand loads in flight per warp.  The fp16 split needs
// 128 columns per tile; its kernels are compiled for three tiles = 12 warps (168 registers).
__host__ __device__ constexpr int tc_max_warps(int prec) {
  return prec == LRDS_PRECISION_TF32X3 ? 8 : prec == LRDS_PRECISION_F16X3 ? 12 : TC_MAX_WARPS;
}
constexpr int TC_TAIL_BYTES = 96;  // mbarriers (5 x 8 B) + TMEM slot (at 48) + the tiles' hand-off counters (4 x 4 B at 64) after the image
constexpr float TC_ACT_SCALE = 64.f;  // F16X3: hidden activations enter the tensor core as 64 * GELU(h)
__host__ __device__ constexpr bool tc_is_x3(int prec) { return prec == LRDS_PRECISION_TF32X3 || prec == LRDS_PRECISION_F16X3; }
__host__ __device__ constexpr bool tc_is_half(int prec) { return prec == LRDS_PRECISION_BF16 || prec == LRDS_PRECISION_F16X3; }

struct TcLayout {
  int prec, parts, es, kstep;
  int Kin, Nout, nh;
  uint32_t part_bytes, off_in, off_hid, off_out;  // one part = all layers of one (hi | lo) image
  uint32_t off_bhid, off_bout, off_scale, bytes;  // fp32 biases + 16 scale floats behind the parts; total bytes (multiple of 16)
  int a_cols, d_cols, tile_cols;                  // TMEM columns: one A part, the accumulator, one tile
};

__host__ __device__ inline TcLayout tc_layout(int d, int nh, int prec) {
  TcLayout L{};
  L.prec = prec;
  L.parts = tc_is_x3(prec) ? 2 : 1;
  L.es = tc_is_half(prec) ? 2 : 4;
  L.kstep = tc_is_half(prec) ? 16 : 8;
  L.Kin = (d + L.kstep - 1) / L.kstep * L.kstep;
  L.Nout = (d + 15) / 16 * 16;
  L.nh = nh;
  L.off_in = 0;
  L.off_hid = (uint32_t)(C * L.Kin * L.es);
  L.off_out = L.off_hid + (uint32_t)(nh * C * C * L.es);
  L.part_bytes = L.off_out + (uint32_t)(L.Nout * C * L.es);
  L.off_bhid = L.parts * L.part_bytes;
  L.off_bout = L.off_bhid + (uint32_t)((nh > 0 ? nh : 1) * C * 4);
  L.off_scale = L.off_bout + (uint32_t)(L.Nout * 4);  // [0..8) weight multipliers, [8..16) accumulator un-scales per layer
  L.bytes = L.off_scale + 64u;
  L.a_cols = (L.Kin > C ? L.Kin : C) * L.es / 4;
  L.d_cols = L.Nout > C ? L.Nout : C;
  L.tile_cols = L.parts * L.a_cols + L.d_cols;
  return L;
}

// ---- weight image ------------------------------------------------------------------------------------------------
// F16X3 scales (one block): layer l = 0 (input), 1..nh (hidden), nh+1 (output): multiplier 2^k with max |W| 2^k in
// [2^14, 2^15) and the accumulator un-scale 2^-k (/ TC_ACT_SCALE for the layers fed by hidden activations).
static __global__ void tc_scales_kernel(const lrds_mlp w, const TcLayout L, uint8_t* __restrict__ img) {
  __shared__ float red[32];
  float* sc = reinterpret_cast<float*>(img + L.off_scale);
  for (int l = 0; l < L.nh + 2; ++l) {
    const float* p = l == 0 ? w.w_in_t : (l <= L.nh ? w.w_hid_t + (int64_t)(l - 1) * C * C : w.w_out_t);
    const int n = l == 0 ? w.d * C : (l <= L.nh ? C * C : C * w.d_pad);
    float m = 0.f;
    for (int i = threadIdx.x; i < n; i += blockDim.x) m = fmaxf(m, fabsf(p[i]));
    m = block_reduce(m, MaxOp{}, 0.f, red);
    if (threadIdx.x == 0) {
      const int k = pow2_exponent_for(m);
      sc[l] = ldexpf(1.0f, k);
      sc[8 + l] = ldexpf(1.0f, -k) / (l == 0 ? 1.0f : TC_ACT_SCALE);
    }
  }
}

// B operand of layer (N x K, K-major, no swizzle): 16-byte K chunk kc of row n at  kc * N * 16 + n * 16.
static __global__ void pack_tc_image_kernel(const lrds_mlp w, const TcLayout L, uint8_t* __restrict__ img) {
  const int E = 16 / L.es;
  const int n_in = C * L.Kin, n_hid = L.nh * C * C, n_out = L.Nout * C;
  const int total = n_in + n_hid + n_out;
  const float* sc = reinterpret_cast<const float*>(img + L.off_scale);  // written by tc_scales_kernel (F16X3)
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
    float v;
    uint32_t off;
    int n, k, N, layer;
    if (idx < n_in) {
      n = idx / L.Kin; k = idx % L.Kin; N = C; off = L.off_in; layer = 0;
      v = k < w.d ? w.w_in_t[(int64_t)k * C + n] : 0.f;
    } else if (idx < n_in + n_hid) {
      const int r = idx - n_in, l = r / (C * C);
      n = (r / C) % C; k = r % C; N = C; off = L.off_hid + (uint32_t)(l * C * C * L.es); layer = 1 + l;
      v = w.w_hid_t[(int64_t)l * C * C + (int64_t)k * C + n];
    } else {
      const int r = idx - n_in - n_hid;
      n = r / C; k = r % C; N = L.Nout; off = L.off_out; layer = L.nh + 1;
      v = n < w.d_pad ? w.w_out_t[(int64_t)k * w.d_pad + n] : 0.f;
    }
    const uint32_t byte = off + (uint32_t)(k / E) * N * 16u + (uint32_t)n * 16u + (uint32_t)(k % E) * L.es;
    if (L.prec == LRDS_PRECISION_BF16) {
      *reinterpret_cast<uint16_t*>(img + byte) = (uint16_t)(ptx::pack_bf16x2(v, 0.f) & 0xFFFFu);
    } else if (L.prec == LRDS_PRECISION_F16X3) {
      put_hi_lo(img, L.part_bytes, byte, v * sc[layer]);  // exact scaling (power of two)
    } else {
      const float hi = ptx::to_tf32(v);
      *reinterpret_cast<float*>(img + byte) = hi;
      if (L.parts == 2) *reinterpret_cast<float*>(img + L.part_bytes + byte) = ptx::to_tf32(v - hi);
    }
  }
  float* bh = reinterpret_cast<float*>(img + L.off_bhid);
  float* bo = reinterpret_cast<float*>(img + L.off_bout);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < (L.nh > 0 ? L.nh : 1) * C; i += gridDim.x * blockDim.x)
    bh[i] = i < L.nh * C ? w.b_hid[i] : 0.f;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < L.Nout; i += gridDim.x * blockDim.x)
    bo[i] = i < w.d_pad ? w.b_out[i] : 0.f;
}

// ---- the tile protocol ----------------------------------------------------------------------------------------------
// D[dcol] (+)= A . B on the tensor core: A in TMEM (hi at a_hi, lo at a_lo, a_step columns per K step), B in shared
// memory (hi image at b, lo image at b + b_part, b_step bytes per K step, K-major descriptors with strides lbo / sbo).
// X3: three passes of (hi, lo) products, small terms first (lo.hi, hi.lo, hi.hi); otherwise the single hi.hi pass.
// UNROLL unrolls the pass loop: the issuer's instruction stream of the throughput kernels is on their critical path.
template <bool X3, bool UNROLL, bool TF32 = false>
__device__ __forceinline__ void mma_passes(uint32_t dcol, uint32_t a_hi, uint32_t a_lo, uint32_t a_step, uint32_t b, uint32_t b_part,
                                           uint32_t b_step, uint32_t lbo, uint32_t sbo, int ksteps, uint32_t idesc) {
  uint32_t acc = 0;
#pragma unroll(UNROLL ? 3 : 1)
  for (int pass = X3 ? 0 : 2; pass < 3; ++pass) {
    const uint32_t a = pass == 0 ? a_lo : a_hi;
    const uint32_t bb = b + (pass == 1 ? b_part : 0u);
    for (int ks = 0; ks < ksteps; ++ks) {
      const uint64_t bdesc = ptx::make_smem_desc(bb + (uint32_t)ks * b_step, lbo, sbo);
      if (TF32) ptx::mma_tf32_ts(dcol, a + (uint32_t)ks * a_step, bdesc, idesc, acc);
      else ptx::mma_bf16_ts(dcol, a + (uint32_t)ks * a_step, bdesc, idesc, acc);  // kind::f16 (bf16 or fp16 per idesc)
      acc = 1;
    }
  }
}

// CTA prologue of the tensor-core kernels.  Warp 0 allocates `tmem_cols` TMEM columns; thread 0 initialises the nbars
// mbarriers behind the weight image and nsbar more at `sbar` (one arrival each) and zeroes the ncnt hand-off counters
// at `cnts`.  After the fences and the CTA barrier thread 0 stages the weight image on bars[0], which also expects
// `extra_bytes` of the kernel's own bulk copies, issued by extra().  Returns the TMEM address once bars[0] completes.
template <class F>
__device__ __forceinline__ uint32_t tc_cta_begin(uint8_t* smem, const TcLayout& TL, const uint8_t* image, uint32_t tmem_cols,
                                                  int warp, int nbars, uint64_t* sbar, int nsbar, uint32_t* cnts, int ncnt,
                                                  uint32_t extra_bytes, F&& extra) {
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + TL.bytes);
  uint32_t* slot = reinterpret_cast<uint32_t*>(smem + TL.bytes + 48);
  if (warp == 0) ptx::tmem_alloc(slot, tmem_cols);
  if (threadIdx.x == 0) {
    for (int i = 0; i < nbars; ++i) ptx::mbar_init(bars + i, 1);
    for (int i = 0; i < nsbar; ++i) ptx::mbar_init(sbar + i, 1);
    for (int i = 0; i < ncnt; ++i) cnts[i] = 0u;
    ptx::fence_mbar_init();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  if (threadIdx.x == 0) {  // drift weights staged once per CTA by the TMA engine
    ptx::mbar_expect_tx(bars, TL.bytes + extra_bytes);
    ptx::bulk_g2s(smem, image, TL.bytes, bars);
    extra();
  }
  ptx::mbar_wait(bars, 0);
  return *slot;
}
// CTA epilogue: every warp is done with the tensor memory, warp 0 frees it
__device__ __forceinline__ void tc_cta_end(int warp, uint32_t tmem, uint32_t tmem_cols) {
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 0) ptx::tmem_dealloc(tmem, tmem_cols);
}

// ---- the policy --------------------------------------------------------------------------------------------------
template <int PREC>
struct TcMlp {
  static constexpr bool kX3 = tc_is_x3(PREC);
  static constexpr bool kHalf = tc_is_half(PREC);
  static constexpr bool kF16 = PREC == LRDS_PRECISION_F16X3;
  static constexpr bool kPipe = tc_max_warps(PREC) <= 8;  // 255-register kernels prefetch their mixture operands
  TcLayout L;
  const uint8_t* img;   // weight image in shared memory
  uint32_t img_s;       // its shared-window address
  uint32_t tm_tile;     // TMEM address of the tile's column 0 at lane 0 (MMA operands)
  uint32_t tm_lane;     // the same at this warp's first lane (tcgen05.ld / st)
  uint64_t* bar;        // the tile's MMA-completion mbarrier
  uint32_t phase;
  uint32_t* cnt;        // the tile's hand-off counter: one increment per warp and hand-off
  uint32_t target;      // its value once every warp of the tile has arrived for the current hand-off
  uint32_t tile_warps;  // warps that take part in a hand-off
  uint32_t issue_mask;  // bit (n & 1): this warp issues the tile's hand-offs n with that parity (warp-uniform)
  uint32_t hand;        // hand-offs so far
  int dp;               // columns of x held by the body (d rounded up to 8, zero padded)
  float vmax = 0.f, xmax = 0.f;  // F16X3: largest hidden pre-activation / |coordinate| this thread has converted to fp16
  __device__ __forceinline__ bool saturated() const { return kF16 && (vmax > F16X3_MAX_PREACT || xmax > F16X3_MAX_COORD); }

  // The tile's fields: TMEM address of its column 0, this warp, the tile's MMA mbarrier and hand-off counter, the
  // warps that take part in a hand-off and the hand-offs this warp issues (issue_mask)
  __device__ __forceinline__ void init(const TcLayout& TL, const uint8_t* smem, uint32_t tmem_tile, int warp, uint64_t* tile_bar,
                                       uint32_t* tile_cnt, uint32_t warps, uint32_t mask, int d_pad) {
    L = TL;
    img = smem;
    img_s = ptx::smem_u32(smem);
    tm_tile = tmem_tile;
    tm_lane = tmem_tile + ((uint32_t)((warp & 3) * 32) << 16);
    bar = tile_bar;
    phase = 0;
    cnt = tile_cnt;
    target = 0u;
    tile_warps = warps;
    issue_mask = mask;
    hand = 0u;
    dp = d_pad;
  }

  // (hi, lo) operand bits of an activation.  The 3-pass splits truncate (one LOP3): hi = the top 11 significand bits,
  // lo = v - hi is exact in fp32; the tf32 tensor core drops lo's bits below tf32 itself, the fp16 conversion rounds
  // them (error 2^-22 of v either way).  The one-pass tf32 mode rounds.
  static __device__ __forceinline__ uint32_t split_hi(float v) {
    if (kX3) return __float_as_uint(v) & 0xFFFFE000u;
    return __float_as_uint(ptx::to_tf32(v));
  }
  __device__ __forceinline__ uint32_t a_col(int part) const { return (uint32_t)(part * L.a_cols); }
  __device__ __forceinline__ uint32_t d_col() const { return (uint32_t)(L.parts * L.a_cols); }
  __device__ __forceinline__ float unscale(int layer) const {  // F16X3: accumulator -> pre-activation
    return reinterpret_cast<const float*>(img + L.off_scale)[8 + layer];
  }

  // This warp's part of the tile's next batch is in place (A rows stored / accumulator rows read).  Every warp
  // increments the tile's counter (release, no round trip) and goes on; the hand-off's issuer warp polls the counter,
  // issues the batch `f` from warp-uniform registers and commits it to the tile's mbarrier.  Nobody else blocks here:
  // the warps wait for the batch on the mbarrier when they need its result.  Which warps issue is the kernel's choice
  // (issue_mask): the throughput kernels let the warps of the least loaded SM sub-partitions take turns.
  // `done` = the mbarrier the batch commits to (default: the tile's; a batch that completes while the tile already
  // works on the next one needs its own, or the tile's barrier would run two phases ahead of a waiter)
  template <class F>
  __device__ __forceinline__ void arrive_issue(F&& f, uint64_t* done = nullptr) {
    ptx::tmem_wait_st();
    ptx::tc_fence_before();
    __syncwarp();
    if ((threadIdx.x & 31) == 0) ptx::red_add_release(cnt, 1u);
    const bool mine = (issue_mask >> (hand & 1u)) & 1u;
    ++hand;
    if (mine) issue_when_ready(f, done);
    else target += tile_warps;
  }
  // polls the tile's counter until every warp has arrived for the next hand-off, then issues and commits its batch
  template <class F>
  __device__ __forceinline__ void issue_when_ready(F&& f, uint64_t* done = nullptr) {
    target += tile_warps;
    while ((int32_t)(ptx::ld_acquire(cnt) - target) < 0) {
    }
    ptx::tc_fence_after();
    if (ptx::elect_one()) {
      f();
      ptx::mma_commit(done ? done : bar);
    }
    __syncwarp();
  }

  // one layer of the network: D = A . W^T
  __device__ __forceinline__ void gemm(uint32_t b_off, int K, int N) const {
    const uint32_t idesc = PREC == LRDS_PRECISION_BF16 ? ptx::make_idesc_bf16(128, N)
                           : kF16                      ? ptx::make_idesc_f16(128, N)
                                                       : ptx::make_idesc_tf32(128, N);
    mma_passes<kX3, true, !kHalf>(tm_tile + d_col(), tm_tile + a_col(0), tm_tile + a_col(1), 8u, img_s + b_off, L.part_bytes,
                                  2u * (uint32_t)N * 16u, (uint32_t)N * 16u, 128u, K / L.kstep, idesc);  // two 16-byte K chunks per MMA
  }
  // the same at the tile's next hand-off
  __device__ __forceinline__ void issue(uint32_t b_off, int K, int N) {
    arrive_issue([&]() { gemm(b_off, K, N); });
  }
  __device__ __forceinline__ void wait() {
    ptx::mbar_wait(bar, phase);
    phase ^= 1u;
    ptx::tc_fence_after();
  }

  // A operand <- 8 consecutive fp32 values (columns c0 .. c0+7 of the K axis), tf32 kinds
  __device__ __forceinline__ void store8(int c0, const float (&v)[8]) {
    uint32_t hi[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) hi[i] = split_hi(v[i]);
    ptx::tmem_st8(tm_lane + a_col(0) + c0, hi);
    if (kX3) {
      uint32_t lo[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) lo[i] = __float_as_uint(v[i] - __uint_as_float(hi[i]));
      ptx::tmem_st8(tm_lane + a_col(1) + c0, lo);
    }
  }
  // A operand <- 16 consecutive fp32 values as 8 packed columns c0 .. c0+7, 16-bit kinds
  __device__ __forceinline__ void store16_half(int c0, const float (&v)[16]) {
    uint32_t r[8];
    if (kF16) {
      uint32_t rl[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        u64 hi, lo;
        xmax = max3abs(xmax, v[2 * i], v[2 * i + 1]);
        f2::split(f2::pack(v[2 * i], v[2 * i + 1]), hi, lo);
        float h0, h1, l0, l1;
        f2::unpack(hi, h0, h1);
        f2::unpack(lo, l0, l1);
        r[i] = ptx::pack_f16x2(h0, h1);
        rl[i] = ptx::pack_f16x2(l0, l1);
      }
      ptx::tmem_st8(tm_lane + a_col(0) + c0, r);
      ptx::tmem_st8(tm_lane + a_col(1) + c0, rl);
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i) r[i] = ptx::pack_bf16x2(v[2 * i], v[2 * i + 1]);
      ptx::tmem_st8(tm_lane + a_col(0) + c0, r);
    }
  }

  // A operand <- x: this thread's groups g0, g0 + gstep, ... of 8 columns (16 dims packed in the 16-bit kinds, 8 dims in
  // the tf32 kinds, where Kin == dp); the default stores all of x
  __device__ __forceinline__ void store_x(const Col4& x, int g0 = 0, int gstep = 1) {
    if (kHalf) {
      for (int c0 = 8 * g0; c0 < L.Kin / 2; c0 += 8 * gstep) {
        float v[16];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int j0 = 2 * c0 + 8 * h;
          float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
          if (j0 < dp) {
            a = x.ld4(j0 >> 2);
            b = x.ld4((j0 >> 2) + 1);
          }
          v[8 * h + 0] = a.x; v[8 * h + 1] = a.y; v[8 * h + 2] = a.z; v[8 * h + 3] = a.w;
          v[8 * h + 4] = b.x; v[8 * h + 5] = b.y; v[8 * h + 6] = b.z; v[8 * h + 7] = b.w;
        }
        store16_half(c0, v);
      }
    } else {
      for (int c0 = 8 * g0; c0 < L.Kin; c0 += 8 * gstep) {
        const float4 a = x.ld4(c0 >> 2), b = x.ld4((c0 >> 2) + 1);
        const float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
        store8(c0, v);
      }
    }
  }

  // F16X3: accumulator columns [c_begin, c_end), W (32 or 16) at a time, * un-scale + bias -> GELU -> A operand of the
  // next layer, on packed fp32x2 arithmetic
  template <bool GLOBAL_BIAS, int W = 32>
  __device__ __forceinline__ void epilogue_f16(const float* __restrict__ bias, int layer, int c_begin = 0, int c_end = C) {
    static_assert(W == 32 || W == 16, "tcgen05.ld / st widths");
    const u64 us2 = f2::pk(unscale(layer));
#pragma unroll 1
    for (int c0 = c_begin; c0 < c_end; c0 += W) {
      uint32_t r[W];
      if constexpr (W == 32) ptx::tmem_ld32(tm_lane + d_col() + c0, r);
      else ptx::tmem_ld16(tm_lane + d_col() + c0, r);
      ptx::tmem_wait_ld();
      const float4* b4 = reinterpret_cast<const float4*>(bias + c0);  // warp-uniform, 16-byte aligned
      uint32_t ph[W / 2], pl[W / 2];
#pragma unroll
      for (int i = 0; i < W / 4; ++i) {
        const float4 b = GLOBAL_BIAS ? __ldg(b4 + i) : b4[i];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const u64 acc = f2::pack(__uint_as_float(r[4 * i + 2 * e]), __uint_as_float(r[4 * i + 2 * e + 1]));
          const u64 v = f2::fma(acc, us2, e ? f2::pack(b.z, b.w) : f2::pack(b.x, b.y));
          {
            float va, vb;
            f2::unpack(v, va, vb);
            vmax = max3(vmax, va, vb);
          }
          const u64 g = gelu_pair(v, 5.0f, TC_ACT_SCALE);  // TC_ACT_SCALE / 2 = 2^5
          u64 hi, lo;
          f2::split(g, hi, lo);
          float h0, h1, l0, l1;
          f2::unpack(hi, h0, h1);
          f2::unpack(lo, l0, l1);
          ph[2 * i + e] = ptx::pack_f16x2(h0, h1);
          pl[2 * i + e] = ptx::pack_f16x2(l0, l1);
        }
      }
      if constexpr (W == 32) {
        ptx::tmem_st16(tm_lane + a_col(0) + c0 / 2, ph);
        ptx::tmem_st16(tm_lane + a_col(1) + c0 / 2, pl);
      } else {
        ptx::tmem_st8(tm_lane + a_col(0) + c0 / 2, ph);
        ptx::tmem_st8(tm_lane + a_col(1) + c0 / 2, pl);
      }
    }
  }

  // accumulator (64 columns) [* un-scale] + bias -> GELU -> A operand of the next layer
  template <bool GLOBAL_BIAS>
  __device__ __forceinline__ void epilogue(const float* __restrict__ bias, int layer) {
    if constexpr (kF16) {
      epilogue_f16<GLOBAL_BIAS>(bias, layer);
    } else {
#pragma unroll 1
      for (int c0 = 0; c0 < C; c0 += 32) {
        uint32_t r[32];
        ptx::tmem_ld32(tm_lane + d_col() + c0, r);
        ptx::tmem_wait_ld();
        float g[32];
        const float4* b4 = reinterpret_cast<const float4*>(bias + c0);  // warp-uniform, 16-byte aligned
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 b = GLOBAL_BIAS ? __ldg(b4 + i) : b4[i];
          gelu_exact2(__uint_as_float(r[4 * i + 0]) + b.x, __uint_as_float(r[4 * i + 1]) + b.y, g[4 * i + 0], g[4 * i + 1]);
          gelu_exact2(__uint_as_float(r[4 * i + 2]) + b.z, __uint_as_float(r[4 * i + 3]) + b.w, g[4 * i + 2], g[4 * i + 3]);
        }
        if (kHalf) {
          float lo16[16], hi16[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) { lo16[i] = g[i]; hi16[i] = g[16 + i]; }
          store16_half(c0 / 2, lo16);
          store16_half(c0 / 2 + 8, hi16);
        } else {
          uint32_t hi[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) hi[i] = split_hi(g[i]);
          ptx::tmem_st32(tm_lane + a_col(0) + c0, hi);
          if (kX3) {
#pragma unroll
            for (int i = 0; i < 32; ++i) hi[i] = __float_as_uint(g[i] - __uint_as_float(hi[i]));
            ptx::tmem_st32(tm_lane + a_col(1) + c0, hi);
          }
        }
      }
    }
  }

  // BIAS_SH: the table row holding bias1 has been staged in shared memory
  template <bool BIAS_SH>
  __device__ __forceinline__ void hidden(const float* __restrict__ bias1, const Col4& x) {
    store_x(x);
    issue(L.off_in, L.Kin, C);
    const float* bh = reinterpret_cast<const float*>(img + L.off_bhid);
    for (int l = 0; l < L.nh; ++l) {
      wait();
      if (l == 0) epilogue<!BIAS_SH>(bias1, 0);
      else epilogue<false>(bh + (l - 1) * C, l);
      issue(L.off_hid + (uint32_t)(l * C * C * L.es), C, C);
    }
    wait();
    if (L.nh == 0) epilogue<!BIAS_SH>(bias1, 0);
    else epilogue<false>(bh + (L.nh - 1) * C, L.nh);
    issue(L.off_out, C, L.Nout);
    wait();
  }

  // the same as four (dim 2q, dim 2q+1) pairs (F16X3)
  __device__ __forceinline__ void out_chunk2(int j0, u64 (&out)[JC / 2]) {
    uint32_t r[8];
    ptx::tmem_ld8(tm_lane + d_col() + j0, r);
    ptx::tmem_wait_ld();
    const ulonglong2* b2 = reinterpret_cast<const ulonglong2*>(img + L.off_bout + j0 * 4);
    const ulonglong2 a = b2[0], b = b2[1];
    const u64 us2 = f2::pk(unscale(L.nh + 1));
    out[0] = f2::fma(f2::pack(__uint_as_float(r[0]), __uint_as_float(r[1])), us2, a.x);
    out[1] = f2::fma(f2::pack(__uint_as_float(r[2]), __uint_as_float(r[3])), us2, a.y);
    out[2] = f2::fma(f2::pack(__uint_as_float(r[4]), __uint_as_float(r[5])), us2, b.x);
    out[3] = f2::fma(f2::pack(__uint_as_float(r[6]), __uint_as_float(r[7])), us2, b.y);
  }

  __device__ __forceinline__ void out_chunk(int j0, float (&out)[JC]) {
    uint32_t r[8];
    ptx::tmem_ld8(tm_lane + d_col() + j0, r);
    ptx::tmem_wait_ld();
    const float4* b4 = reinterpret_cast<const float4*>(img + L.off_bout + j0 * 4);
    const float4 a = b4[0], b = b4[1];
    const float bs[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    if (kF16) {
      const float us = unscale(L.nh + 1);
#pragma unroll
      for (int c = 0; c < 8; ++c) out[c] = fmaf(__uint_as_float(r[c]), us, bs[c]);
    } else {
#pragma unroll
      for (int c = 0; c < 8; ++c) out[c] = __uint_as_float(r[c]) + bs[c];
    }
  }
};

__host__ __device__ inline uint32_t tc_stage_bytes(const lrds_spec& s, int level) {
  return level > 0 ? (stage_layout(s, level).total + 15u) & ~15u : 0u;
}

// ---- kernel --------------------------------------------------------------------------------------------------------
// shared memory: [weight image | mbarriers + TMEM slot | operand stage (STAGED) | particle columns]
template <int KIND, int PREC, int STAGE, class TR>
__global__ void __launch_bounds__(tc_max_warps(PREC) * 32, 1)
rollout_tc_kernel(const RolloutArgs a, const uint8_t* __restrict__ image, const uint32_t tmem_cols) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  const TcLayout TL = tc_layout(a.s.d, a.s.mlp.num_hidden, PREC);
  const int tid = threadIdx.x, warp = tid >> 5, nwarps = blockDim.x >> 5;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + TL.bytes);  // [0] image, [1 + t] tile t
  uint32_t* cnts = reinterpret_cast<uint32_t*>(smem_raw + TL.bytes + 64);  // [t] hand-offs of tile t
  uint8_t* stage = smem_raw + TL.bytes + TC_TAIL_BYTES;
  float* cols = reinterpret_cast<float*>(stage + tc_stage_bytes(a.s, STAGE));
  const uint32_t tmem = tc_cta_begin(smem_raw, TL, image, tmem_cols, warp, 5, nullptr, 0, cnts, 4, 0u, []() {});
  const int tile = warp >> 2;
  const int tile_warps = min(4, nwarps - 4 * tile);
  TcMlp<PREC> mlp;
  // the tile's last warp issues its batches: its sub-partition carries the fewest warps
  mlp.init(TL, smem_raw, tmem + (uint32_t)(tile * TL.tile_cols), warp, bars + 1 + tile, cnts + tile, (uint32_t)tile_warps,
           (warp & 3) == tile_warps - 1 ? 3u : 0u, a.s.mlp.d_pad);
  rollout_body<KIND, STAGE, TR>(a, cols, stage, mlp);
  tc_cta_end(warp, tmem, tmem_cols);
}

// ---- host side -------------------------------------------------------------------------------------------------------
struct TcPlan {
  int warps, grid, staged;
  uint32_t tmem_cols;
  size_t smem;
};

// Warps per CTA (one CTA per SM, at most wmax warps) for `need` particle warps: as few waves as possible over the
// SMs, then as few idle lanes as possible
inline int plan_warps(int need, int sms, int wmax) {
  const int waves = (need + sms * wmax - 1) / (sms * wmax);
  const int w = (need + sms * waves - 1) / (sms * waves);
  return w < 1 ? 1 : (w > wmax ? wmax : w);
}
// TMEM columns to allocate for `cols` used ones: a power of two, at least 32
inline uint32_t plan_tmem_cols(int cols) {
  uint32_t c = 32;
  while ((int)c < cols) c <<= 1;
  return c;
}

// Launches a tensor-core rollout kernel (arguments: the rollout, the weight image, then `args`) with the plan's grid and
// shared memory and `threads` threads per CTA; `what` names the kernel in the error message.
template <class K, class... A>
int launch_tc(K kernel, const char* what, const RolloutArgs& a, const TcPlan& p, int threads, cudaStream_t st, A... args) {
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem);
  if (e == cudaSuccess) {
    kernel<<<p.grid, threads, p.smem, st>>>(a, static_cast<const uint8_t*>(a.s.mlp.tc_image), args...);
    e = cudaGetLastError();
  }
  if (e != cudaSuccess)
    return cuda_fail(e, "%s launch (grid %d x %d threads, %zu B smem, %u TMEM cols)", what, p.grid, threads, p.smem, p.tmem_cols);
  return LRDS_OK;
}

// Operand staging (LINEAR kind) is used when its shared-memory cost does not reduce the warps per CTA.
inline int plan_rollout_tc(const lrds_spec& s, int smem_cap, int sms, TcPlan* out, const char** why) {
  const TcLayout TL = tc_layout(s.d, s.mlp.num_hidden, s.precision);
  const ColLayout CL = col_layout(s);
  const size_t fixed = (size_t)TL.bytes + TC_TAIL_BYTES;
  const size_t per_warp = (size_t)CL.total * 32 * sizeof(float);
  if (TL.tile_cols > 512) { *why = "TMEM columns of one tile exceed 512"; return LRDS_ERR_RESOURCES; }
  if (fixed + per_warp > (size_t)smem_cap) { *why = "weight image + one warp of particle state exceed shared memory"; return LRDS_ERR_RESOURCES; }
  const int tmax = 512 / TL.tile_cols;
  const int need = (s.B + 31) / 32;
  auto pick = [&](size_t extra) {
    if (fixed + extra + per_warp > (size_t)smem_cap) return 0;
    int wmax = (int)(((size_t)smem_cap - fixed - extra) / per_warp);
    wmax = wmax < tc_max_warps(s.precision) ? wmax : tc_max_warps(s.precision);
    wmax = wmax < 4 * tmax ? wmax : 4 * tmax;
    return plan_warps(need, sms, wmax);
  };
  const int w_plain = pick(0);
  int level = 0, w = w_plain;
  size_t stage = 0;
  if (s.kind == LRDS_ROLLOUT_LINEAR) {
    for (int lv = 2; lv >= 1; --lv) {  // the deepest staging level that does not cost warps
      const size_t bytes = tc_stage_bytes(s, lv);
      const int wl = pick(bytes);
      if (wl >= w_plain) { level = lv; w = wl; stage = bytes; break; }
    }
  }
  const bool staged = level > 0;
  out->warps = w;
  out->grid = (need + w - 1) / w;
  out->staged = level;
  out->tmem_cols = plan_tmem_cols((w + 3) / 4 * TL.tile_cols);
  out->smem = fixed + (staged ? stage : 0) + per_warp * w;
  return LRDS_OK;
}

}  // namespace lrds
