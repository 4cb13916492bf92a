// Parameter gradient of the drift network over all stored states of a rollout: the batched pass of the
// log-variance objectives (sde_sampler/losses/oc.py:105-131 through 364-394 / 830-860: autograd through
// FourierMLP.forward, models/mlp.py:135-143, under the clip of ClippedCtrl, models/reparam.py:33-43).
//
//   rows r = (s, b):   v_1 = W_in x_r + bias1[s]            g_l = GELU(v_l)
//                      v_{l+1} = W_l g_l + b_l              net = W_out g_{nh+1} + b_out
//   given cot_r = d loss / d clip(net_r):   delta_net = cot_r [|net_r| <= clip],  delta_l = (delta_{l+1} W_l) GELU'(v_l)
//   wanted:   dW_out = sum_r delta_net g_{nh+1}^T,  dW_l = sum_r delta_{l+1} g_l^T,  dW_in = sum_r delta_1 x_r^T,
//             the bias sums, and  dbias1[s] = sum_b delta_1  (the cotangent of TimeEmbed + input bias)
//
// One CTA per SM walks over tiles of 128 rows (four threads <-> row <-> TMEM lane; they split the columns in quarters).
// Per tile the activations are recomputed on the tensor cores exactly like the rollout does (fp16 (hi, lo) 3-pass
// GEMMs, A operand in TMEM, the rollout's own weight image as B), GELU' is kept in TMEM, the backward-data GEMMs read
// the SAME weight image as an MN-major B operand (contraction over the image's rows), and the weight gradients are
// GEMMs whose contraction index is the row: both operands come from shared memory in MN-major layout
//     A = [g_l | 1]  (features + a block of ones: its accumulator row is the bias gradient),   B = delta_{l+1}
// and accumulate in TMEM (fp32) over ALL tiles of the CTA; the accumulators are written once per CTA and summed over
// the CTAs in a fixed order by a second kernel (run-to-run deterministic, no atomics).
//
// Precision: forward and backward-data products are fp32-grade (3-pass); the weight-gradient operands are single fp16
// roundings (relative 2^-12 per product, unbiased, averaged over >= 10^5 rows), the cotangents scaled by a power of two
// (`cot_scale`, chosen by the caller so that max |cot| cot_scale ~ 4) to sit in fp16's normal range.
#include <cuda_fp16.h>

#include "lrds_internal.h"
#include "lrds_mlp_tc.cuh"

namespace lrds {

struct MgLayout {
  uint32_t tail, xbuf, gbuf, gstride, dbuf, xstage, cstage, bytes;
};
__host__ __device__ inline MgLayout mg_layout(const TcLayout& TL, int d, bool staged) {
  MgLayout M;
  M.tail = TL.bytes;
  M.xbuf = (TL.bytes + TC_TAIL_BYTES + 127u) & ~127u;
  M.gbuf = M.xbuf + (uint32_t)(TL.Kin / 8) * MG_GROUP;
  M.gstride = 9u * MG_GROUP;  // 8 feature groups + the block of ones
  M.dbuf = M.gbuf + (uint32_t)(TL.nh + 1) * M.gstride;
  M.xstage = M.dbuf + 8u * MG_GROUP;  // an A operand spans 16 groups from its start: always inside [xbuf, xstage)
  // one tile's rows of x / of the cotangents, as in global memory (left out when they do not fit: d > 56)
  const uint32_t stage = staged ? (128u * (uint32_t)d * 4u + 127u) & ~127u : 0u;
  M.cstage = M.xstage + stage;
  M.bytes = M.cstage + stage;
  return M;
}

// Optional phase timers (-DLRDS_MG_TIMING, tools/mlp_grad_timing.py only): threads 0 and 32 of CTA 0 accumulate the cycles
// between the marks of the tile loop.
#ifdef LRDS_MG_TIMING
__device__ unsigned long long g_mg_timing[2 * 24];
#define MG_MARK(i)                                              \
  do {                                                          \
    if (tm_on) {                                                \
      const long long now_ = clock64();                         \
      tm_acc[i] += (unsigned long long)(now_ - tm_last);        \
      tm_last = now_;                                           \
    }                                                           \
  } while (0)
#else
#define MG_MARK(i) do { } while (0)
#endif

struct MlpGradArgs {
  lrds_mlp mlp;
  const float* bias1;   // [S][64]
  const float* x;       // [S][B][d]
  const float* cot;     // [S][B][d]
  const float* step_w;  // [S] or null: cot is multiplied by step_w[s] row_w[b]
  const float* row_w;   // [B] or null
  float clip, cot_scale;
  const float* cot_scale_dev;  // device copy of cot_scale (replaces it when given: no host round trip to choose it)
  int S, B, tiles_per_s;
  int64_t tiles;
  int staged;         // the tile rows travel through the TMA staging areas
  float* part;        // [grid][P]
  float* dbias_part;  // [tiles * 4][64]
  int P;
};

__global__ void __launch_bounds__(MG_THREADS, 1) mlp_grad_kernel(const MlpGradArgs a) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  uint8_t* const smem = smem_raw;
  const int d = a.mlp.d, dp = a.mlp.d_pad, nh = a.mlp.num_hidden;
  const TcLayout TL = tc_layout(d, nh, LRDS_PRECISION_F16X3);
  const MgLayout ML = mg_layout(TL, d, a.staged != 0);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, q = warp & 3, h = warp >> 2;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + ML.tail);  // [0] image, [1] MMA batches, [2] x rows, [3] cotangent rows
  uint32_t* slot = reinterpret_cast<uint32_t*>(smem + ML.tail + 48);
  const int64_t t0 = a.tiles * blockIdx.x / gridDim.x, t1 = a.tiles * (blockIdx.x + 1) / gridDim.x;
  float* part = a.part + (int64_t)blockIdx.x * a.P;
  if (t0 >= t1) {  // more CTAs than tiles
    for (int i = tid; i < a.P; i += MG_THREADS) part[i] = 0.f;
    return;
  }
  if (warp == 0) ptx::tmem_alloc(slot, MG_TMEM_COLS);
  if (tid == 0) {
    ptx::mbar_init(bars, 1);
    ptx::mbar_init(bars + 1, 1);
    ptx::mbar_init(bars + 2, 1);
    ptx::mbar_init(bars + 3, 1);
    ptx::fence_mbar_init();
  }
  for (int l = 0; l <= nh; ++l) {  // the blocks of ones behind the activation buffers
    uint4* ones = reinterpret_cast<uint4*>(smem + ML.gbuf + (uint32_t)l * ML.gstride + 8u * MG_GROUP);
    for (int i = tid; i < 128; i += MG_THREADS) ones[i] = make_uint4(0x3C003C00u, 0x3C003C00u, 0x3C003C00u, 0x3C003C00u);
  }
  ptx::fence_proxy_async();
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  if (tid == 0) {
    ptx::mbar_expect_tx(bars, TL.bytes);
    ptx::bulk_g2s(smem, a.mlp.tc_image, TL.bytes, bars);
  }
  ptx::mbar_wait(bars, 0);
  const uint32_t tmem = *slot;
  const uint32_t tm_lane = tmem + ((uint32_t)(q * 32) << 16);
  const uint32_t img_s = ptx::smem_u32(smem);
  const uint32_t xbuf_s = img_s + ML.xbuf, gbuf_s = img_s + ML.gbuf, dbuf_s = img_s + ML.dbuf;
  uint64_t* bar = bars + 1;
  uint32_t phase = 0;
  const float* sc = reinterpret_cast<const float*>(smem + TL.off_scale);
  const float* bhid = reinterpret_cast<const float*>(smem + TL.off_bhid);
  const float* bout = reinterpret_cast<const float*>(smem + TL.off_bout);
  const int rloc = 32 * q + lane;  // row of the tile = TMEM lane
  const int Kin = TL.Kin, Nout = TL.Nout;

  // ---- MMA batches (one elected thread of warp 0) ----
  auto mma_fwd = [&](uint32_t b_off, int K, int N) { mg_mma_fwd(tmem, img_s, TL, b_off, K, N); };
  auto mma_bwd = [&](uint32_t b_off, int Nimg) { mg_mma_bwd(tmem, img_s, TL, b_off, Nimg, C); };
  auto mma_wgrad = [&](uint32_t a_s, uint32_t acc_col, int N, uint32_t accumulate) {  // ACC += A^T delta over the 128 rows
    const uint32_t idesc = ptx::make_idesc_f16(128, N) | ptx::IDESC_A_MN | ptx::IDESC_B_MN;
    for (int ks = 0; ks < 8; ++ks) {
      const uint64_t ad = ptx::make_smem_desc(a_s + (uint32_t)ks * 256u, 128u, MG_GROUP);
      const uint64_t bd = ptx::make_smem_desc(dbuf_s + (uint32_t)ks * 256u, 128u, MG_GROUP);
      ptx::mma_f16_ss(tmem + acc_col, ad, bd, idesc, accumulate | (ks > 0));
    }
  };
  // this thread's 16 columns of delta as the B operand of the weight-gradient GEMM: one fp16 rounding (a second, (hi, lo)
  // operand halves the rounding noise of the weight gradients at +22 % kernel time: measured, not kept)
  auto store_delta = [&](const float (&dl)[16]) {
    uint32_t pr[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) pr[i] = ptx::pack_f16x2(dl[2 * i], dl[2 * i + 1]);
    uint8_t* db8 = smem + ML.dbuf + (uint32_t)(2 * h) * MG_GROUP + (uint32_t)rloc * 16u;
    *reinterpret_cast<uint4*>(db8) = make_uint4(pr[0], pr[1], pr[2], pr[3]);
    *reinterpret_cast<uint4*>(db8 + MG_GROUP) = make_uint4(pr[4], pr[5], pr[6], pr[7]);
  };
  auto hand = [&](auto&& issue) {  // operands stored -> the batch is issued and committed to `bar`
    ptx::fence_proxy_async();
    ptx::tmem_wait_st();
    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 0) {
      if (ptx::elect_one()) {
        ptx::tc_fence_after();
        issue();
        ptx::mma_commit(bar);
      }
      __syncwarp();
    }
  };
  auto wait = [&]() {
    ptx::mbar_wait(bar, phase);
    phase ^= 1u;
    ptx::tc_fence_after();
  };

  const float cot_scale = a.cot_scale_dev ? __ldg(a.cot_scale_dev) : a.cot_scale;
  const float inv_cs = 1.0f / cot_scale;
  bool first = true, pending = false;
#ifdef LRDS_MG_TIMING
  const bool tm_on = blockIdx.x == 0 && (tid == 0 || tid == 32);
  unsigned long long tm_acc[24] = {};
  long long tm_last = clock64();
#endif
  // The rows of a tile are contiguous in global memory (128 x d floats): the TMA engine copies them into shared memory one
  // stage ahead (x of tile t + 1 while tile t runs, its cotangents behind tile t's output stage) and every thread picks
  // its 16 values from there - per-thread global loads of rows 4 d bytes apart cost 32 wavefronts each.  Tiles that are
  // ragged (the last of a time slice) or not 16-byte aligned in global memory take the per-thread loads.
  const uint32_t stage_bytes = 128u * (uint32_t)d * 4u;
  const float* xs = reinterpret_cast<const float*>(smem + ML.xstage);
  const float* cs = reinterpret_cast<const float*>(smem + ML.cstage);
  uint32_t phx = 0, phc = 0;
  auto tile_row0 = [&](int64_t tile) { return (tile / a.tiles_per_s) * (int64_t)a.B + (tile % a.tiles_per_s) * 128; };
  auto tile_fast = [&](int64_t tile) -> bool {
    if (!a.staged || (int)(tile % a.tiles_per_s) * 128 + 128 > a.B) return false;
    const int64_t e0 = tile_row0(tile) * d;
    return ((reinterpret_cast<uintptr_t>(a.x + e0) | reinterpret_cast<uintptr_t>(a.cot + e0)) & 15u) == 0;
  };
  auto fetch = [&](const float* src, uint32_t stage_off, uint64_t* b, int64_t tile) {  // one thread
    ptx::mbar_expect_tx(b, stage_bytes);
    ptx::bulk_g2s(smem + stage_off, src + tile_row0(tile) * d, stage_bytes, b);
  };
  auto load16 = [&](const float* __restrict__ src, int64_t r, bool valid, float (&v)[16]) {
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const int j = 16 * h + i;
      v[i] = (valid && j < d) ? __ldg(src + r * d + j) : 0.f;
    }
  };
  auto pick16 = [&](const float* stage, float (&v)[16]) {
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const int j = 16 * h + i;
      v[i] = j < d ? stage[rloc * d + j] : 0.f;
    }
  };
  if (tid == 0 && tile_fast(t0)) {
    fetch(a.x, ML.xstage, bars + 2, t0);
    fetch(a.cot, ML.cstage, bars + 3, t0);
  }
  float xv[16], cv[16];
  for (int64_t tile = t0; tile < t1; ++tile) {
    const int s = (int)(tile / a.tiles_per_s);
    const int row = (int)(tile % a.tiles_per_s) * 128 + rloc;
    const bool valid = row < a.B;
    const int64_t r = (int64_t)s * a.B + (valid ? row : 0);
    const bool fast = tile_fast(tile), next_fast = tile + 1 < t1 && tile_fast(tile + 1);
    if (fast) {
      ptx::mbar_wait(bars + 2, phx);
      phx ^= 1u;
      pick16(xs, xv);
    } else {
      load16(a.x, r, valid, xv);
    }
    MG_MARK(0);
    if (pending) wait();  // the previous tile's last batch has read its buffers
    MG_MARK(1);
    if (h < Kin / 16) {
      uint32_t ph[8], pl[8], pr[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        split_pack(xv[2 * i], xv[2 * i + 1], ph[i], pl[i]);
        pr[i] = ptx::pack_f16x2(xv[2 * i], xv[2 * i + 1]);
      }
      ptx::tmem_st8(tm_lane + MG_A_HI + 8 * h, ph);
      ptx::tmem_st8(tm_lane + MG_A_LO + 8 * h, pl);
      uint8_t* xb = smem + ML.xbuf + (uint32_t)(2 * h) * MG_GROUP + (uint32_t)rloc * 16u;
      *reinterpret_cast<uint4*>(xb) = make_uint4(pr[0], pr[1], pr[2], pr[3]);
      *reinterpret_cast<uint4*>(xb + MG_GROUP) = make_uint4(pr[4], pr[5], pr[6], pr[7]);
    }
    hand([&] { mma_fwd(TL.off_in, Kin, C); });
    if (tid == 0 && next_fast) fetch(a.x, ML.xstage, bars + 2, tile + 1);  // every thread has picked its x values
    MG_MARK(2);

    // ---- forward: bias + GELU, GELU' to TMEM, the activation to TMEM (next GEMM) and shared memory (its weight gradient) ----
    for (int l = 0; l <= nh; ++l) {
      wait();
      MG_MARK(3 + 2 * l);
      uint32_t pg[8];
      float vmax = 0.f;
      mg_forward_layer<false>(tm_lane, h, l, sc[8 + l],
                              l == 0 ? reinterpret_cast<const float4*>(a.bias1 + (int64_t)s * C + 16 * h)
                                     : reinterpret_cast<const float4*>(bhid + (l - 1) * C + 16 * h),
                              pg, vmax);
      uint8_t* gb8 = smem + ML.gbuf + (uint32_t)l * ML.gstride + (uint32_t)(2 * h) * MG_GROUP + (uint32_t)rloc * 16u;
      *reinterpret_cast<uint4*>(gb8) = make_uint4(pg[0], pg[1], pg[2], pg[3]);
      *reinterpret_cast<uint4*>(gb8 + MG_GROUP) = make_uint4(pg[4], pg[5], pg[6], pg[7]);
      if (l < nh) hand([&] { mma_fwd(TL.off_hid + (uint32_t)(l * C * C * 2), C, C); });
      else hand([&] { mma_fwd(TL.off_out, C, Nout); });
      MG_MARK(4 + 2 * l);
    }

    // ---- output: clip mask and cotangent -> delta_net (16-column block h) ----
    wait();
    MG_MARK(9);
    if (fast) {
      ptx::mbar_wait(bars + 3, phc);
      phc ^= 1u;
      pick16(cs, cv);
    } else {
      load16(a.cot, r, valid, cv);
    }
    if (h < Nout / 16) {
      const float us = sc[8 + nh + 1];
      float wgt = valid ? cot_scale : 0.f;
      if (a.step_w) wgt *= __ldg(a.step_w + s);
      if (a.row_w) wgt *= __ldg(a.row_w + (valid ? row : 0));
      uint32_t rr[16];
      ptx::tmem_ld16(tm_lane + MG_D + 16 * h, rr);
      ptx::tmem_wait_ld();
      float dl[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const int j = 16 * h + i;
        const float net = fmaf(__uint_as_float(rr[i]), us, bout[j]);
        const float c = cv[i] * wgt;
        dl[i] = (a.clip > 0.f && !(fabsf(net) <= a.clip)) ? 0.f : c;
      }
      uint32_t ph[8], pl[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) split_pack(dl[2 * i], dl[2 * i + 1], ph[i], pl[i]);
      ptx::tmem_st8(tm_lane + MG_A_HI + 8 * h, ph);
      ptx::tmem_st8(tm_lane + MG_A_LO + 8 * h, pl);
      store_delta(dl);
    }
    {
      const uint32_t acc0 = first ? 0u : 1u;
      hand([&] {
        mma_wgrad(gbuf_s + (uint32_t)nh * ML.gstride, MG_ACC + 64u * (uint32_t)(nh + 1), Nout, acc0);
        mma_bwd(TL.off_out, Nout);
      });
      if (tid == 0 && next_fast) fetch(a.cot, ML.cstage, bars + 3, tile + 1);
    }
    MG_MARK(10);

    // ---- backward: delta_l = (delta_{l+1} W) GELU'(v_l), l = nh + 1 .. 1 ----
    for (int l = nh + 1; l >= 1; --l) {
      wait();
      MG_MARK(11 + 2 * (nh + 1 - l));
      const float ub = 1.0f / sc[l];  // the layer that consumes g_l (hidden layer l, or the output layer) is scaled by sc[l]
      uint32_t rr[16], gp[8];
      ptx::tmem_ld16(tm_lane + MG_D + 16 * h, rr);
      ptx::tmem_ld8(tm_lane + MG_GP + 32 * (l - 1) + 8 * h, gp);
      ptx::tmem_wait_ld();
      float dl[16];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float2 gd = unpack_gp(gp[i]);
        dl[2 * i] = __uint_as_float(rr[2 * i]) * ub * gd.x;
        dl[2 * i + 1] = __uint_as_float(rr[2 * i + 1]) * ub * gd.y;
      }
      if (l > 1) {
        uint32_t ph[8], pl[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) split_pack(dl[2 * i], dl[2 * i + 1], ph[i], pl[i]);
        ptx::tmem_st8(tm_lane + MG_A_HI + 8 * h, ph);
        ptx::tmem_st8(tm_lane + MG_A_LO + 8 * h, pl);
      }
      store_delta(dl);
      const uint32_t acc0 = first ? 0u : 1u;
      if (l > 1) {
        hand([&] {
          mma_wgrad(gbuf_s + (uint32_t)(l - 2) * ML.gstride, MG_ACC + 64u * (uint32_t)(l - 1), C, acc0);
          mma_bwd(TL.off_hid + (uint32_t)((l - 2) * C * C * 2), C);
        });
      } else {
        hand([&] { mma_wgrad(xbuf_s, MG_ACC, C, acc0); });
        // dbias1 contribution of this warp's 32 rows: column sums of its 16 columns by a reduce-scatter over the lanes
        // (four halvings leave column (lane >> 1) & 15 in every lane, the last exchange adds the two half sums)
#pragma unroll
        for (int stp = 0; stp < 4; ++stp) {
          const int o = 16 >> stp, n = 8 >> stp;
          const bool up = (lane & o) != 0;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            if (i < n) {
              const float send = up ? dl[i] : dl[i + n], keep = up ? dl[i + n] : dl[i];
              dl[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
            }
          }
        }
        dl[0] += __shfl_xor_sync(0xffffffffu, dl[0], 1);
        if ((lane & 1) == 0) a.dbias_part[(tile * 4 + q) * C + 16 * h + (lane >> 1)] = dl[0] * inv_cs;
      }
      MG_MARK(12 + 2 * (nh + 1 - l));
    }
    first = false;
    pending = true;
  }
  if (pending) wait();
#ifdef LRDS_MG_TIMING
  if (tm_on)
    for (int i = 0; i < 24; ++i) g_mg_timing[(tid == 0 ? 0 : 24) + i] = tm_acc[i];
#endif

  // ---- the CTA's accumulators -> its slice of `part` (layout of lrds_mlp: w_in_t, w_hid_t, b_hid, w_out_t, b_out) ----
  {
    const int m = rloc;
    const float inv_w = inv_cs / TC_ACT_SCALE;
    const int o_hid = d * C, o_bhid = o_hid + nh * C * C, o_out = o_bhid + nh * C, o_bout = o_out + C * dp;
    for (int i = 0; i <= nh + 1; ++i) {
      const int ncol = i == nh + 1 ? Nout : C;
      for (int c0 = 8 * h; c0 < ncol; c0 += 32) {
        uint32_t rr[8];
        ptx::tmem_ld8(tm_lane + MG_ACC + 64 * i + c0, rr);
        ptx::tmem_wait_ld();
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const int n = c0 + e;
          const float v = __uint_as_float(rr[e]);
          if (i == 0) {
            if (m < d) part[m * C + n] = v * inv_cs;
          } else if (i <= nh) {
            if (m < C) part[o_hid + (i - 1) * C * C + m * C + n] = v * inv_w;
            else if (m == C) part[o_bhid + (i - 1) * C + n] = v * inv_cs;
          } else if (n < dp) {
            if (m < C) part[o_out + m * dp + n] = v * inv_w;
            else if (m == C) part[o_bout + n] = v * inv_cs;
          }
        }
      }
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 0) ptx::tmem_dealloc(tmem, MG_TMEM_COLS);
}

// blocks [0, ceil(P / 256)): grads[p] = sum over the CTAs' slices;  blocks behind: dbias1[s][c] = sum over the 4 *
// tiles_per_s warp partials of time row s - both in a fixed order
__global__ void __launch_bounds__(256) mlp_grad_reduce_kernel(const float* __restrict__ part, int ncta, int P,
                                                              float* __restrict__ out, const float* __restrict__ dbp,
                                                              int rows_per_s, float* __restrict__ dbias1) {
  const int pblocks = (P + 255) / 256;
  if ((int)blockIdx.x < pblocks) {
    const int p = blockIdx.x * 256 + threadIdx.x;
    if (p >= P) return;
    float acc = 0.f;
    for (int c = 0; c < ncta; ++c) acc += part[(int64_t)c * P + p];
    out[p] = acc;
    return;
  }
  __shared__ float red[4][C];
  const int s = blockIdx.x - pblocks, c = threadIdx.x & (C - 1), g = threadIdx.x >> 6;
  const float* src = dbp + (int64_t)s * rows_per_s * C;
  float acc = 0.f;
  for (int r = g; r < rows_per_s; r += 4) acc += src[(int64_t)r * C + c];
  red[g][c] = acc;
  __syncthreads();
  if (g == 0) dbias1[(int64_t)s * C + c] = (red[0][c] + red[1][c]) + (red[2][c] + red[3][c]);
}

int mlp_grad_params(int d, int nh) {
  const int dp = (d + 7) / 8 * 8;
  return d * C + nh * C * C + nh * C + C * dp + dp;
}

bool mlp_grad_applicable(int d, int nh) { return d >= 1 && d <= 64 && nh >= 0 && nh <= 2; }

int64_t mlp_grad_scratch_floats(int d, int nh, int S, int B) {
  const int64_t tiles = (int64_t)S * ((B + 127) / 128);
  return (int64_t)device_limits().sms * mlp_grad_params(d, nh) + tiles * 4 * C;
}

int launch_mlp_grad(const lrds_mlp& mlp, const float* bias1, const float* x, const float* cot, const float* step_w,
                    const float* row_w, float clip, float cot_scale, const float* cot_scale_dev, int S, int B,
                    float* grads, float* dbias1, float* scratch, cudaStream_t st) {
  if (!mlp_grad_applicable(mlp.d, mlp.num_hidden))
    return fail(LRDS_ERR_UNSUPPORTED, "mlp_grad: built for d <= 64 and at most 2 hidden layers (got d = %d, %d hidden)", mlp.d,
                mlp.num_hidden);
  if (!mlp.tc_image) return fail(LRDS_ERR_INVALID, "mlp_grad: mlp.tc_image (the F16X3 weight image of lrds_pack_mlp_tc) is required");
  MlpGradArgs a{};
  a.mlp = mlp;
  a.bias1 = bias1; a.x = x; a.cot = cot; a.step_w = step_w; a.row_w = row_w;
  a.clip = clip; a.cot_scale = cot_scale; a.cot_scale_dev = cot_scale_dev;
  a.S = S; a.B = B;
  a.tiles_per_s = (B + 127) / 128;
  a.tiles = (int64_t)S * a.tiles_per_s;
  a.P = mlp_grad_params(mlp.d, mlp.num_hidden);
  const DeviceLimits dl = device_limits();
  const int grid = dl.sms;
  a.part = scratch;
  a.dbias_part = scratch + (int64_t)grid * a.P;
  const TcLayout TL = tc_layout(mlp.d, mlp.num_hidden, LRDS_PRECISION_F16X3);
  a.staged = mg_layout(TL, mlp.d, true).bytes <= (uint32_t)dl.smem_optin;
  const MgLayout ML = mg_layout(TL, mlp.d, a.staged != 0);
  cudaError_t e = cudaFuncSetAttribute(mlp_grad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ML.bytes);
  if (e == cudaSuccess) {
    mlp_grad_kernel<<<grid, MG_THREADS, ML.bytes, st>>>(a);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) {
    mlp_grad_reduce_kernel<<<(a.P + 255) / 256 + S, 256, 0, st>>>(a.part, grid, a.P, grads, a.dbias_part,
                                                                  4 * a.tiles_per_s, dbias1);
    e = cudaGetLastError();
  }
  return e == cudaSuccess ? LRDS_OK : cuda_fail(e, "mlp_grad launch (grid %d, %u B smem)", grid, ML.bytes);
}

}  // namespace lrds

#ifdef LRDS_MG_TIMING
extern "C" int lrds_debug_mlp_grad_timing(unsigned long long* host_out) {  // tools only
  return (int)cudaMemcpyFromSymbol(host_out, lrds::g_mg_timing, sizeof(lrds::g_mg_timing));
}
#endif
