// Implicit-GEMM convolution / inner-product on the sm_100a tensor cores.
//
// Replaces, for the MNC inference path, Caffe's Convolution layer
// (caffe-mnc/src/caffe/layers/cudnn_conv_layer.cu:11-54, conv_layer.cu:8-23 +
// util/im2col.cu:9-39) and InnerProduct layer (inner_product_layer.cu:21-27).
//
// Design (B200-first, not a port):
//  * activations live in HBM as NHWC, split into two bf16 planes (hi, lo) with
//    x ~= hi + lo (16 mantissa bits).  Weights likewise, stored [Cout][tap][Cin].
//  * one persistent CTA per SM; warp 0 = TMA producer, warp 1 = MMA issuer
//    (single elected thread, tcgen05.mma), warp 2 owns TMEM, warps 4..7 = epilogue.
//  * im2col is folded into the TMA descriptor: the A tile for filter tap (dy,dx)
//    is the 4-D box [1, TH, TW, 64ch] at (h0+dy, w0+dx); out-of-image rows/cols
//    are zero-filled by TMA, which *is* the conv zero padding.
//  * fp32-class accuracy on bf16 tensor cores: D += Ahi*Bhi + Ahi*Blo + Alo*Bhi
//    (the dropped Alo*Blo term is ~2^-18 relative).  Accumulators are fp32 in
//    TMEM, double-buffered so the epilogue of tile i overlaps the MMAs of tile i+1.
//  * epilogue: tcgen05.ld -> +bias -> ReLU -> re-split to (hi, lo) bf16 NHWC, or
//    raw fp32 (split-K partials / final logits).
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_fp8.h>
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>

#include "mnc_b200.h"
#include "ptx.cuh"
#include "tri.cuh"
#include "launch_util.h"

namespace mnc {

struct IgemmArgs {
  int batch, H, W;
  int Cin, Cout;
  int taps;  // 1 (inner product / 1x1) or 9 (3x3, pad 1, stride 1)
  int tiles_h, tiles_w, tiles_n;
  int k_steps;  // taps * Cin / 64
  int split_k;
  int relu;
  // 0: split bf16 (hi, lo); 1: fp32; 2: split bf16 after a fused 2x2/2 ceil-mode max pool;
  // 4: tri-plane (fp16 hi, e4m3 lo, e4m3 hi copy -- see "precision mode 1" below); 5: tri-plane
  // after the fused max pool
  int out_mode;
  const float* bias;
  __nv_bfloat16* out_hi;   // modes 4/5: the fp16 plane
  __nv_bfloat16* out_lo;   // modes 4/5: the e4m3 residual plane
  uint8_t* out_x;          // modes 4/5: the e4m3 copy of the value
  float* out_f32;
  float acc_scale;         // accumulator -> true value (1 for bf16 operands; 2^-(ea+ew) in mode 1)
  float out_scale;         // modes 4/5: 2^ea of the tensor being written
  unsigned int* amax;      // optional: atomicMax of |output| as float bits (scale calibration)
  long long out_pix_stride;  // elements between consecutive pixels (rows)
  int out_ch_offset;
  long long split_stride;  // elements between split-K partial planes (fp32 mode)
  int vec_ok;              // 16-byte vector stores are aligned
  int tma_store;           // out_mode 0 only: epilogue stages tiles in smem and TMA-stores them
  // Mixed-size batches: image b fills the top-left of the padded blob.  img_hw [batch][2] holds
  // its size at input resolution; at this launch's trunk level (input halved `level` times,
  // ceil mode) its extent is ((h + 2^level - 1) >> level, ...).  Pixels outside their image's
  // extent are written as exact zeros and never enter a pool window or the published maximum.
  // nullptr: every pixel of the blob is inside.
  const int* img_hw;
  int level;
  int img_rows;            // > 0: tile "images" are single rows, image b = img / img_rows (conv1_1)
};

// Extent (rows, cols) of image b at p.level, clamped to the blob.
__device__ __forceinline__ int2 img_extent(const IgemmArgs& p, int b, int H, int W) {
  if (p.img_hw == nullptr) return make_int2(H, W);
  const int m = (1 << p.level) - 1;
  return make_int2(min(H, (__ldg(p.img_hw + 2 * b) + m) >> p.level),
                   min(W, (__ldg(p.img_hw + 2 * b + 1) + m) >> p.level));
}

constexpr int kBlockM = 128;

// BK = K elements per pipeline stage: 64 (128-byte rows, SWIZZLE_128B) or 32 (64-byte rows,
// SWIZZLE_64B: half-size stages, i.e. twice the pipeline depth in the same shared memory).
// CL = 2: the CTA pair of a cluster runs ONE M = 256 MMA per instruction (cta_group::2): each CTA
// holds its own 128 pixel rows of A and only HALF of the weight tile (BN / 2 rows), so per MAC an
// SM takes in 2/3 of the operand bytes of the single-CTA 128 x 256 tile -- operand delivery into
// the SM (~61 B/clk measured from L2), not the tensor pipe, is what bounds these kernels once the
// tensor work per MAC drops (profiles/README.md, r02 findings).
template <int BN, int BK, int CL = 1>
struct IgemmCfg {
  static constexpr int kABytes = kBlockM * BK * 2;  // one 2-byte plane of the A tile
  static constexpr int kBBytes = (BN / CL) * BK * 2;  // one 2-byte plane of this CTA's part of B
  static constexpr int kStageBytes = 2 * kABytes + 2 * kBBytes;
  static constexpr int kStagesRaw = (192 * 1024) / kStageBytes;
  static constexpr int kStages = kStagesRaw > 8 ? 8 : kStagesRaw;
  static constexpr int kTmemCols = (2 * BN <= 128) ? 128 : (2 * BN <= 256 ? 256 : 512);
  // epilogue staging: 2 buffers x (hi, lo) x 128 rows x 32 channels x 2 B
  static constexpr int kStagingBytes = 2 * 2 * 128 * 64;
  static constexpr int kBarrierBytes = 1024;
  static constexpr int kSmemBytes =
      kStages * kStageBytes + 1024 /*align*/ + kBarrierBytes + kStagingBytes;
};

struct Tile {
  int img, h0, w0, n0, ks;
  int kb, kn, kstride;   // this work item's k-steps: kb, kb + kstride, ... (kn of them)
  bool dummy;
};

// Work item `t` of CTA `rank` in a cluster of CL CTAs.  A cluster processes CL consecutive
// spatial tiles that share one Cout tile (so the weight tile can be multicast); when the spatial
// tile count is not a multiple of CL the last item carries a dummy tile (all-zero A, no stores).
template <int CL>
__device__ __forceinline__ Tile decode_tile(const IgemmArgs& p, int t, int rank, int TH, int TW,
                                            int BN) {
  const int per_img = p.tiles_h * p.tiles_w;
  const int spatial = p.batch * per_img;
  const int groups = (spatial + CL - 1) / CL;
  const int g = t % groups;
  const int rest = t / groups;
  const int nt = rest % p.tiles_n;
  Tile tl;
  tl.ks = rest / p.tiles_n;
  const int sp = g * CL + rank;
  tl.dummy = sp >= spatial;
  if (tl.dummy) {
    tl.img = p.batch;  // out of bounds in the batch dimension: TMA zero-fills the A tile
    tl.h0 = 0;
    tl.w0 = 0;
  } else {
    tl.img = sp / per_img;
    const int r = sp % per_img;
    tl.h0 = (r / p.tiles_w) * TH;
    tl.w0 = (r % p.tiles_w) * TW;
  }
  tl.n0 = nt * BN;
  // Split-K work items take INTERLEAVED k-steps (ks, ks + split, ks + 2*split, ...): the CTAs that
  // share a row tile start together and advance in step, so at any moment they read adjacent
  // 128-byte segments of the same activation rows -- DRAM sees ~split*128 contiguous bytes per row
  // instead of isolated 128-byte touches 200 KB apart (fc6_maskest: K = 100352, 963 MB read once).
  tl.kb = tl.ks;
  tl.kstride = p.split_k;
  tl.kn = (p.k_steps - tl.ks + p.split_k - 1) / p.split_k;
  return tl;
}

// ---------------------------------------------------------------------- precision mode 1 format
// "tri-plane" activations / weights (DESIGN.md section 3): a tensor with per-tensor exponent e is
// stored as   h = fp16(x * 2^e)            (main operand, kind::f16)
//             l = e4m3((x*2^e - h) * 2^6)  (residual, 2^-11 of h at most)
//             c = e4m3(x * 2^e * 2^-5)     (low-precision copy of the value)
// for activations, and with the residual scaled by 2^5 / the copy by 2^-6 for weights, so that
//   X.W * 2^(ex+ew) = Xh.Wh  +  Xl.Wc  +  Xc.Wl      (2^6 * 2^-6 = 2^-5 * 2^5 = 1)
// The first product runs as fp16 MMAs, the two corrections as ONE K-concatenated chain of FP8
// MMAs at twice the rate: 2 tensor-work units per MAC instead of the 3 of the split-bf16 scheme,
// at 1.1e-5 relative error per layer (scripts/fp8_correction_model.py; measured in tests).
// (element conversions: tri.cuh)

// ---------------------------------------------------------------------------------- epilogue
// Shared by the per-tap kernel and the halo kernel: warps 4..7 drain the TMEM accumulators of
// every tile this CTA owns (bias, ReLU, optional 2x2 ceil-mode max pool, re-split, store).
// NG = 2: two warp groups (warps 4..7 and 8..11; a warp may read the TMEM lane quarter warp_id % 4)
// drain alternate 32-column chunks of every tile -- for the low-K layers (conv1_1, conv1_2) the
// epilogue, not the MMA, is the longest stage of the pipeline.  Each group then owns ONE staging
// buffer (waiting for its previous bulk store to finish reading it) instead of two.
template <int TH, int TW, int BN, int CL, bool ACC2 = false, int NG = 1>
__device__ __forceinline__ void run_epilogue(const IgemmArgs& p, const CUtensorMap* tm_o_hi_p,
                                             const CUtensorMap* tm_o_lo_p,
                                             const CUtensorMap* tm_o_x_p, uint8_t* staging,
                                             uint64_t* tfull_bar, uint64_t* tempty_bar,
                                             uint32_t tmem_base, int rank, int first, int stride,
                                             int total_tiles) {
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int q = (warp - 4) & 3;   // TMEM lane quarter == warp_id % 4
  const int grp = (warp - 4) >> 2;  // 0 .. NG-1
  constexpr int NBUF = 2 / NG;      // staging buffers per group
  const int lead = 128 + grp * 128; // the group's bulk-store thread
  const int row = q * 32 + lane;
  int local = 0;
  int chunk_ctr = 0;
  float amx = 0.f;   // max |output| seen by this thread (valid pixels only)
  const float asc = p.acc_scale;
  for (int t = first; t < total_tiles; t += stride, ++local) {
    const Tile tl = decode_tile<CL>(p, t, rank, TH, TW, BN);
    const int img = tl.img, h0 = tl.h0, w0 = tl.w0, n0 = tl.n0, ks = tl.ks;
    const int acc = local & 1;
    const uint32_t acc_phase = (local >> 1) & 1;
    const int h = h0 + row / TW;
    const int w = w0 + row % TW;
    const bool inblob = !tl.dummy && (h < p.H) && (w < p.W);
    // this tile's image and its row in it (conv1_1 runs one-row images), and the image's extent
    const int eb = p.img_rows > 0 ? img / p.img_rows : img;
    const int eh = p.img_rows > 0 ? img - eb * p.img_rows : h0;
    const int2 ext = tl.dummy ? make_int2(0, 0)
                              : img_extent(p, eb, p.img_rows > 0 ? p.img_rows : p.H, p.W);
    const int hrow = eh + (h - h0);   // row within the image
    const bool valid = inblob && hrow < ext.x && w < ext.y;
    const long long pix = (static_cast<long long>(img) * p.H + h) * p.W + w;
    ptx::mbar_wait(&tfull_bar[acc], acc_phase);
    ptx::tc_fence_after();
#pragma unroll 1
    for (int c0 = grp * 32; c0 < BN; c0 += 32 * NG) {
      uint32_t r[32];
      // ACC2: the tile's sum is split over two column blocks (see conv_halo_tc_kernel)
      constexpr int kAccCols = ACC2 ? 2 * BN : BN;
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * kAccCols + c0;
      ptx::tmem_ld_32x32b_x32(taddr, r);
      if (ACC2) {
        uint32_t r2[32];
        ptx::tmem_ld_32x32b_x32(taddr + BN, r2);
        ptx::tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j)
          r[j] = __float_as_uint(__uint_as_float(r[j]) + __uint_as_float(r2[j]));
      } else {
        ptx::tmem_ld_wait();
      }
      const int ch0 = n0 + c0;
      if (p.out_mode == 3) continue;  // diagnostic: accumulators are drained and discarded
      if (p.out_mode == 2 || p.out_mode == 5) {
        // Fused 2x2 stride-2 ceil-mode max pool (pooling_layer.cu:11-47).  A warp holds 32/TW
        // whole image rows of the pixel tile (TW = 16: two rows, TW = 8: four), so the pool window
        // of an even (row, column) is lanes {l, l^1, l^TW, l^(TW+1)}: two shuffles per channel.
        // Each of the 4 lanes of a window then stores 8 of the chunk's 32 channels.
        // The 4 lanes of a window end up with 8 channels each by a reduce-scatter: exchange halves
        // with the x neighbour (16 shuffles), then quarters with the y neighbour (8) -- 24 shuffles
        // and 24 max per chunk instead of 64 + 64 for all-channels-everywhere.
        const bool odd_x = (lane & 1) != 0;
        const bool odd_y = ((lane / TW) & 1) != 0;
        const int part = (odd_x ? 2 : 0) | (odd_y ? 1 : 0);   // this lane stores channels part*8 .. +7
        const int hl = (row / TW) & ~1;   // tile-local top row / left column of this lane's window
        const int wl = (row % TW) & ~1;
        // max commutes with the monotone epilogue  x -> relu(x * scale + bias)  (scale > 0), so the
        // window maximum is taken on the RAW accumulators and the epilogue arithmetic runs on the 8
        // surviving channels of each lane only (bit-identical: fma and max are monotone / exact)
        float x[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) x[j] = __uint_as_float(r[j]);
        // ragged tile: rows outside the blob or outside this image's extent never win (a padded
        // pixel's raw accumulator is not zero: it sees the image's edge through the 3x3 window)
        if (!__all_sync(0xffffffffu, valid)) {
#pragma unroll
          for (int j = 0; j < 32; ++j) x[j] = valid ? x[j] : -3.402823466e+38f;
        }
        float y[16], m[8];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const float keep = odd_x ? x[j + 16] : x[j];
          const float send = odd_x ? x[j] : x[j + 16];
          y[j] = fmaxf(keep, __shfl_xor_sync(0xffffffffu, send, 1));
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float keep = odd_y ? y[j + 8] : y[j];
          const float send = odd_y ? y[j] : y[j + 8];
          m[j] = fmaxf(keep, __shfl_xor_sync(0xffffffffu, send, TW));
        }
        const int hp = (h0 + hl) >> 1;
        const int wp = (w0 + wl) >> 1;
        const int Ho = (p.H + 1) >> 1, Wo = (p.W + 1) >> 1;
        const int chp = ch0 + part * 8;
        if (!tl.dummy && hp < Ho && wp < Wo && (h0 + hl) < p.H && (w0 + wl) < p.W &&
            chp < p.Cout) {
          // pooled pixel inside the image's level+1 extent <=> its window's top-left pixel is
          // inside the level extent; outside it the output is an exact zero
          const bool pin = (h0 + hl) < ext.x && (w0 + wl) < ext.y;
          const long long ppix = (static_cast<long long>(img) * Ho + hp) * Wo + wp;
          const long long poff = ppix * p.out_pix_stride + p.out_ch_offset + chp;
          float bv[8];
          if (p.bias != nullptr && chp + 8 <= p.Cout && (reinterpret_cast<uintptr_t>(p.bias + chp) & 15) == 0) {
            const float4 b0 = __ldg(reinterpret_cast<const float4*>(p.bias + chp));
            const float4 b1 = __ldg(reinterpret_cast<const float4*>(p.bias + chp) + 1);
            bv[0] = b0.x, bv[1] = b0.y, bv[2] = b0.z, bv[3] = b0.w;
            bv[4] = b1.x, bv[5] = b1.y, bv[6] = b1.z, bv[7] = b1.w;
          } else {
#pragma unroll
            for (int j = 0; j < 8; ++j)
              bv[j] = (p.bias != nullptr && chp + j < p.Cout) ? __ldg(p.bias + chp + j) : 0.f;
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            m[j] = m[j] * asc + bv[j];
            if (p.relu) m[j] = fmaxf(m[j], 0.f);
            m[j] = pin ? m[j] : 0.f;
            if (chp + j < p.Cout) amx = fmaxf(amx, fabsf(m[j]));   // max |pooled output|
          }
          if (p.out_mode == 5) {
            uint32_t hw[4], lw[2], cw[2];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const Tri2 tr = tri_pack2(m[2 * e], m[2 * e + 1], p.out_scale);
              hw[e] = tr.h;
              if (e & 1) {
                lw[e >> 1] |= static_cast<uint32_t>(tr.l) << 16;
                cw[e >> 1] |= static_cast<uint32_t>(tr.c) << 16;
              } else {
                lw[e >> 1] = tr.l;
                cw[e >> 1] = tr.c;
              }
            }
            *reinterpret_cast<uint4*>(reinterpret_cast<__half*>(p.out_hi) + poff) =
                make_uint4(hw[0], hw[1], hw[2], hw[3]);
            *reinterpret_cast<uint2*>(reinterpret_cast<uint8_t*>(p.out_lo) + poff) = make_uint2(lw[0], lw[1]);
            *reinterpret_cast<uint2*>(p.out_x + poff) = make_uint2(cw[0], cw[1]);
            continue;
          }
          __nv_bfloat16* ph = p.out_hi + poff;
          __nv_bfloat16* pl = p.out_lo + poff;
          uint32_t hw[4], lw[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float x0 = m[2 * e], x1 = m[2 * e + 1];
            const __nv_bfloat16 h0b = __float2bfloat16_rn(x0);
            const __nv_bfloat16 h1b = __float2bfloat16_rn(x1);
            const __nv_bfloat16 l0b = __float2bfloat16_rn(x0 - __bfloat162float(h0b));
            const __nv_bfloat16 l1b = __float2bfloat16_rn(x1 - __bfloat162float(h1b));
            hw[e] = static_cast<uint32_t>(__bfloat16_as_ushort(h0b)) |
                    (static_cast<uint32_t>(__bfloat16_as_ushort(h1b)) << 16);
            lw[e] = static_cast<uint32_t>(__bfloat16_as_ushort(l0b)) |
                    (static_cast<uint32_t>(__bfloat16_as_ushort(l1b)) << 16);
          }
          *reinterpret_cast<uint4*>(ph) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
          *reinterpret_cast<uint4*>(pl) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
        }
      } else if (p.tma_store) {
        // ---- out_mode 0 / 4 via shared-memory staging + TMA store: each thread owns one pixel row
        // of the 128 x 32-channel chunk (64 B per 2-byte plane, written with the 64B-swizzle
        // pattern so the 16-byte stores are bank-conflict free; the one-byte planes of mode 4 are
        // 32 B per row, unswizzled); one elected thread then issues the bulk tensor stores.  TMA
        // clips ragged tiles, channel tails and the cluster's dummy tile, and the global writes
        // are whole rows.
        const bool tri = (p.out_mode == 4);
        const int buf = chunk_ctr % NBUF;
        uint8_t* sb = staging + (grp * NBUF + buf) * (2 * 128 * 64);
        if (threadIdx.x == lead) ptx::tma_store_wait_read<NBUF - 1>();  // this buffer's previous store
        ptx::named_bar_sync(1 + grp, 128);
        if (ch0 < p.Cout) {
          // bias: 8 x 16-byte loads when the chunk is whole and aligned (the usual case)
          float bv[32];
          if (p.bias != nullptr && ch0 + 32 <= p.Cout &&
              (reinterpret_cast<uintptr_t>(p.bias + ch0) & 15) == 0) {
#pragma unroll
            for (int j4 = 0; j4 < 8; ++j4) {
              const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.bias + ch0) + j4);
              bv[4 * j4] = b4.x;
              bv[4 * j4 + 1] = b4.y;
              bv[4 * j4 + 2] = b4.z;
              bv[4 * j4 + 3] = b4.w;
            }
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              bv[j] = (p.bias != nullptr && ch0 + j < p.Cout) ? __ldg(p.bias + ch0 + j) : 0.f;
          }
          float mx = 0.f;
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            uint32_t hw[4], lw[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              float x0 = __uint_as_float(r[g * 8 + 2 * e]) * asc + bv[g * 8 + 2 * e];
              float x1 = __uint_as_float(r[g * 8 + 2 * e + 1]) * asc + bv[g * 8 + 2 * e + 1];
              if (p.relu) {
                x0 = fmaxf(x0, 0.f);
                x1 = fmaxf(x1, 0.f);
              }
              if (!valid) {   // outside the image: exact zeros (TMA clips rows outside the blob)
                x0 = 0.f;
                x1 = 0.f;
              }
              mx = fmaxf(mx, fmaxf(fabsf(x0), fabsf(x1)));
              if (tri) {
                const Tri2 tr = tri_pack2(x0, x1, p.out_scale);
                hw[e] = tr.h;
                // lw[0..1]: residual bytes, lw[2..3]: copy bytes (8 channels each)
                if (e & 1) {
                  lw[e >> 1] |= static_cast<uint32_t>(tr.l) << 16;
                  lw[2 + (e >> 1)] |= static_cast<uint32_t>(tr.c) << 16;
                } else {
                  lw[e >> 1] = tr.l;
                  lw[2 + (e >> 1)] = tr.c;
                }
              } else {
                // packed conversions: (x0, x1) -> bf16x2 in one instruction; the hi values come
                // back as floats by a shift / mask of the packed word
                const __nv_bfloat162 hp = __floats2bfloat162_rn(x0, x1);
                const uint32_t hbits = *reinterpret_cast<const uint32_t*>(&hp);
                const float f0 = __uint_as_float(hbits << 16);
                const float f1 = __uint_as_float(hbits & 0xffff0000u);
                const __nv_bfloat162 lp = __floats2bfloat162_rn(x0 - f0, x1 - f1);
                hw[e] = hbits;
                lw[e] = *reinterpret_cast<const uint32_t*>(&lp);
              }
            }
            const int off = row * 64 + ((g ^ ((row >> 1) & 3)) << 4);
            *reinterpret_cast<uint4*>(sb + off) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
            if (tri) {
              *reinterpret_cast<uint2*>(sb + 128 * 64 + row * 32 + g * 8) = make_uint2(lw[0], lw[1]);
              *reinterpret_cast<uint2*>(sb + 128 * 96 + row * 32 + g * 8) = make_uint2(lw[2], lw[3]);
            } else {
              *reinterpret_cast<uint4*>(sb + 128 * 64 + off) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
            }
          }
          if (valid) amx = fmaxf(amx, mx);
        }
        ptx::fence_proxy_async();
        ptx::named_bar_sync(1 + grp, 128);
        if (threadIdx.x == lead && ch0 < p.Cout) {
          ptx::tma_store_4d(tm_o_hi_p, sb, ch0, w0, h0, img);
          ptx::tma_store_4d(tm_o_lo_p, sb + 128 * 64, ch0, w0, h0, img);
          if (tri) ptx::tma_store_4d(tm_o_x_p, sb + 128 * 96, ch0, w0, h0, img);
          ptx::tma_store_commit();
        }
        ++chunk_ctr;
      } else if (inblob && ch0 < p.Cout) {
        float v[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          float x = __uint_as_float(r[j]) * asc;
          if (p.bias != nullptr && ch0 + j < p.Cout) x += __ldg(p.bias + ch0 + j);
          if (p.relu) x = fmaxf(x, 0.f);
          v[j] = valid ? x : 0.f;   // outside the image: exact zeros
          if (ch0 + j < p.Cout) amx = fmaxf(amx, fabsf(v[j]));
        }
        const bool fullchunk = (ch0 + 32 <= p.Cout) && p.vec_ok;
        if (p.out_mode == 0) {
          __nv_bfloat16* ph = p.out_hi + pix * p.out_pix_stride + p.out_ch_offset + ch0;
          __nv_bfloat16* pl = p.out_lo + pix * p.out_pix_stride + p.out_ch_offset + ch0;
          if (fullchunk) {
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              uint32_t hw[4], lw[4];
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const float x0 = v[g * 8 + 2 * e], x1 = v[g * 8 + 2 * e + 1];
                const __nv_bfloat16 h0b = __float2bfloat16_rn(x0);
                const __nv_bfloat16 h1b = __float2bfloat16_rn(x1);
                const __nv_bfloat16 l0b = __float2bfloat16_rn(x0 - __bfloat162float(h0b));
                const __nv_bfloat16 l1b = __float2bfloat16_rn(x1 - __bfloat162float(h1b));
                hw[e] = static_cast<uint32_t>(__bfloat16_as_ushort(h0b)) |
                        (static_cast<uint32_t>(__bfloat16_as_ushort(h1b)) << 16);
                lw[e] = static_cast<uint32_t>(__bfloat16_as_ushort(l0b)) |
                        (static_cast<uint32_t>(__bfloat16_as_ushort(l1b)) << 16);
              }
              *reinterpret_cast<uint4*>(ph + g * 8) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
              *reinterpret_cast<uint4*>(pl + g * 8) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
            }
          } else {
            for (int j = 0; j < 32 && ch0 + j < p.Cout; ++j) {
              const __nv_bfloat16 hb = __float2bfloat16_rn(v[j]);
              ph[j] = hb;
              pl[j] = __float2bfloat16_rn(v[j] - __bfloat162float(hb));
            }
          }
        } else {
          float* po = p.out_f32 + ks * p.split_stride + pix * p.out_pix_stride +
                      p.out_ch_offset + ch0;
          if (fullchunk) {
#pragma unroll
            for (int g = 0; g < 8; ++g)
              *reinterpret_cast<float4*>(po + g * 4) =
                  make_float4(v[g * 4], v[g * 4 + 1], v[g * 4 + 2], v[g * 4 + 3]);
          } else {
            for (int j = 0; j < 32 && ch0 + j < p.Cout; ++j) po[j] = v[j];
          }
        }
      }
    }
    ptx::tc_fence_before();
    if (CL == 2)   // CTA pair: the leader's MMA warp waits for the accumulators of BOTH CTAs
      ptx::mbar_arrive_cluster(ptx::mapa_u32(ptx::smem_u32(&tempty_bar[acc]), 0));
    else
      ptx::mbar_arrive(&tempty_bar[acc]);
  }
  if (threadIdx.x == lead) ptx::tma_store_wait_read<0>();  // smem must outlive the bulk stores
  if (p.amax != nullptr) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) amx = fmaxf(amx, __shfl_xor_sync(0xffffffffu, amx, o));
    if (lane == 0 && amx > 0.f) atomicMax(p.amax, __float_as_uint(amx));
  }
}

// PM (precision mode): 0 = split-bf16 operands (planes hi, lo; 3 bf16 MMAs per k slice);
// 1 = tri-plane operands (fp16 value, e4m3 residual, e4m3 copy; see above): per 64 K-elements
// 4 fp16 MMAs + 4 FP8 MMAs (K = 32 each, double rate) instead of 12 bf16 MMAs.  A stage holds
// A:[h | l | c] then B:[h | c | l] -- same bytes as mode 0 (one 2-byte and two 1-byte planes).
template <int TH, int TW, int BN, int CL, int BK, int PM = 0>
__global__ void __launch_bounds__(256, 1)
igemm_tc_kernel(const __grid_constant__ CUtensorMap tm_a_hi, const __grid_constant__ CUtensorMap tm_a_lo,
                const __grid_constant__ CUtensorMap tm_a_x,
                const __grid_constant__ CUtensorMap tm_b_hi, const __grid_constant__ CUtensorMap tm_b_lo,
                const __grid_constant__ CUtensorMap tm_b_x,
                const __grid_constant__ CUtensorMap tm_o_hi, const __grid_constant__ CUtensorMap tm_o_lo,
                const __grid_constant__ CUtensorMap tm_o_x,
                const IgemmArgs p) {
  static_assert(TH * TW == kBlockM, "pixel tile must have 128 rows");
  using Cfg = IgemmCfg<BN, BK, CL>;
  constexpr int kStages = Cfg::kStages;
  constexpr int kABytes = Cfg::kABytes;
  constexpr int kBlockK = BK;
  constexpr bool kPair = (CL == 2);

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kStages * Cfg::kStageBytes);
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* tfull_bar = empty_bar + kStages;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
  uint8_t* staging = smem + kStages * Cfg::kStageBytes + Cfg::kBarrierBytes;  // 1024-aligned

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int spatial_tiles = p.batch * p.tiles_h * p.tiles_w;
  const int total_tiles = p.split_k * p.tiles_n * ((spatial_tiles + CL - 1) / CL);
  const int kchunks = p.Cin / kBlockK;
  const int rank = kPair ? static_cast<int>(ptx::cluster_ctarank()) : 0;
  const int first = blockIdx.x / CL;      // work items are owned by clusters
  const int stride = gridDim.x / CL;
  constexpr uint16_t kMask = static_cast<uint16_t>((1u << CL) - 1u);

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tm_a_hi);
    ptx::prefetch_tmap(&tm_a_lo);
    ptx::prefetch_tmap(&tm_b_hi);
    ptx::prefetch_tmap(&tm_b_lo);
    if (PM == 1) {
      ptx::prefetch_tmap(&tm_a_x);
      ptx::prefetch_tmap(&tm_b_x);
    }
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < kStages; ++s) {
      ptx::mbar_init(&full_bar[s], 1);    // pair: only the leader's is used (both CTAs' bytes)
      ptx::mbar_init(&empty_bar[s], 1);   // pair: released in both CTAs by the leader's commit
    }
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(&tfull_bar[a], 1);
      ptx::mbar_init(&tempty_bar[a], 128 * CL);  // pair: the leader's collects both epilogues
    }
    ptx::fence_barrier_init();
  }
  if (warp == 2) {
    if (kPair)
      ptx::tmem_alloc_2sm<Cfg::kTmemCols>(tmem_slot);
    else
      ptx::tmem_alloc<Cfg::kTmemCols>(tmem_slot);
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (kPair) ptx::cluster_sync_all();  // peers' barriers are initialised before any remote arrive
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    {  // whole warp, warp-uniform arguments; one lane is elected inside each issue (ptx.cuh)
      int stage = 0;
      uint32_t phase = 0;
      // B planes: mode 0 [hi | lo] of kBBytes each; mode 1 [h (kBBytes) | c | l (kBBytes/2 each)]
      constexpr int kNP = (PM == 0) ? 2 : 3;
      const CUtensorMap* amaps[3] = {&tm_a_hi, &tm_a_lo, &tm_a_x};
      const CUtensorMap* bmaps[3] = {&tm_b_hi, &tm_b_lo, &tm_b_x};
      for (int t = first; t < total_tiles; t += stride) {
        const Tile tl = decode_tile<CL>(p, t, rank, TH, TW, BN);
        for (int i = 0, k = tl.kb; i < tl.kn; ++i, k += tl.kstride) {
          ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* st = smem + stage * Cfg::kStageBytes;
          // pair: the leader's barrier counts the bytes of both CTAs' loads
          if (!kPair || rank == 0)
            ptx::mbar_arrive_expect_tx_w(&full_bar[stage], CL * Cfg::kStageBytes);
          const uint32_t bar_cl = kPair ? ptx::mapa_u32(ptx::smem_u32(&full_bar[stage]), 0) : 0u;
          const int tap = k / kchunks;
          const int kc = k - tap * kchunks;
          int dy = 0, dx = 0;
          if (p.taps == 9) {
            dy = tap / 3 - 1;
            dx = tap % 3 - 1;
          }
#pragma unroll
          for (int pl = 0; pl < kNP; ++pl) {
            const int aoff = (PM == 0) ? pl * kABytes : (pl == 0 ? 0 : kABytes + (pl - 1) * (kABytes / 2));
            const int boff = (PM == 0) ? pl * Cfg::kBBytes
                                       : (pl == 0 ? 0 : Cfg::kBBytes + (pl - 1) * (Cfg::kBBytes / 2));
            if (kPair) {
              ptx::tma_load_4d_2sm_w(st + aoff, amaps[pl], bar_cl, kc * kBlockK, tl.w0 + dx,
                                     tl.h0 + dy, tl.img);
              ptx::tma_load_2d_2sm_w(st + 2 * kABytes + boff, bmaps[pl], bar_cl,
                                     tap * p.Cin + kc * kBlockK, tl.n0 + rank * (BN / CL));
            } else {
              ptx::tma_load_4d_w(st + aoff, amaps[pl], &full_bar[stage], kc * kBlockK, tl.w0 + dx,
                                 tl.h0 + dy, tl.img);
              ptx::tma_load_2d_w(st + 2 * kABytes + boff, bmaps[pl], &full_bar[stage],
                                 tap * p.Cin + kc * kBlockK, tl.n0);
            }
          }
          if (++stage == kStages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1 && rank == 0) {
    // -------------------------------------------------------------- MMA issuer (pair: leader only)
    {  // whole warp, warp-uniform arguments; one lane is elected inside each issue (ptx.cuh)
      // mode 1: format code 0 = fp16 for kind::f16 and E4M3 for kind::f8f6f4 (same descriptor)
      constexpr uint32_t idesc1 = (PM == 0) ? ptx::umma_idesc_bf16_m128(BN) : ptx::umma_idesc_fmt0_m128(BN);
      // pair: M = 256 (m_dim field = M >> 4 at bit 24)
      constexpr uint32_t idesc = kPair ? ((idesc1 & ~(0x1Fu << 24)) | ((256u >> 4) << 24)) : idesc1;
      int stage = 0;
      uint32_t phase = 0;
      int local = 0;
      for (int t = first; t < total_tiles; t += stride, ++local) {
        const Tile tl = decode_tile<CL>(p, t, rank, TH, TW, BN);
        const int kn = tl.kn;
        const int acc = local & 1;
        const uint32_t acc_phase = (local >> 1) & 1;
        ptx::mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
        ptx::tc_fence_after();
        const uint32_t tmem_d = tmem_base + acc * BN;
        for (int i = 0; i < kn; ++i) {
          ptx::mbar_wait(&full_bar[stage], phase);
          ptx::tc_fence_after();
          const uint32_t a_hi = ptx::smem_u32(smem + stage * Cfg::kStageBytes);
          const uint32_t b_hi = a_hi + 2 * kABytes;
          if (PM == 0) {
            const uint32_t a_lo = a_hi + kABytes;
            const uint32_t b_lo = b_hi + Cfg::kBBytes;
#pragma unroll
            for (int kk = 0; kk < kBlockK / 16; ++kk) {
              const uint64_t da_hi = ptx::umma_desc_rows<BK * 2>(a_hi + kk * 32);
              const uint64_t da_lo = ptx::umma_desc_rows<BK * 2>(a_lo + kk * 32);
              const uint64_t db_hi = ptx::umma_desc_rows<BK * 2>(b_hi + kk * 32);
              const uint64_t db_lo = ptx::umma_desc_rows<BK * 2>(b_lo + kk * 32);
              // small cross terms first, then the dominant product
              const uint32_t acc0 = (i > 0 || kk > 0) ? 1u : 0u;
              if (kPair) {
                ptx::umma_f16_ss_2sm_w(tmem_d, da_lo, db_hi, idesc, acc0);
                ptx::umma_f16_ss_2sm_w(tmem_d, da_hi, db_lo, idesc, 1u);
                ptx::umma_f16_ss_2sm_w(tmem_d, da_hi, db_hi, idesc, 1u);
              } else {
                ptx::umma_bf16_ss_w(tmem_d, da_lo, db_hi, idesc, acc0);
                ptx::umma_bf16_ss_w(tmem_d, da_hi, db_lo, idesc, 1u);
                ptx::umma_bf16_ss_w(tmem_d, da_hi, db_hi, idesc, 1u);
              }
            }
          } else {
            const uint32_t a_l = a_hi + kABytes, a_c = a_l + kABytes / 2;
            const uint32_t b_c = b_hi + Cfg::kBBytes, b_l = b_c + Cfg::kBBytes / 2;
            // corrections (FP8, K = 32 per instruction): residual x copy, copy x residual
#pragma unroll
            for (int kk = 0; kk < kBlockK / 32; ++kk) {
              const uint64_t da_l = ptx::umma_desc_rows<BK>(a_l + kk * 32);
              const uint64_t db_c = ptx::umma_desc_rows<BK>(b_c + kk * 32);
              const uint64_t da_c = ptx::umma_desc_rows<BK>(a_c + kk * 32);
              const uint64_t db_l = ptx::umma_desc_rows<BK>(b_l + kk * 32);
              const uint32_t acc0 = (i > 0 || kk > 0) ? 1u : 0u;
              if (kPair) {
                ptx::umma_f8_ss_2sm_w(tmem_d, da_l, db_c, idesc, acc0);
                ptx::umma_f8_ss_2sm_w(tmem_d, da_c, db_l, idesc, 1u);
              } else {
                ptx::umma_f8_ss_w(tmem_d, da_l, db_c, idesc, acc0);
                ptx::umma_f8_ss_w(tmem_d, da_c, db_l, idesc, 1u);
              }
            }
            // main product (fp16, K = 16 per instruction)
#pragma unroll
            for (int kk = 0; kk < kBlockK / 16; ++kk) {
              const uint64_t da = ptx::umma_desc_rows<BK * 2>(a_hi + kk * 32);
              const uint64_t db = ptx::umma_desc_rows<BK * 2>(b_hi + kk * 32);
              if (kPair)
                ptx::umma_f16_ss_2sm_w(tmem_d, da, db, idesc, 1u);
              else
                ptx::umma_bf16_ss_w(tmem_d, da, db, idesc, 1u);
            }
          }
          if (kPair)
            ptx::umma_commit_2sm_w(&empty_bar[stage], kMask);  // frees the stage in both CTAs
          else
            ptx::umma_commit_w(&empty_bar[stage]);
          if (++stage == kStages) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (kPair)
          ptx::umma_commit_2sm_w(&tfull_bar[acc], kMask);      // both epilogues may drain
        else
          ptx::umma_commit_w(&tfull_bar[acc]);
      }
    }
  } else if (warp >= 4) {
    // ---------------------------------------------------------------- epilogue
    run_epilogue<TH, TW, BN, CL>(p, &tm_o_hi, &tm_o_lo, &tm_o_x, staging, tfull_bar, tempty_bar,
                                 tmem_base, rank, first, stride, total_tiles);
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (kPair) ptx::cluster_sync_all();  // no CTA leaves while a peer may still signal its barriers
  if (warp == 2) {
    ptx::tc_fence_after();
    if (kPair)
      ptx::tmem_dealloc_2sm<Cfg::kTmemCols>(tmem_base);
    else
      ptx::tmem_dealloc<Cfg::kTmemCols>(tmem_base);
  }
}

// ------------------------------------------------------------------------------ halo kernel
// 3x3 convolution for the low-Cin layers (conv1_2, conv2_x), where the per-tap kernel is bound by
// the rate at which activation tiles arrive in shared memory (each pixel is fetched 9 times, once
// per filter tap).  Here the pixel tile is 16 rows x 8 columns and ONE TMA box [18][10][64ch]
// brings in the tile plus its halo; every filter tap is then a *shifted window* of that box:
// the tcgen05 shared-memory descriptor takes start = halo + ((ky*10 + kx) * 128 B) and a stride
// between 8-row groups of 1280 B (one halo row) instead of the canonical 1024 B.  This is legal
// because the 128B swizzle is a pure function of the shared-memory address (verified on B200 by
// scripts/exp/umma_offset_test.cu: all 9 windows read back exactly).  Activation traffic into the
// SM drops from 9 x 32 KB to 46 KB per (tile, 64-channel chunk); weights stream per tap through
// their own ring of stages.
constexpr int kHaloTH = 16, kHaloTW = 8;
constexpr int kHaloRows = (kHaloTH + 2) * (kHaloTW + 2);          // 180 pixels
constexpr int kHaloPlaneBytes = kHaloRows * 128;                   // 23040 (2-byte plane of 64 channels)
constexpr int kHaloPlanePad = (kHaloPlaneBytes + 1023) / 1024 * 1024;  // 23552
constexpr int kHaloPlane8Bytes = kHaloRows * 64;                   // 11520 (1-byte plane)
constexpr int kHaloPlane8Pad = (kHaloPlane8Bytes + 1023) / 1024 * 1024;  // 12288
constexpr int kHaloNA = 2;

// PM 0: A = [hi | lo] bf16 planes, B per tap = [hi | lo]; three products as two instructions
//       (stacked N, two accumulator column blocks).
// PM 1: A = [h (fp16) | l | c (e4m3, 64-byte rows, SWIZZLE_64B)], B per tap = [h | c | l]; per
//       64 channels 4 fp16 MMAs + 4 FP8 MMAs into ONE accumulator block.  The shifted-window
//       descriptors work for the one-byte planes as well (start + (ky*10+kx)*64 B, SBO 640 B:
//       scripts/exp/umma_offset_sw64_fp8_test.cu, all 9 windows exact on B200).
// CL 2 (PM 1 only): a CTA pair computes two pixel tiles against one Cout tile with M = 256
// cta_group::2 MMAs; each CTA brings in its own halo box and HALF of every tap's weights, so the
// weight fills and the tensor core's B-operand reads per CTA halve (these layers are bound by
// shared-memory bandwidth, profiles/README.md finding 11).
template <int BN, int PM, int CL = 1>
struct HaloCfg {
  static constexpr int kABytes = (PM == 0) ? 2 * kHaloPlanePad : kHaloPlanePad + 2 * kHaloPlane8Pad;
  static constexpr int kATx = (PM == 0) ? 2 * kHaloPlaneBytes : kHaloPlaneBytes + 2 * kHaloPlane8Bytes;
  static constexpr int kBBytes = (BN / CL) * 128;                 // one 2-byte plane of one tap's weights
  static constexpr int kBStage = 2 * kBBytes;                     // PM 1: h (kBBytes) + c + l (kBBytes/2 each)
  static constexpr int kNBfit = (192 * 1024 - kHaloNA * kABytes) / kBStage;
  static constexpr int kNB = kNBfit > 12 ? 12 : kNBfit;
  // accumulators: PM 0 two column blocks per tile ([hi*hi + lo*hi | hi*lo]), PM 1 one; double-buffered
  static constexpr int kAccCols = (PM == 0) ? 2 * BN : BN;
  static constexpr int kTmemCols = (2 * kAccCols <= 128) ? 128 : (2 * kAccCols <= 256 ? 256 : 512);
  static constexpr int kStagingBytes = 2 * 2 * 128 * 64;
  static constexpr int kBarrierBytes = 1024;
  static constexpr int kRingBytes = kHaloNA * kABytes + kNB * kBStage;
  static constexpr int kSmemBytes = kRingBytes + 1024 + kBarrierBytes + kStagingBytes;
};

template <int BN, int PM, int CL>
__global__ void __launch_bounds__(384, 1)
conv_halo_tc_kernel(const __grid_constant__ CUtensorMap tm_a_hi, const __grid_constant__ CUtensorMap tm_a_lo,
                    const __grid_constant__ CUtensorMap tm_a_x,
                    const __grid_constant__ CUtensorMap tm_b_hi, const __grid_constant__ CUtensorMap tm_b_lo,
                    const __grid_constant__ CUtensorMap tm_b_x,
                    const __grid_constant__ CUtensorMap tm_o_hi, const __grid_constant__ CUtensorMap tm_o_lo,
                    const __grid_constant__ CUtensorMap tm_o_x, const IgemmArgs p) {
  static_assert(CL == 1 || PM == 1, "CTA pairs: precision mode 1 only");
  using Cfg = HaloCfg<BN, PM, CL>;
  constexpr int TH = kHaloTH, TW = kHaloTW, NB = Cfg::kNB;
  // two epilogue warp groups (warps 4..7, 8..11) drain alternate 32-column chunks: with one
  // group a single warp per scheduler carried 4 chunks per tile at BN = 128 and the epilogue, not
  // the MMA, set the pace (r02 ncu: the MMA warp waited on tempty)
  constexpr int kNG = 2;
  constexpr bool kPair = (CL == 2);
  constexpr uint16_t kMask = static_cast<uint16_t>((1u << CL) - 1u);
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  uint8_t* a_ring = smem;
  uint8_t* b_ring = smem + kHaloNA * Cfg::kABytes;
  uint64_t* a_full = reinterpret_cast<uint64_t*>(smem + Cfg::kRingBytes);
  uint64_t* a_empty = a_full + kHaloNA;
  uint64_t* b_full = a_empty + kHaloNA;
  uint64_t* b_empty = b_full + NB;
  uint64_t* tfull_bar = b_empty + NB;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
  uint8_t* staging = smem + Cfg::kRingBytes + Cfg::kBarrierBytes;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int spatial_tiles = p.batch * p.tiles_h * p.tiles_w;
  const int total_tiles = p.tiles_n * ((spatial_tiles + CL - 1) / CL);
  const int kchunks = p.Cin / 64;
  const int rank = kPair ? static_cast<int>(ptx::cluster_ctarank()) : 0;
  const int first = blockIdx.x / CL, stride = gridDim.x / CL;   // work items are owned by clusters

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tm_a_hi);
    ptx::prefetch_tmap(&tm_a_lo);
    ptx::prefetch_tmap(&tm_b_hi);
    ptx::prefetch_tmap(&tm_b_lo);
    if (PM == 1) {
      ptx::prefetch_tmap(&tm_a_x);
      ptx::prefetch_tmap(&tm_b_x);
    }
  }
  if (warp == 1 && lane == 0) {
    // pair: the leader's full barriers count both CTAs' bytes; the leader's commits release the
    // empty barriers of both CTAs; the leader's tempty collects both epilogues
    for (int s = 0; s < kHaloNA; ++s) {
      ptx::mbar_init(&a_full[s], 1);
      ptx::mbar_init(&a_empty[s], 1);
    }
    for (int s = 0; s < NB; ++s) {
      ptx::mbar_init(&b_full[s], 1);
      ptx::mbar_init(&b_empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(&tfull_bar[a], 1);
      ptx::mbar_init(&tempty_bar[a], 128 * kNG * CL);
    }
    ptx::fence_barrier_init();
  }
  if (warp == 2) {
    if (kPair)
      ptx::tmem_alloc_2sm<Cfg::kTmemCols>(tmem_slot);
    else
      ptx::tmem_alloc<Cfg::kTmemCols>(tmem_slot);
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (kPair) ptx::cluster_sync_all();  // peers' barriers are initialised before any remote arrive
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    {  // whole warp, warp-uniform arguments; one lane is elected inside each issue (ptx.cuh)
      int as = 0, bs = 0;
      uint32_t aph = 0, bph = 0;
      for (int t = first; t < total_tiles; t += stride) {
        const Tile tl = decode_tile<CL>(p, t, rank, TH, TW, BN);
        const int nrow = tl.n0 + rank * (BN / CL);    // this CTA's share of the Cout tile
        for (int kc = 0; kc < kchunks; ++kc) {
          ptx::mbar_wait(&a_empty[as], aph ^ 1);
          uint8_t* sa = a_ring + as * Cfg::kABytes;
          if (!kPair || rank == 0) ptx::mbar_arrive_expect_tx_w(&a_full[as], CL * Cfg::kATx);
          if (kPair) {
            const uint32_t bar = ptx::mapa_u32(ptx::smem_u32(&a_full[as]), 0);
            ptx::tma_load_4d_2sm_w(sa, &tm_a_hi, bar, kc * 64, tl.w0 - 1, tl.h0 - 1, tl.img);
            ptx::tma_load_4d_2sm_w(sa + kHaloPlanePad, &tm_a_lo, bar, kc * 64, tl.w0 - 1, tl.h0 - 1,
                                   tl.img);
            ptx::tma_load_4d_2sm_w(sa + kHaloPlanePad + kHaloPlane8Pad, &tm_a_x, bar, kc * 64,
                                   tl.w0 - 1, tl.h0 - 1, tl.img);
          } else {
            ptx::tma_load_4d_w(sa, &tm_a_hi, &a_full[as], kc * 64, tl.w0 - 1, tl.h0 - 1, tl.img);
            ptx::tma_load_4d_w(sa + kHaloPlanePad, &tm_a_lo, &a_full[as], kc * 64, tl.w0 - 1,
                               tl.h0 - 1, tl.img);
            if (PM == 1)
              ptx::tma_load_4d_w(sa + kHaloPlanePad + kHaloPlane8Pad, &tm_a_x, &a_full[as], kc * 64,
                                 tl.w0 - 1, tl.h0 - 1, tl.img);
          }
          if (++as == kHaloNA) {
            as = 0;
            aph ^= 1;
          }
          for (int tap = 0; tap < 9; ++tap) {
            ptx::mbar_wait(&b_empty[bs], bph ^ 1);
            uint8_t* sb = b_ring + bs * Cfg::kBStage;
            if (!kPair || rank == 0) ptx::mbar_arrive_expect_tx_w(&b_full[bs], CL * Cfg::kBStage);
            const int kcol = tap * p.Cin + kc * 64;
            if (kPair) {
              const uint32_t bar = ptx::mapa_u32(ptx::smem_u32(&b_full[bs]), 0);
              ptx::tma_load_2d_2sm_w(sb, &tm_b_hi, bar, kcol, nrow);
              ptx::tma_load_2d_2sm_w(sb + Cfg::kBBytes, &tm_b_lo, bar, kcol, nrow);
              ptx::tma_load_2d_2sm_w(sb + Cfg::kBBytes + Cfg::kBBytes / 2, &tm_b_x, bar, kcol, nrow);
            } else {
              ptx::tma_load_2d_w(sb, &tm_b_hi, &b_full[bs], kcol, nrow);
              ptx::tma_load_2d_w(sb + Cfg::kBBytes, &tm_b_lo, &b_full[bs], kcol, nrow);
              if (PM == 1)
                ptx::tma_load_2d_w(sb + Cfg::kBBytes + Cfg::kBBytes / 2, &tm_b_x, &b_full[bs], kcol, nrow);
            }
            if (++bs == NB) {
              bs = 0;
              bph ^= 1;
            }
          }
        }
      }
    }
  } else if (warp == 1 && rank == 0) {
    // -------------------------------------------------------------- MMA issuer (pair: leader only)
    {  // whole warp, warp-uniform arguments; one lane is elected inside each issue (ptx.cuh)
      // PM 0: the per-instruction overhead of tcgen05.mma (~40 cycles) matters at these small N, so
      // the three split-precision products are issued as two instructions: the hi and lo weight
      // planes sit back to back in the stage, so A_hi x [B_hi | B_lo] is ONE N = 2*BN MMA into
      // columns [0, 2BN), and A_lo x B_hi accumulates into columns [0, BN).  The epilogue adds
      // the two column blocks.
      constexpr uint32_t idesc1 = ptx::umma_idesc_bf16_m128(2 * BN);
      constexpr uint32_t idesc2 = ptx::umma_idesc_bf16_m128(BN);
      constexpr uint32_t idesc_f1 = ptx::umma_idesc_fmt0_m128(BN);   // PM 1: fp16 / e4m3, N = BN
      // pair: M = 256 (m_dim field = M >> 4 at bit 24)
      constexpr uint32_t idesc_f = kPair ? ((idesc_f1 & ~(0x1Fu << 24)) | ((256u >> 4) << 24)) : idesc_f1;
      constexpr uint32_t kSbo = (TW + 2) * 128;  // one halo row of a 2-byte plane
      constexpr uint32_t kSbo8 = (TW + 2) * 64;  // ... of a 1-byte plane
      constexpr uint64_t kHiA16 = static_cast<uint64_t>(ptx::desc_hi_sw128_sbo(kSbo)) << 32;
      constexpr uint64_t kHiA8 = static_cast<uint64_t>(ptx::desc_hi_sw64_sbo(kSbo8)) << 32;
      constexpr uint64_t kHiB16 = static_cast<uint64_t>(ptx::kDescHiSw128) << 32;
      constexpr uint64_t kHiB8 = static_cast<uint64_t>(ptx::kDescHiSw64) << 32;
      int as = 0, bs = 0, local = 0;
      uint32_t aph = 0, bph = 0;
      for (int t = first; t < total_tiles; t += stride, ++local) {
        const int acc = local & 1;
        const uint32_t acc_phase = (local >> 1) & 1;
        ptx::mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
        ptx::tc_fence_after();
        const uint32_t tmem_d = tmem_base + acc * Cfg::kAccCols;
        for (int kc = 0; kc < kchunks; ++kc) {
          ptx::mbar_wait(&a_full[as], aph);
          ptx::tc_fence_after();
          const uint32_t a_hi0 = ptx::smem_u32(a_ring + as * Cfg::kABytes);
          const uint32_t a_lo0 = a_hi0 + kHaloPlanePad;                    // PM 1: the residual plane
          const uint32_t a_c0 = a_lo0 + kHaloPlane8Pad;                    // PM 1: the copy plane
          for (int tap = 0; tap < 9; ++tap) {
            ptx::mbar_wait(&b_full[bs], bph);
            ptx::tc_fence_after();
            // shifted window (reading all taps from offset 0 instead is no faster: the windows cost
            // nothing extra; what bounds the Cout = 64 layer is shared-memory bandwidth)
            const uint32_t wpix = (tap / 3) * (TW + 2) + (tap % 3);
            const uint32_t lb = ptx::desc_lo(ptx::smem_u32(b_ring + bs * Cfg::kBStage));
            if (PM == 0) {
              // descriptor low words (start address >> 4); + 2 per 16-element k slice
              const uint32_t la_hi = ptx::desc_lo(a_hi0 + wpix * 128);
              const uint32_t la_lo = ptx::desc_lo(a_lo0 + wpix * 128);
#pragma unroll
              for (int kk = 0; kk < 4; ++kk) {
                const uint32_t accum = (kc > 0 || tap > 0 || kk > 0) ? 1u : 0u;
                ptx::umma_bf16_ss_w32<ptx::desc_hi_sw128_sbo(kSbo), ptx::kDescHiSw128>(
                    tmem_d, la_hi + 2 * kk, lb + 2 * kk, idesc1, accum);
                ptx::umma_bf16_ss_w32<ptx::desc_hi_sw128_sbo(kSbo), ptx::kDescHiSw128>(
                    tmem_d, la_lo + 2 * kk, lb + 2 * kk, idesc2, 1u);
              }
            } else {
              const uint32_t la_h = ptx::desc_lo(a_hi0 + wpix * 128);
              const uint32_t la_l = ptx::desc_lo(a_lo0 + wpix * 64);
              const uint32_t la_c = ptx::desc_lo(a_c0 + wpix * 64);
              const uint32_t lb_c = lb + (Cfg::kBBytes >> 4);                         // copy plane of B
              const uint32_t lb_l = lb_c + (Cfg::kBBytes >> 5);                       // residual plane of B
              // corrections (FP8, K = 32): residual x copy, copy x residual
#pragma unroll
              for (int kk = 0; kk < 2; ++kk) {
                const uint32_t accum = (kc > 0 || tap > 0 || kk > 0) ? 1u : 0u;
                if (kPair) {
                  ptx::umma_f8_ss_2sm_w(tmem_d, kHiA8 | (la_l + 2 * kk), kHiB8 | (lb_c + 2 * kk), idesc_f, accum);
                  ptx::umma_f8_ss_2sm_w(tmem_d, kHiA8 | (la_c + 2 * kk), kHiB8 | (lb_l + 2 * kk), idesc_f, 1u);
                } else {
                  ptx::umma_f8_ss_w32<ptx::desc_hi_sw64_sbo(kSbo8), ptx::kDescHiSw64>(
                      tmem_d, la_l + 2 * kk, lb_c + 2 * kk, idesc_f, accum);
                  ptx::umma_f8_ss_w32<ptx::desc_hi_sw64_sbo(kSbo8), ptx::kDescHiSw64>(
                      tmem_d, la_c + 2 * kk, lb_l + 2 * kk, idesc_f, 1u);
                }
              }
              // main product (fp16, K = 16)
#pragma unroll
              for (int kk = 0; kk < 4; ++kk) {
                if (kPair)
                  ptx::umma_f16_ss_2sm_w(tmem_d, kHiA16 | (la_h + 2 * kk), kHiB16 | (lb + 2 * kk), idesc_f, 1u);
                else
                  ptx::umma_bf16_ss_w32<ptx::desc_hi_sw128_sbo(kSbo), ptx::kDescHiSw128>(
                      tmem_d, la_h + 2 * kk, lb + 2 * kk, idesc_f, 1u);
              }
            }
            if (kPair)
              ptx::umma_commit_2sm_w(&b_empty[bs], kMask);   // frees the stage in both CTAs
            else
              ptx::umma_commit_w(&b_empty[bs]);
            if (++bs == NB) {
              bs = 0;
              bph ^= 1;
            }
          }
          if (kPair)
            ptx::umma_commit_2sm_w(&a_empty[as], kMask);
          else
            ptx::umma_commit_w(&a_empty[as]);
          if (++as == kHaloNA) {
            as = 0;
            aph ^= 1;
          }
        }
        if (kPair)
          ptx::umma_commit_2sm_w(&tfull_bar[acc], kMask);     // both epilogues may drain
        else
          ptx::umma_commit_w(&tfull_bar[acc]);
      }
    }
  } else if (warp >= 4) {
    run_epilogue<TH, TW, BN, CL, PM == 0, kNG>(p, &tm_o_hi, &tm_o_lo, &tm_o_x, staging, tfull_bar,
                                               tempty_bar, tmem_base, rank, first, stride, total_tiles);
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (kPair) ptx::cluster_sync_all();  // no CTA leaves while a peer may still signal its barriers
  if (warp == 2) {
    ptx::tc_fence_after();
    if (kPair)
      ptx::tmem_dealloc_2sm<Cfg::kTmemCols>(tmem_base);
    else
      ptx::tmem_dealloc<Cfg::kTmemCols>(tmem_base);
  }
}

// ------------------------------------------------------------------------------ conv1_1
// conv1_1 (3 -> 64 channels, K = 27) on the tensor cores.  The SIMT kernel spends 0.65 ms per batch
// of 8 on 8.3 G fp32 FMAs; as an MMA the layer is 37.5k tiles x 4 instructions and the kernel is
// bound by writing its 1.23 GB of output.  There is nothing for TMA to im2col (3 channels), so
// four producer warps build the A tile themselves: thread p gathers the 27-value patch of pixel p
// from the fp32 NCHW blob (coalesced along the row; neighbours' re-reads hit L1), splits each value
// into (hi, lo) bf16, pads K to 32 and writes the two 64-byte rows of the tile with the 64B swizzle
// pattern the tcgen05 descriptor (SWIZZLE_64B, K-major) expects.  Weights: one [hi(64) ; lo(64)] x 32
// tile, loaded once by TMA; per 16-wide k slice  A_hi x [B_hi ; B_lo]  (N = 128) and  A_lo x B_hi
// (N = 64), the same stacked-N scheme as conv_halo_tc_kernel, so run_epilogue<.., ACC2> is reused
// unchanged (bias, ReLU, re-split, swizzled staging, TMA store).  The image batch is viewed as
// batch*H one-row images so that a tile is 128 consecutive pixels of a row.
constexpr int kC11K = 32;                       // 27 padded
constexpr int kC11ABytes = kBlockM * kC11K * 2; // one bf16 plane of the A tile: 8 KB
constexpr int kC11Stages = 2;
constexpr int kC11BBytes = 128 * kC11K * 2;     // stacked weight tile: 8 KB
constexpr int kC11Ring = kC11Stages * 2 * kC11ABytes + kC11BBytes;  // 40 KB
constexpr int kC11Staging = 2 * 2 * 128 * 64;
constexpr int kC11Smem = kC11Ring + 1024 /*barriers*/ + kC11Staging + 1024 /*align*/;
constexpr int kC11Threads = 640;   // 4 control + 8 epilogue + 8 producer warps

__global__ void __launch_bounds__(kC11Threads, 1)
conv1_1_tc_kernel(const float* __restrict__ data, int B, int H, int W,
                  const __grid_constant__ CUtensorMap tm_b, const __grid_constant__ CUtensorMap tm_o_hi,
                  const __grid_constant__ CUtensorMap tm_o_lo, const __grid_constant__ CUtensorMap tm_o_x,
                  const IgemmArgs p) {
  constexpr int BN = 64;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  uint8_t* a_ring = smem;
  uint8_t* b_tile = smem + kC11Stages * 2 * kC11ABytes;
  uint64_t* a_full = reinterpret_cast<uint64_t*>(smem + kC11Ring);
  uint64_t* a_empty = a_full + kC11Stages;
  uint64_t* b_full = a_empty + kC11Stages;
  uint64_t* tfull_bar = b_full + 1;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
  uint8_t* staging = smem + kC11Ring + 1024;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int total_tiles = p.batch * p.tiles_w;   // p.batch = B*H one-row images
  const int first = blockIdx.x, stride = gridDim.x;

  if (warp == 0 && lane == 0) ptx::prefetch_tmap(&tm_b);
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < kC11Stages; ++s) {
      ptx::mbar_init(&a_full[s], 128);
      ptx::mbar_init(&a_empty[s], 1);
    }
    ptx::mbar_init(b_full, 1);
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(&tfull_bar[a], 1);
      ptx::mbar_init(&tempty_bar[a], 256);
    }
    ptx::fence_barrier_init();
  }
  if (warp == 2) ptx::tmem_alloc<256>(tmem_slot);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // weights: once per CTA
    ptx::mbar_arrive_expect_tx_w(b_full, kC11BBytes);
    ptx::tma_load_2d_w(b_tile, &tm_b, b_full, 0, 0);
  } else if (warp == 1) {
    // -------------------------------------------------------------- MMA issuer (whole warp)
    constexpr uint32_t idesc1 = ptx::umma_idesc_bf16_m128(2 * BN);
    constexpr uint32_t idesc2 = ptx::umma_idesc_bf16_m128(BN);
    ptx::mbar_wait(b_full, 0);
    ptx::tc_fence_after();
    const uint32_t b_addr = ptx::smem_u32(b_tile);
    int as = 0, local = 0;
    uint32_t aph = 0;
    for (int t = first; t < total_tiles; t += stride, ++local) {
      const int acc = local & 1;
      const uint32_t acc_phase = (local >> 1) & 1;
      ptx::mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
      ptx::mbar_wait(&a_full[as], aph);
      ptx::tc_fence_after();
      const uint32_t tmem_d = tmem_base + acc * (2 * BN);
      const uint32_t a_hi = ptx::smem_u32(a_ring + as * 2 * kC11ABytes);
      const uint32_t a_lo = a_hi + kC11ABytes;
#pragma unroll
      for (int kk = 0; kk < kC11K / 16; ++kk) {
        const uint64_t da_hi = ptx::umma_desc_sw64(a_hi + kk * 32);
        const uint64_t da_lo = ptx::umma_desc_sw64(a_lo + kk * 32);
        const uint64_t db = ptx::umma_desc_sw64(b_addr + kk * 32);
        ptx::umma_bf16_ss_w(tmem_d, da_hi, db, idesc1, kk > 0 ? 1u : 0u);
        ptx::umma_bf16_ss_w(tmem_d, da_lo, db, idesc2, 1u);
      }
      ptx::umma_commit_w(&a_empty[as]);
      ptx::umma_commit_w(&tfull_bar[acc]);
      if (++as == kC11Stages) {
        as = 0;
        aph ^= 1;
      }
    }
  } else if (warp >= 4 && warp < 12) {
    run_epilogue<1, 128, BN, 1, true, 2>(p, &tm_o_hi, &tm_o_lo, &tm_o_x, staging, tfull_bar,
                                         tempty_bar, tmem_base, 0, first, stride, total_tiles);
  } else if (warp >= 12) {
    // -------------------------------------------------------------- A producers (128 threads)
    // two producer groups (warps 12..15, 16..19): group g builds the tiles with local index
    // parity g into ring stage g, so consecutive tiles are gathered / converted concurrently
    const int pg = (warp - 12) >> 2;
    const int pr = (threadIdx.x - 384) & 127;   // tile row = pixel within the 128-pixel row segment
    const long long plane = static_cast<long long>(H) * W;
    const int as = pg;
    uint32_t aph = 0;
    for (int t = first + pg * stride; t < total_tiles; t += 2 * stride) {
      const int img = t / p.tiles_w;             // one-row image index = b*H + h
      const int w = (t - img * p.tiles_w) * 128 + pr;
      const int b = img / H, h = img - b * H;
      // gather the patch first (global-load latency overlaps the wait for the stage)
      float v[27];
      const float* xb = data + static_cast<long long>(b) * 3 * plane;
#pragma unroll
      for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int ky = 0; ky < 3; ++ky)
#pragma unroll
          for (int kx = 0; kx < 3; ++kx) {
            const int hh = h + ky - 1, ww = w + kx - 1;
            const bool ok = hh >= 0 && hh < H && ww >= 0 && ww < W && w < W;
            v[c * 9 + ky * 3 + kx] = ok ? __ldg(xb + c * plane + static_cast<long long>(hh) * W + ww) : 0.f;
          }
      uint32_t hw[16], lw[16];   // 32 bf16 each, k = 27..31 are zero
#pragma unroll
      for (int e = 0; e < 16; ++e) {
        const float x0 = (2 * e < 27) ? v[2 * e] : 0.f;
        const float x1 = (2 * e + 1 < 27) ? v[(2 * e + 1 < 27) ? 2 * e + 1 : 0] : 0.f;
        const __nv_bfloat16 h0 = __float2bfloat16_rn(x0), h1 = __float2bfloat16_rn(x1);
        const __nv_bfloat16 l0 = __float2bfloat16_rn(x0 - __bfloat162float(h0));
        const __nv_bfloat16 l1 = __float2bfloat16_rn(x1 - __bfloat162float(h1));
        hw[e] = static_cast<uint32_t>(__bfloat16_as_ushort(h0)) |
                (static_cast<uint32_t>(__bfloat16_as_ushort(h1)) << 16);
        lw[e] = static_cast<uint32_t>(__bfloat16_as_ushort(l0)) |
                (static_cast<uint32_t>(__bfloat16_as_ushort(l1)) << 16);
      }
      ptx::mbar_wait(&a_empty[as], aph ^ 1);
      uint8_t* sa = a_ring + as * 2 * kC11ABytes;
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        const int off = pr * 64 + ((g ^ ((pr >> 1) & 3)) << 4);   // SWIZZLE_64B
        *reinterpret_cast<uint4*>(sa + off) = make_uint4(hw[4 * g], hw[4 * g + 1], hw[4 * g + 2], hw[4 * g + 3]);
        *reinterpret_cast<uint4*>(sa + kC11ABytes + off) =
            make_uint4(lw[4 * g], lw[4 * g + 1], lw[4 * g + 2], lw[4 * g + 3]);
      }
      ptx::fence_proxy_async();      // generic-proxy writes -> visible to the tensor core's async proxy
      ptx::mbar_arrive(&a_full[as]);
      aph ^= 1;
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc<256>(tmem_base);
  }
}

// ------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn == nullptr) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) !=
            cudaSuccess ||
        qres != cudaDriverEntryPointSuccess) {
      return nullptr;
    }
    fn = reinterpret_cast<EncodeTiledFn>(ptr);
  }
  return fn;
}

static CUtensorMapSwizzle swizzle_for_row(int row_bytes) {
  return row_bytes >= 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                          : (row_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
}

// [N][H][W][C] activation plane of `eb`-byte elements (2: bf16 / fp16, 1: e4m3), box
// [1][TH][TW][bk], swizzle mode = the box row width (bk * eb bytes), zero OOB fill.
static int make_act_map(CUtensorMap* m, const void* base, int N, int H, int W, int C, int TH,
                        int TW, int bk, int eb = 2) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) return MNC_ERR_DRIVER;
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  cuuint64_t strides[3] = {(cuuint64_t)C * eb, (cuuint64_t)W * C * eb, (cuuint64_t)H * W * C * eb};
  cuuint32_t box[4] = {(cuuint32_t)bk, (cuuint32_t)TW, (cuuint32_t)TH, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(m, eb == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_UINT8, 4,
                   const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   swizzle_for_row(bk * eb), CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? MNC_OK : MNC_ERR_DRIVER;
}

// [Cout][Ktot] weight plane, box [box_rows][bk].
static int make_wgt_map(CUtensorMap* m, const void* base, int Cout, long long Ktot, int box_rows,
                        int bk, int eb = 2) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) return MNC_ERR_DRIVER;
  cuuint64_t dims[2] = {(cuuint64_t)Ktot, (cuuint64_t)Cout};
  cuuint64_t strides[1] = {(cuuint64_t)Ktot * eb};
  cuuint32_t box[2] = {(cuuint32_t)bk, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, eb == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_UINT8, 2,
                   const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   swizzle_for_row(bk * eb), CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? MNC_OK : MNC_ERR_DRIVER;
}

// output plane seen as [N][H][W][Cout] with pixel stride `pix_stride` elements; box
// [1][TH][TW][32]: 2-byte planes with the 64-byte swizzle of the epilogue's staging layout,
// 1-byte planes (32-byte rows) unswizzled.
static int make_out_map(CUtensorMap* m, const void* base, int N, int H, int W, int Cout,
                        long long pix_stride, int TH, int TW, int eb = 2) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) return MNC_ERR_DRIVER;
  cuuint64_t dims[4] = {(cuuint64_t)Cout, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  cuuint64_t strides[3] = {(cuuint64_t)pix_stride * eb, (cuuint64_t)W * pix_stride * eb,
                           (cuuint64_t)H * W * pix_stride * eb};
  cuuint32_t box[4] = {32, (cuuint32_t)TW, (cuuint32_t)TH, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(m, eb == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_UINT8, 4,
                   const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   eb == 2 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_NONE,
                   CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? MNC_OK : MNC_ERR_DRIVER;
}

static int sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
  }
  return n;
}

struct Maps {
  CUtensorMap a[3], b[3], o[3];
};

template <int TH, int TW, int BN, int CL, int BK, int PM>
static int launch_igemm(const Maps& m, const IgemmArgs& a, int max_ctas, cudaStream_t stream) {
  using Cfg = IgemmCfg<BN, BK, CL>;
  auto kern = igemm_tc_kernel<TH, TW, BN, CL, BK, PM>;
  static SmemGrant grant;
  if (!ensure_dynamic_smem(kern, Cfg::kSmemBytes, grant)) return MNC_ERR_CUDA;
  const int spatial = a.batch * a.tiles_h * a.tiles_w;
  const int total = a.split_k * a.tiles_n * ((spatial + CL - 1) / CL);
  int grid = sm_count();
  if (max_ctas > 0 && max_ctas < grid) grid = max_ctas;
  if (total * CL < grid) grid = total * CL;
  grid = (grid / CL) * CL;
  if (grid < CL) grid = CL;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(256);
  cfg.dynamicSmemBytes = Cfg::kSmemBytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CL;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, m.a[0], m.a[1], m.a[2], m.b[0], m.b[1], m.b[2],
                                     m.o[0], m.o[1], m.o[2], a);
  return e == cudaSuccess ? MNC_OK : MNC_ERR_CUDA;
}

template <int BN, int PM, int CL>
static int launch_halo(const Maps& m, const IgemmArgs& a, int max_ctas, cudaStream_t stream) {
  using Cfg = HaloCfg<BN, PM, CL>;
  auto kern = conv_halo_tc_kernel<BN, PM, CL>;
  static SmemGrant grant;
  if (!ensure_dynamic_smem(kern, Cfg::kSmemBytes, grant)) return MNC_ERR_CUDA;
  const int spatial = a.batch * a.tiles_h * a.tiles_w;
  const int total = a.tiles_n * ((spatial + CL - 1) / CL);
  int grid = sm_count();
  if (max_ctas > 0 && max_ctas < grid) grid = max_ctas;
  if (total * CL < grid) grid = total * CL;
  grid = (grid / CL) * CL;
  if (grid < CL) grid = CL;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(384);
  cfg.dynamicSmemBytes = Cfg::kSmemBytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CL;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, m.a[0], m.a[1], m.a[2], m.b[0], m.b[1], m.b[2],
                                     m.o[0], m.o[1], m.o[2], a);
  return e == cudaSuccess ? MNC_OK : MNC_ERR_CUDA;
}

}  // namespace mnc

using namespace mnc;

// Cluster size used by mnc_igemm_tc launches (1 or 2).  2 = pairs of CTAs along the pixel/row
// dimension share each weight tile through TMA multicast (halves weight traffic from L2).
static int g_igemm_cluster = 2;
static int g_halo_pair = 1;
static int g_igemm_bk = 0;  // 0 = per-shape default
static int g_igemm_halo = 1;  // halo-reuse kernel for 3x3 convs with Cout tiles <= 128
extern "C" int mnc_igemm_set_halo(int on) {
  g_igemm_halo = on ? 1 : 0;
  return MNC_OK;
}
static int g_igemm_tma_store = 1;
extern "C" int mnc_igemm_set_tma_store(int on) {
  g_igemm_tma_store = on ? 1 : 0;
  return MNC_OK;
}
extern "C" int mnc_igemm_set_cluster(int cl) {
  if (cl != 1 && cl != 2) return MNC_ERR_ARG;
  g_igemm_cluster = cl;
  return MNC_OK;
}
// A/B switch: CTA pairs in the halo kernel (precision mode 1; on by default, off = one CTA per tile)
extern "C" int mnc_igemm_set_halo_pair(int on) {
  g_halo_pair = on ? 1 : 0;
  return MNC_OK;
}

// K elements per pipeline stage for mnc_igemm_tc launches: 64, 32, or 0 = default (64; the
// 192-wide Cout tile exists only with 32).
extern "C" int mnc_igemm_set_block_k(int bk) {
  if (bk != 0 && bk != 32 && bk != 64) return MNC_ERR_ARG;
  g_igemm_bk = bk;
  return MNC_OK;
}

// General form.  in_fmt 0: operands are split-bf16 planes (a0 = hi, a1 = lo; w0 = hi, w1 = lo);
// in_fmt 1: tri-plane operands (a0 = fp16 value, a1 = e4m3 residual, a2 = e4m3 copy; w0 = fp16,
// w1 = e4m3 copy, w2 = e4m3 residual -- layouts above).  out_mode 0 / 2: split-bf16 (out0 = hi,
// out1 = lo), 1: fp32 (out0), 4 / 5: tri-plane (out0 = fp16, out1 = residual, out2 = copy) with
// exponent scale `out_scale`; 2 and 5 apply the fused 2x2 ceil-mode max pool.  acc_scale turns the
// accumulator into the true value (2^-(ea+ew) for tri-plane operands, 1 otherwise).  amax
// (optional, device) receives atomicMax(|output|) as float bits.
// img_hw (optional, device int32 [batch][2]) + level: per-image extents of a mixed-size batch
// (IgemmArgs::img_hw); nullptr = the whole blob.
extern "C" int mnc_igemm_tc3(int in_fmt, const void* a0, const void* a1, const void* a2, int batch,
                             int H, int W, int Cin, const void* w0, const void* w1, const void* w2,
                             int Cout, int taps, const float* bias, int relu, int out_mode,
                             void* out0, void* out1, void* out2, long long out_pix_stride,
                             int out_ch_offset, int split_k, long long split_stride, int bn,
                             int max_ctas, float acc_scale, float out_scale, unsigned int* amax,
                             const int* img_hw, int level, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (Cin % 64 != 0 || (taps != 1 && taps != 9) || batch <= 0 || H <= 0 || W <= 0 || Cout <= 0)
    return MNC_ERR_ARG;
  if (level < 0 || level > 16) return MNC_ERR_ARG;
  if (in_fmt != 0 && in_fmt != 1) return MNC_ERR_ARG;
  if (out_mode != 0 && out_mode != 1 && out_mode != 2 && out_mode != 3 && out_mode != 4 && out_mode != 5)
    return MNC_ERR_ARG;
  const bool tri_out = (out_mode == 4 || out_mode == 5);
  const bool pooled = (out_mode == 2 || out_mode == 5);
  int bk = g_igemm_bk;
  if (split_k < 1) split_k = 1;
  if (split_k > 1 && out_mode != 1) return MNC_ERR_ARG;
  if (pooled && (taps != 9 || Cout % 8 != 0 || out_pix_stride % 8 != 0 || out_ch_offset % 8 != 0))
    return MNC_ERR_ARG;
  if (tri_out && (out_pix_stride % 16 != 0 || out_ch_offset % 16 != 0 ||
                  (reinterpret_cast<uintptr_t>(out0) | reinterpret_cast<uintptr_t>(out1) |
                   reinterpret_cast<uintptr_t>(out2)) % 16 != 0))
    return MNC_ERR_ARG;
  const bool conv = (taps == 9);
  if (bn == 0) bn = (Cout <= 64) ? 64 : (Cout <= 128 ? 128 : 256);
  const bool halo = conv && g_igemm_halo && (bn == 64 || bn == 128) && split_k == 1;
  const int TH = conv ? (halo ? kHaloTH : 8) : 1, TW = conv ? (halo ? kHaloTW : 16) : 128;
  if (bn != 64 && bn != 128 && bn != 192 && bn != 256) return MNC_ERR_ARG;
  const bool bk_forced = (bk != 0);
  if (bk == 0) bk = 64;              // measured: BLOCK_K 64 wins at BN 256 (profiles/r01_igemm_bk32_bn192.log)
  // BN 192: a CTA pair holds 96 weight rows each, so 64-wide stages fit three deep (and keep the
  // FP8 planes' rows at 64 B -- 32-byte rows cost 27 % more L2 sectors, r02 ncu); a single CTA
  // needs the half-size stages
  if (bn == 192 && !bk_forced) bk = (g_igemm_cluster == 2) ? 64 : 32;
  if (bn < 128 || (bn == 128 && conv)) bk = 64;

  IgemmArgs a;
  a.batch = batch;
  a.H = H;
  a.W = W;
  a.Cin = Cin;
  a.Cout = Cout;
  a.taps = taps;
  a.tiles_h = (H + TH - 1) / TH;
  a.tiles_w = (W + TW - 1) / TW;
  a.tiles_n = (Cout + bn - 1) / bn;
  a.k_steps = taps * (Cin / bk);
  if (split_k > a.k_steps) split_k = a.k_steps;
  a.split_k = split_k;
  a.relu = relu;
  a.out_mode = out_mode;
  a.bias = bias;
  a.out_hi = static_cast<__nv_bfloat16*>(out0);
  a.out_lo = static_cast<__nv_bfloat16*>(out1);
  a.out_x = static_cast<uint8_t*>(out2);
  a.out_f32 = static_cast<float*>(out0);
  a.out_pix_stride = out_pix_stride;
  a.out_ch_offset = out_ch_offset;
  a.split_stride = split_stride;
  a.acc_scale = acc_scale;
  a.out_scale = out_scale;
  a.amax = amax;
  a.img_hw = img_hw;
  a.level = level;
  a.img_rows = 0;
  const int vec = (out_mode == 1) ? 4 : 8;
  a.vec_ok = (out_pix_stride % vec == 0) && (out_ch_offset % vec == 0) &&
             (reinterpret_cast<uintptr_t>(out0) % 16 == 0) &&
             (out_mode == 1 || reinterpret_cast<uintptr_t>(out1) % 16 == 0) &&
             (split_stride % vec == 0);

  Maps m;
  int rc;
  if (halo) bk = 64;
  // halo kernel: the activation box is the pixel tile plus a one-pixel border
  const int box_h = halo ? TH + 2 : TH, box_w = halo ? TW + 2 : TW;
  if ((rc = make_act_map(&m.a[0], a0, batch, H, W, Cin, box_h, box_w, bk, 2)) != MNC_OK) return rc;
  if ((rc = make_act_map(&m.a[1], a1, batch, H, W, Cin, box_h, box_w, bk, in_fmt ? 1 : 2)) != MNC_OK)
    return rc;
  m.a[2] = m.a[1];
  if (in_fmt == 1 && (rc = make_act_map(&m.a[2], a2, batch, H, W, Cin, box_h, box_w, bk, 1)) != MNC_OK)
    return rc;
  const long long ktot = static_cast<long long>(taps) * Cin;
  // epilogue through shared memory + TMA store when the output planes allow a tensor map
  m.o[0] = m.a[0];  // placeholders when unused
  m.o[1] = m.a[1];
  m.o[2] = m.a[1];
  a.tma_store = 0;
  if (out_mode == 0 && g_igemm_tma_store && out_pix_stride % 8 == 0 && out_ch_offset % 8 == 0 &&
      reinterpret_cast<uintptr_t>(out0) % 16 == 0 && reinterpret_cast<uintptr_t>(out1) % 16 == 0) {
    const __nv_bfloat16* bh = static_cast<const __nv_bfloat16*>(out0) + out_ch_offset;
    const __nv_bfloat16* bl = static_cast<const __nv_bfloat16*>(out1) + out_ch_offset;
    if (make_out_map(&m.o[0], bh, batch, H, W, Cout, out_pix_stride, TH, TW) == MNC_OK &&
        make_out_map(&m.o[1], bl, batch, H, W, Cout, out_pix_stride, TH, TW) == MNC_OK)
      a.tma_store = 1;
  }
  if (out_mode == 4) {
    const __nv_bfloat16* bh = static_cast<const __nv_bfloat16*>(out0) + out_ch_offset;
    const uint8_t* bl = static_cast<const uint8_t*>(out1) + out_ch_offset;
    const uint8_t* bc = static_cast<const uint8_t*>(out2) + out_ch_offset;
    if (make_out_map(&m.o[0], bh, batch, H, W, Cout, out_pix_stride, TH, TW, 2) != MNC_OK ||
        make_out_map(&m.o[1], bl, batch, H, W, Cout, out_pix_stride, TH, TW, 1) != MNC_OK ||
        make_out_map(&m.o[2], bc, batch, H, W, Cout, out_pix_stride, TH, TW, 1) != MNC_OK)
      return MNC_ERR_DRIVER;
    a.tma_store = 1;
  }
  // halo kernel: CTA pairs exist for precision mode 1 only
  const int cl = halo ? ((in_fmt == 1 && g_igemm_cluster == 2 && g_halo_pair) ? 2 : 1) : g_igemm_cluster;
  if ((rc = make_wgt_map(&m.b[0], w0, Cout, ktot, bn / cl, bk, 2)) != MNC_OK) return rc;
  if ((rc = make_wgt_map(&m.b[1], w1, Cout, ktot, bn / cl, bk, in_fmt ? 1 : 2)) != MNC_OK) return rc;
  m.b[2] = m.b[1];
  if (in_fmt == 1 && (rc = make_wgt_map(&m.b[2], w2, Cout, ktot, bn / cl, bk, 1)) != MNC_OK) return rc;
  if (halo) {
    a.k_steps = 9 * (Cin / 64);
    if (in_fmt == 1 && cl == 2) {
      if (bn == 64) return launch_halo<64, 1, 2>(m, a, max_ctas, stream);
      return launch_halo<128, 1, 2>(m, a, max_ctas, stream);
    }
    if (in_fmt == 1) {
      if (bn == 64) return launch_halo<64, 1, 1>(m, a, max_ctas, stream);
      return launch_halo<128, 1, 1>(m, a, max_ctas, stream);
    }
    if (bn == 64) return launch_halo<64, 0, 1>(m, a, max_ctas, stream);
    return launch_halo<128, 0, 1>(m, a, max_ctas, stream);
  }

#define MNC_LAUNCH_PM(TH_, TW_, BN_, BK_, PM_)                                      \
  return (cl == 2) ? launch_igemm<TH_, TW_, BN_, 2, BK_, PM_>(m, a, max_ctas, stream) \
                   : launch_igemm<TH_, TW_, BN_, 1, BK_, PM_>(m, a, max_ctas, stream)
#define MNC_LAUNCH(TH_, TW_, BN_, BK_)                          \
  do {                                                          \
    if (in_fmt == 1) MNC_LAUNCH_PM(TH_, TW_, BN_, BK_, 1);      \
    MNC_LAUNCH_PM(TH_, TW_, BN_, BK_, 0);                       \
  } while (0)
  if (conv) {
    if (bn == 64) MNC_LAUNCH(8, 16, 64, 64);
    if (bn == 128) MNC_LAUNCH(8, 16, 128, 64);
    if (bn == 192 && bk == 32) MNC_LAUNCH(8, 16, 192, 32);
    if (bn == 192) MNC_LAUNCH(8, 16, 192, 64);
    if (bk == 32) MNC_LAUNCH(8, 16, 256, 32);
    MNC_LAUNCH(8, 16, 256, 64);
  } else {
    if (bn == 64) MNC_LAUNCH(1, 128, 64, 64);
    if (bn == 128 && bk == 32) MNC_LAUNCH(1, 128, 128, 32);
    if (bn == 128) MNC_LAUNCH(1, 128, 128, 64);
    if (bn == 192 && bk == 32) MNC_LAUNCH(1, 128, 192, 32);
    if (bn == 192) MNC_LAUNCH(1, 128, 192, 64);
    if (bk == 32) MNC_LAUNCH(1, 128, 256, 32);
    MNC_LAUNCH(1, 128, 256, 64);
  }
#undef MNC_LAUNCH
#undef MNC_LAUNCH_PM
}

extern "C" int mnc_igemm_tc2(int in_fmt, const void* a0, const void* a1, const void* a2, int batch,
                             int H, int W, int Cin, const void* w0, const void* w1, const void* w2,
                             int Cout, int taps, const float* bias, int relu, int out_mode,
                             void* out0, void* out1, void* out2, long long out_pix_stride,
                             int out_ch_offset, int split_k, long long split_stride, int bn,
                             int max_ctas, float acc_scale, float out_scale, unsigned int* amax,
                             void* stream_) {
  return mnc_igemm_tc3(in_fmt, a0, a1, a2, batch, H, W, Cin, w0, w1, w2, Cout, taps, bias, relu,
                       out_mode, out0, out1, out2, out_pix_stride, out_ch_offset, split_k,
                       split_stride, bn, max_ctas, acc_scale, out_scale, amax, nullptr, 0, stream_);
}

// Split-bf16 operands, outputs 0 / 1 / 2 (the round-1 entry point; kept for its callers).
extern "C" int mnc_igemm_tc(const void* a_hi, const void* a_lo, int batch, int H, int W, int Cin,
                            const void* w_hi, const void* w_lo, int Cout, int taps,
                            const float* bias, int relu, int out_mode, void* out0, void* out1,
                            long long out_pix_stride, int out_ch_offset, int split_k,
                            long long split_stride, int bn, int max_ctas, void* stream_) {
  return mnc_igemm_tc2(0, a_hi, a_lo, nullptr, batch, H, W, Cin, w_hi, w_lo, nullptr, Cout, taps,
                       bias, relu, out_mode, out0, out1, nullptr, out_pix_stride, out_ch_offset,
                       split_k, split_stride, bn, max_ctas, 1.0f, 1.0f, nullptr, stream_);
}

// conv1_1 on the tensor cores.  w_stacked: bf16 [128][32] = rows 0..63 the hi plane, 64..127 the lo
// plane of weight.reshape(64, 27) (k = c*9 + ky*3 + kx), columns 27..31 zero.
// out_mode 0: split-bf16 planes (out0 = hi, out1 = lo); 4: tri-plane (out0 = fp16, out1 = e4m3
// residual, out2 = e4m3 copy) scaled by out_scale.  amax (optional, device): atomicMax(|output|).
// img_hw (optional, device int32 [batch][2]): per-image sizes of a mixed-size batch; output pixels
// outside their image are written as zeros.
extern "C" int mnc_conv1_1_tc3(const float* data_nchw, int batch, int H, int W, const void* w_stacked,
                               const float* bias, int out_mode, void* out0, void* out1, void* out2,
                               float out_scale, unsigned int* amax, const int* img_hw, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (batch <= 0 || H <= 0 || W <= 0 || (out_mode != 0 && out_mode != 4)) return MNC_ERR_ARG;
  if ((reinterpret_cast<uintptr_t>(out0) | reinterpret_cast<uintptr_t>(out1) |
       reinterpret_cast<uintptr_t>(w_stacked)) % 16 != 0)
    return MNC_ERR_ARG;
  if (out_mode == 4 && (out2 == nullptr || reinterpret_cast<uintptr_t>(out2) % 16 != 0)) return MNC_ERR_ARG;
  IgemmArgs a;
  a.batch = batch * H;   // one-row images
  a.H = 1;
  a.W = W;
  a.Cin = 32;
  a.Cout = 64;
  a.taps = 1;
  a.tiles_h = 1;
  a.tiles_w = (W + 127) / 128;
  a.tiles_n = 1;
  a.k_steps = 1;
  a.split_k = 1;
  a.relu = 1;
  a.out_mode = out_mode;
  a.bias = bias;
  a.out_hi = static_cast<__nv_bfloat16*>(out0);
  a.out_lo = static_cast<__nv_bfloat16*>(out1);
  a.out_f32 = nullptr;
  a.out_pix_stride = 64;
  a.out_ch_offset = 0;
  a.split_stride = 0;
  a.vec_ok = 1;
  a.tma_store = 1;
  a.out_x = static_cast<uint8_t*>(out2);
  a.acc_scale = 1.0f;
  a.out_scale = out_scale;
  a.amax = amax;
  a.img_hw = img_hw;
  a.level = 0;
  a.img_rows = H;
  CUtensorMap tb, to_hi, to_lo, to_x;
  int rc;
  const int eb = (out_mode == 4) ? 1 : 2;
  if ((rc = make_wgt_map(&tb, w_stacked, 128, 32, 128, 32)) != MNC_OK) return rc;
  if ((rc = make_out_map(&to_hi, out0, a.batch, 1, W, 64, 64, 1, 128, 2)) != MNC_OK) return rc;
  if ((rc = make_out_map(&to_lo, out1, a.batch, 1, W, 64, 64, 1, 128, eb)) != MNC_OK) return rc;
  to_x = to_lo;
  if (out_mode == 4 && (rc = make_out_map(&to_x, out2, a.batch, 1, W, 64, 64, 1, 128, 1)) != MNC_OK) return rc;
  static SmemGrant grant;
  if (!ensure_dynamic_smem(conv1_1_tc_kernel, kC11Smem, grant)) return MNC_ERR_CUDA;
  const int total = a.batch * a.tiles_w;
  int grid = sm_count();
  if (total < grid) grid = total;
  conv1_1_tc_kernel<<<grid, kC11Threads, kC11Smem, stream>>>(data_nchw, batch, H, W, tb, to_hi, to_lo,
                                                             to_x, a);
  return cudaGetLastError() == cudaSuccess ? MNC_OK : MNC_ERR_CUDA;
}

extern "C" int mnc_conv1_1_tc2(const float* data_nchw, int batch, int H, int W, const void* w_stacked,
                               const float* bias, int out_mode, void* out0, void* out1, void* out2,
                               float out_scale, unsigned int* amax, void* stream_) {
  return mnc_conv1_1_tc3(data_nchw, batch, H, W, w_stacked, bias, out_mode, out0, out1, out2,
                         out_scale, amax, nullptr, stream_);
}

extern "C" int mnc_conv1_1_tc(const float* data_nchw, int batch, int H, int W, const void* w_stacked,
                              const float* bias, void* out_hi, void* out_lo, void* stream_) {
  return mnc_conv1_1_tc2(data_nchw, batch, H, W, w_stacked, bias, 0, out_hi, out_lo, nullptr, 1.0f,
                         nullptr, stream_);
}
