// SIMT companions of the tensor-core path: conv1_1 (Cin = 3), 2x2 ceil-mode max pooling on
// split NHWC, split-K reduction, layout converters, and an fp32-FMA implicit GEMM with the same
// contract as mnc_igemm_tc that serves as the on-device cross-check.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <cstdint>

#include "mnc_b200.h"

namespace mnc {

__device__ __forceinline__ float bf2f(__nv_bfloat16 x) { return __bfloat162float(x); }
__device__ __forceinline__ void split_f32(float x, __nv_bfloat16& hi, __nv_bfloat16& lo) {
  hi = __float2bfloat16_rn(x);
  lo = __float2bfloat16_rn(x - __bfloat162float(hi));
}

// ------------------------------------------------------------------ SIMT igemm
// 64 pixels x 64 output channels per CTA, 16x16 threads, 4x4 outputs per thread.
__global__ void __launch_bounds__(256)
igemm_simt_kernel(const __nv_bfloat16* __restrict__ a_hi, const __nv_bfloat16* __restrict__ a_lo,
                  int batch, int H, int W, int Cin, const __nv_bfloat16* __restrict__ w_hi,
                  const __nv_bfloat16* __restrict__ w_lo, int Cout, int taps,
                  const float* __restrict__ bias, int relu, int out_mode, void* out0, void* out1,
                  long long out_pix_stride, int out_ch_offset) {
  __shared__ float As[16][64 + 4];
  __shared__ float Bs[16][64 + 4];
  const long long M = static_cast<long long>(batch) * H * W;
  const long long m0 = static_cast<long long>(blockIdx.x) * 64;
  const int n0 = blockIdx.y * 64;
  const int tid = threadIdx.x;
  const int tx = tid % 16, ty = tid / 16;
  const long long Ktot = static_cast<long long>(taps) * Cin;

  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  const int lp = tid / 4;        // local pixel / cout row loaded by this thread
  const int lc = (tid % 4) * 4;  // 4 consecutive channels
  const long long m = m0 + lp;
  int img = 0, h = 0, w = 0;
  if (m < M) {
    img = static_cast<int>(m / (static_cast<long long>(H) * W));
    const int r = static_cast<int>(m % (static_cast<long long>(H) * W));
    h = r / W;
    w = r % W;
  }
  for (int tap = 0; tap < taps; ++tap) {
    const int dy = (taps == 9) ? tap / 3 - 1 : 0;
    const int dx = (taps == 9) ? tap % 3 - 1 : 0;
    const int hs = h + dy, ws = w + dx;
    const bool in_ok = (m < M) && hs >= 0 && hs < H && ws >= 0 && ws < W;
    const long long a_off = ((static_cast<long long>(img) * H + hs) * W + ws) * Cin;
    for (int c0 = 0; c0 < Cin; c0 += 16) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        float av = 0.f;
        if (in_ok) av = bf2f(a_hi[a_off + c0 + lc + e]) + bf2f(a_lo[a_off + c0 + lc + e]);
        As[lc + e][lp] = av;
        float bv = 0.f;
        if (n0 + lp < Cout) {
          const long long b_off = static_cast<long long>(n0 + lp) * Ktot + tap * Cin + c0 + lc + e;
          bv = bf2f(w_hi[b_off]) + bf2f(w_lo[b_off]);
        }
        Bs[lc + e][lp] = bv;
      }
      __syncthreads();
#pragma unroll
      for (int k = 0; k < 16; ++k) {
        float a[4], b[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) a[i] = As[k][ty * 4 + i];
#pragma unroll
        for (int j = 0; j < 4; ++j) b[j] = Bs[k][tx * 4 + j];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
      }
      __syncthreads();
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long long mm = m0 + ty * 4 + i;
    if (mm >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int ch = n0 + tx * 4 + j;
      if (ch >= Cout) continue;
      float v = acc[i][j];
      if (bias) v += bias[ch];
      if (relu) v = fmaxf(v, 0.f);
      const long long o = mm * out_pix_stride + out_ch_offset + ch;
      if (out_mode == 0) {
        __nv_bfloat16 hi, lo;
        split_f32(v, hi, lo);
        static_cast<__nv_bfloat16*>(out0)[o] = hi;
        static_cast<__nv_bfloat16*>(out1)[o] = lo;
      } else {
        static_cast<float*>(out0)[o] = v;
      }
    }
  }
}

// ---------------------------------------------------------------- split-K sum
// out = act(sum_s partial[s] + bias).  One thread per 4 consecutive columns (cols % 4 == 0 fast
// path: 16-byte loads of each partial plane, 8-byte stores to both bf16 planes), rows on grid.y.
__global__ void __launch_bounds__(256)
splitk_reduce_kernel(const float* __restrict__ partial, int splits, long long split_stride,
                     long long rows, int cols, const float* __restrict__ bias, int relu,
                     int out_mode, void* out0, void* out1, long long out_row_stride,
                     int out_ch_offset, int vec, const int* __restrict__ img_hw, int level, int H,
                     int W) {
  const int c4 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (c4 >= cols) return;
  for (long long r = blockIdx.y; r < rows; r += gridDim.y) {
    // conv launches of mixed-size batches: row r is pixel (b, y, x); outside image b -> zeros
    bool inside = true;
    if (img_hw != nullptr) {
      const long long hw = static_cast<long long>(H) * W;
      const int b = static_cast<int>(r / hw), pr = static_cast<int>(r - b * hw);
      const int m = (1 << level) - 1;
      inside = pr / W < ((__ldg(img_hw + 2 * b) + m) >> level) &&
               pr % W < ((__ldg(img_hw + 2 * b + 1) + m) >> level);
    }
    float v[4] = {0.f, 0.f, 0.f, 0.f};
    const float* p = partial + r * cols + c4;
    if (vec) {
#pragma unroll 8   // loads of 8 splits in flight (a 32-way split was 32 dependent L2 round trips)
      for (int s = 0; s < splits; ++s) {  // fixed order: deterministic
        const float4 x = __ldcs(reinterpret_cast<const float4*>(p + s * split_stride));
        v[0] += x.x;
        v[1] += x.y;
        v[2] += x.z;
        v[3] += x.w;
      }
    } else {
      for (int s = 0; s < splits; ++s)
        for (int e = 0; e < 4 && c4 + e < cols; ++e) v[e] += p[s * split_stride + e];
    }
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      if (bias && c4 + e < cols) v[e] += __ldg(bias + c4 + e);
      if (relu) v[e] = fmaxf(v[e], 0.f);
      if (!inside) v[e] = 0.f;
    }
    const long long o = r * out_row_stride + out_ch_offset + c4;
    if (out_mode == 0) {
      __nv_bfloat16 hi[4], lo[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) split_f32(v[e], hi[e], lo[e]);
      if (vec) {
        *reinterpret_cast<uint2*>(static_cast<__nv_bfloat16*>(out0) + o) = make_uint2(
            static_cast<uint32_t>(__bfloat16_as_ushort(hi[0])) | (static_cast<uint32_t>(__bfloat16_as_ushort(hi[1])) << 16),
            static_cast<uint32_t>(__bfloat16_as_ushort(hi[2])) | (static_cast<uint32_t>(__bfloat16_as_ushort(hi[3])) << 16));
        *reinterpret_cast<uint2*>(static_cast<__nv_bfloat16*>(out1) + o) = make_uint2(
            static_cast<uint32_t>(__bfloat16_as_ushort(lo[0])) | (static_cast<uint32_t>(__bfloat16_as_ushort(lo[1])) << 16),
            static_cast<uint32_t>(__bfloat16_as_ushort(lo[2])) | (static_cast<uint32_t>(__bfloat16_as_ushort(lo[3])) << 16));
      } else {
        for (int e = 0; e < 4 && c4 + e < cols; ++e) {
          static_cast<__nv_bfloat16*>(out0)[o + e] = hi[e];
          static_cast<__nv_bfloat16*>(out1)[o + e] = lo[e];
        }
      }
    } else {
      if (vec) {
        *reinterpret_cast<float4*>(static_cast<float*>(out0) + o) = make_float4(v[0], v[1], v[2], v[3]);
      } else {
        for (int e = 0; e < 4 && c4 + e < cols; ++e) static_cast<float*>(out0)[o + e] = v[e];
      }
    }
  }
}

// -------------------------------------------------------------------- conv1_1
// Weight-stationary SIMT kernel.  Lane l of every warp owns output channels 2l and 2l+1 and keeps
// their 2x27 weights in registers for the whole CTA; the CTA stages a (8+2) x (64+2) x 3 input
// tile in shared memory and each warp walks one 64-pixel row, 4 pixels per step.  All lanes read
// the same input words (broadcast 128/64-bit shared loads, ~4.5 wavefronts per pixel) against
// 54 FMAs per lane per pixel, so the kernel is FMA-issue bound; a warp's store for one pixel is
// one contiguous 128-byte NHWC row per bf16 plane.  Input is the fp32 NCHW `data` blob.
constexpr int kC11TH = 8, kC11TW = 64;

__global__ void __launch_bounds__(256)
conv1_1_kernel(const float* __restrict__ data, int batch, int H, int W,
               const float* __restrict__ weight, const float* __restrict__ bias,
               __nv_bfloat16* __restrict__ out_hi, __nv_bfloat16* __restrict__ out_lo) {
  constexpr int COUT = 64;
  constexpr int SW = kC11TW + 4;  // row pitch: 66 used, padded to 68 so rows stay 16B-aligned
  __shared__ __align__(16) float tile[3][kC11TH + 2][SW];
  const int tiles_w = (W + kC11TW - 1) / kC11TW;
  const int tiles_h = (H + kC11TH - 1) / kC11TH;
  const int img = blockIdx.x / (tiles_h * tiles_w);
  const int tr = blockIdx.x % (tiles_h * tiles_w);
  const int h0 = (tr / tiles_w) * kC11TH, w0 = (tr % tiles_w) * kC11TW;
  const long long HW = static_cast<long long>(H) * W;
  for (int i = threadIdx.x; i < 3 * (kC11TH + 2) * (kC11TW + 2); i += blockDim.x) {
    const int c = i / ((kC11TH + 2) * (kC11TW + 2));
    const int rem = i % ((kC11TH + 2) * (kC11TW + 2));
    const int y = rem / (kC11TW + 2), x = rem % (kC11TW + 2);
    const int hs = h0 + y - 1, wsx = w0 + x - 1;
    float v = 0.f;
    if (hs >= 0 && hs < H && wsx >= 0 && wsx < W)
      v = __ldg(data + (static_cast<long long>(img) * 3 + c) * HW + static_cast<long long>(hs) * W + wsx);
    tile[c][y][x] = v;
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float w0r[27], w1r[27];  // Caffe weight order [co][c][ky][kx]
#pragma unroll
  for (int k = 0; k < 27; ++k) {
    w0r[k] = __ldg(weight + (2 * lane) * 27 + k);
    w1r[k] = __ldg(weight + (2 * lane + 1) * 27 + k);
  }
  const float b0 = bias ? __ldg(bias + 2 * lane) : 0.f;
  const float b1 = bias ? __ldg(bias + 2 * lane + 1) : 0.f;
  __syncthreads();
  const int y = warp;  // 8 warps <-> 8 tile rows
  const int h = h0 + y;
  if (h >= H) return;
#pragma unroll 1
  for (int x0 = 0; x0 < kC11TW; x0 += 4) {
    if (w0 + x0 >= W) break;
    float a0[4] = {0.f, 0.f, 0.f, 0.f}, a1[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
      for (int ky = 0; ky < 3; ++ky) {
        // 6 consecutive inputs x0 .. x0+5 of row y+ky (tile column x0 is image column w0+x0-1)
        const float4 v4 = *reinterpret_cast<const float4*>(&tile[c][y + ky][x0]);
        const float2 v2 = *reinterpret_cast<const float2*>(&tile[c][y + ky][x0 + 4]);
        const float in[6] = {v4.x, v4.y, v4.z, v4.w, v2.x, v2.y};
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
          const int k = c * 9 + ky * 3 + kx;
#pragma unroll
          for (int p = 0; p < 4; ++p) {
            a0[p] = fmaf(in[p + kx], w0r[k], a0[p]);
            a1[p] = fmaf(in[p + kx], w1r[k], a1[p]);
          }
        }
      }
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      const int w = w0 + x0 + p;
      if (w >= W) break;
      const long long pix = (static_cast<long long>(img) * H + h) * W + w;
      const float x0v = fmaxf(a0[p] + b0, 0.f), x1v = fmaxf(a1[p] + b1, 0.f);
      __nv_bfloat16 hh0, ll0, hh1, ll1;
      split_f32(x0v, hh0, ll0);
      split_f32(x1v, hh1, ll1);
      *reinterpret_cast<uint32_t*>(out_hi + pix * COUT + 2 * lane) =
          static_cast<uint32_t>(__bfloat16_as_ushort(hh0)) | (static_cast<uint32_t>(__bfloat16_as_ushort(hh1)) << 16);
      *reinterpret_cast<uint32_t*>(out_lo + pix * COUT + 2 * lane) =
          static_cast<uint32_t>(__bfloat16_as_ushort(ll0)) | (static_cast<uint32_t>(__bfloat16_as_ushort(ll1)) << 16);
    }
  }
}

// ------------------------------------------------------------- 2x2 max pooling
// One thread per (pixel, 8-channel group); 16-byte loads/stores on both planes.
__global__ void maxpool2x2_split_kernel(const __nv_bfloat16* __restrict__ in_hi,
                                        const __nv_bfloat16* __restrict__ in_lo, int batch, int H,
                                        int W, int C, __nv_bfloat16* __restrict__ out_hi,
                                        __nv_bfloat16* __restrict__ out_lo) {
  const int Ho = (H + 1) / 2, Wo = (W + 1) / 2, C8 = C / 8;
  const long long total = static_cast<long long>(batch) * Ho * Wo * C8;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int cg = static_cast<int>(i % C8);
    long long r = i / C8;
    const int wo = static_cast<int>(r % Wo);
    r /= Wo;
    const int ho = static_cast<int>(r % Ho);
    const int img = static_cast<int>(r / Ho);
    float best[8];
    uint16_t bh[8], bl[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      best[j] = -3.402823466e+38f;
      bh[j] = 0;
      bl[j] = 0;
    }
    for (int dy = 0; dy < 2; ++dy) {
      const int h = ho * 2 + dy;
      if (h >= H) continue;
      for (int dx = 0; dx < 2; ++dx) {
        const int w = wo * 2 + dx;
        if (w >= W) continue;
        const long long off = ((static_cast<long long>(img) * H + h) * W + w) * C + cg * 8;
        const uint4 vh = *reinterpret_cast<const uint4*>(in_hi + off);
        const uint4 vl = *reinterpret_cast<const uint4*>(in_lo + off);
        const uint32_t hw[4] = {vh.x, vh.y, vh.z, vh.w};
        const uint32_t lw[4] = {vl.x, vl.y, vl.z, vl.w};
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const uint16_t hb = static_cast<uint16_t>(hw[j / 2] >> ((j & 1) * 16));
          const uint16_t lb = static_cast<uint16_t>(lw[j / 2] >> ((j & 1) * 16));
          const float v = __uint_as_float(static_cast<uint32_t>(hb) << 16) +
                          __uint_as_float(static_cast<uint32_t>(lb) << 16);
          if (v > best[j]) {  // first maximum wins, as pooling_layer.cu:36
            best[j] = v;
            bh[j] = hb;
            bl[j] = lb;
          }
        }
      }
    }
    uint32_t oh[4], ol[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      oh[e] = static_cast<uint32_t>(bh[2 * e]) | (static_cast<uint32_t>(bh[2 * e + 1]) << 16);
      ol[e] = static_cast<uint32_t>(bl[2 * e]) | (static_cast<uint32_t>(bl[2 * e + 1]) << 16);
    }
    const long long o = ((static_cast<long long>(img) * Ho + ho) * Wo + wo) * C + cg * 8;
    *reinterpret_cast<uint4*>(out_hi + o) = make_uint4(oh[0], oh[1], oh[2], oh[3]);
    *reinterpret_cast<uint4*>(out_lo + o) = make_uint4(ol[0], ol[1], ol[2], ol[3]);
  }
}

// ---------------------------------------------------------- layout converters
__global__ void split_to_nchw_kernel(const __nv_bfloat16* __restrict__ in_hi,
                                     const __nv_bfloat16* __restrict__ in_lo, int batch, int H,
                                     int W, int C, float* __restrict__ out) {
  // tile transpose through shared memory: 32 pixels x 32 channels
  __shared__ float t[32][33];
  const long long HW = static_cast<long long>(H) * W;
  const int img = blockIdx.z;
  const long long p0 = static_cast<long long>(blockIdx.x) * 32;
  const int c0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const long long p = p0 + i;
    const int c = c0 + threadIdx.x;
    float v = 0.f;
    if (p < HW && c < C) {
      const long long off = (static_cast<long long>(img) * HW + p) * C + c;
      v = bf2f(in_hi[off]) + bf2f(in_lo[off]);
    }
    t[i][threadIdx.x] = v;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i;
    const long long p = p0 + threadIdx.x;
    if (p < HW && c < C) out[(static_cast<long long>(img) * C + c) * HW + p] = t[threadIdx.x][i];
  }
}

__global__ void nchw_to_split_kernel(const float* __restrict__ in, int batch, int C, int H, int W,
                                     __nv_bfloat16* __restrict__ out_hi,
                                     __nv_bfloat16* __restrict__ out_lo) {
  __shared__ float t[32][33];
  const long long HW = static_cast<long long>(H) * W;
  const int img = blockIdx.z;
  const long long p0 = static_cast<long long>(blockIdx.x) * 32;
  const int c0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i;
    const long long p = p0 + threadIdx.x;
    float v = 0.f;
    if (p < HW && c < C) v = in[(static_cast<long long>(img) * C + c) * HW + p];
    t[i][threadIdx.x] = v;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const long long p = p0 + i;
    const int c = c0 + threadIdx.x;
    if (p < HW && c < C) {
      __nv_bfloat16 hi, lo;
      split_f32(t[threadIdx.x][i], hi, lo);
      const long long off = (static_cast<long long>(img) * HW + p) * C + c;
      out_hi[off] = hi;
      out_lo[off] = lo;
    }
  }
}

__global__ void f32_to_split_kernel(const float* __restrict__ in, long long n,
                                    __nv_bfloat16* __restrict__ out_hi,
                                    __nv_bfloat16* __restrict__ out_lo) {
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    __nv_bfloat16 hi, lo;
    split_f32(in[i], hi, lo);
    out_hi[i] = hi;
    out_lo[i] = lo;
  }
}
__global__ void split_to_f32_kernel(const __nv_bfloat16* __restrict__ in_hi,
                                    const __nv_bfloat16* __restrict__ in_lo, long long n,
                                    float* __restrict__ out) {
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x)
    out[i] = bf2f(in_hi[i]) + bf2f(in_lo[i]);
}

static inline int grid_for(long long n, int block, int cap = 148 * 16) {
  long long g = (n + block - 1) / block;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return static_cast<int>(g);
}
static inline int check_launch() { return cudaGetLastError() == cudaSuccess ? MNC_OK : MNC_ERR_CUDA; }

}  // namespace mnc

using namespace mnc;

extern "C" int mnc_igemm_simt(const void* a_hi, const void* a_lo, int batch, int H, int W, int Cin,
                              const void* w_hi, const void* w_lo, int Cout, int taps,
                              const float* bias, int relu, int out_mode, void* out0, void* out1,
                              long long out_pix_stride, int out_ch_offset, void* stream) {
  if (Cin % 16 != 0 || (taps != 1 && taps != 9)) return MNC_ERR_ARG;
  const long long M = static_cast<long long>(batch) * H * W;
  dim3 grid(static_cast<unsigned>((M + 63) / 64), static_cast<unsigned>((Cout + 63) / 64));
  igemm_simt_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const __nv_bfloat16*>(a_hi), static_cast<const __nv_bfloat16*>(a_lo), batch, H,
      W, Cin, static_cast<const __nv_bfloat16*>(w_hi), static_cast<const __nv_bfloat16*>(w_lo),
      Cout, taps, bias, relu, out_mode, out0, out1, out_pix_stride, out_ch_offset);
  return check_launch();
}

extern "C" int mnc_splitk_reduce2(const float* partial, int splits, long long split_stride,
                                  long long rows, int cols, const float* bias, int relu,
                                  int out_mode, void* out0, void* out1, long long out_row_stride,
                                  int out_ch_offset, const int* img_hw, int level, int H, int W,
                                  void* stream) {
  if (rows <= 0 || cols <= 0) return MNC_OK;
  if (img_hw != nullptr && (level < 0 || level > 16 || H <= 0 || W <= 0 ||
                            rows % (static_cast<long long>(H) * W) != 0))
    return MNC_ERR_ARG;
  const int vec = (cols % 4 == 0) && (split_stride % 4 == 0) && (out_row_stride % 4 == 0) &&
                  (out_ch_offset % 4 == 0) && (reinterpret_cast<uintptr_t>(partial) % 16 == 0) &&
                  (reinterpret_cast<uintptr_t>(out0) % 16 == 0) &&
                  (out_mode == 1 || reinterpret_cast<uintptr_t>(out1) % 8 == 0);
  const int tx = (cols + 3) / 4;
  const int block = tx >= 256 ? 256 : (tx >= 128 ? 128 : (tx >= 64 ? 64 : 32));
  dim3 grid((tx + block - 1) / block, static_cast<unsigned>(rows < 32768 ? rows : 32768));
  splitk_reduce_kernel<<<grid, block, 0, static_cast<cudaStream_t>(stream)>>>(
      partial, splits, split_stride, rows, cols, bias, relu, out_mode, out0, out1, out_row_stride,
      out_ch_offset, vec, img_hw, level, H, W);
  return check_launch();
}

extern "C" int mnc_splitk_reduce(const float* partial, int splits, long long split_stride,
                                 long long rows, int cols, const float* bias, int relu,
                                 int out_mode, void* out0, void* out1, long long out_row_stride,
                                 int out_ch_offset, void* stream) {
  return mnc_splitk_reduce2(partial, splits, split_stride, rows, cols, bias, relu, out_mode, out0,
                            out1, out_row_stride, out_ch_offset, nullptr, 0, 1, 1, stream);
}

extern "C" int mnc_conv1_1(const float* data_nchw, int batch, int H, int W, const float* weight,
                           const float* bias, int Cout, void* out_hi, void* out_lo, void* stream) {
  if (Cout != 64) return MNC_ERR_ARG;
  const int tiles = batch * ((H + kC11TH - 1) / kC11TH) * ((W + kC11TW - 1) / kC11TW);
  conv1_1_kernel<<<tiles, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      data_nchw, batch, H, W, weight, bias, static_cast<__nv_bfloat16*>(out_hi),
      static_cast<__nv_bfloat16*>(out_lo));
  return check_launch();
}

extern "C" int mnc_maxpool2x2_split(const void* in_hi, const void* in_lo, int batch, int H, int W,
                                    int C, void* out_hi, void* out_lo, void* stream) {
  if (C % 8 != 0) return MNC_ERR_ARG;
  const long long total = static_cast<long long>(batch) * ((H + 1) / 2) * ((W + 1) / 2) * (C / 8);
  maxpool2x2_split_kernel<<<grid_for(total, 256, 148 * 32), 256, 0,
                            static_cast<cudaStream_t>(stream)>>>(
      static_cast<const __nv_bfloat16*>(in_hi), static_cast<const __nv_bfloat16*>(in_lo), batch, H,
      W, C, static_cast<__nv_bfloat16*>(out_hi), static_cast<__nv_bfloat16*>(out_lo));
  return check_launch();
}

extern "C" int mnc_split_to_nchw(const void* in_hi, const void* in_lo, int batch, int H, int W,
                                 int C, float* out_nchw, void* stream) {
  const long long HW = static_cast<long long>(H) * W;
  dim3 grid(static_cast<unsigned>((HW + 31) / 32), static_cast<unsigned>((C + 31) / 32), batch);
  split_to_nchw_kernel<<<grid, dim3(32, 8), 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const __nv_bfloat16*>(in_hi), static_cast<const __nv_bfloat16*>(in_lo), batch, H,
      W, C, out_nchw);
  return check_launch();
}

extern "C" int mnc_nchw_to_split(const float* in_nchw, int batch, int C, int H, int W,
                                 void* out_hi, void* out_lo, void* stream) {
  const long long HW = static_cast<long long>(H) * W;
  dim3 grid(static_cast<unsigned>((HW + 31) / 32), static_cast<unsigned>((C + 31) / 32), batch);
  nchw_to_split_kernel<<<grid, dim3(32, 8), 0, static_cast<cudaStream_t>(stream)>>>(
      in_nchw, batch, C, H, W, static_cast<__nv_bfloat16*>(out_hi),
      static_cast<__nv_bfloat16*>(out_lo));
  return check_launch();
}

extern "C" int mnc_f32_to_split(const float* in, long long n, void* out_hi, void* out_lo,
                                void* stream) {
  f32_to_split_kernel<<<grid_for(n, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      in, n, static_cast<__nv_bfloat16*>(out_hi), static_cast<__nv_bfloat16*>(out_lo));
  return check_launch();
}
extern "C" int mnc_split_to_f32(const void* in_hi, const void* in_lo, long long n, float* out,
                                void* stream) {
  split_to_f32_kernel<<<grid_for(n, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const __nv_bfloat16*>(in_hi), static_cast<const __nv_bfloat16*>(in_lo), n, out);
  return check_launch();
}
