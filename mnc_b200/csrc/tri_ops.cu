// Element-wise producers / consumers of tri-plane activations (precision mode 1, igemm_tc.cu):
// fp32 <-> tri-plane conversion, the split-K reduction epilogue, and MaskPooling + 2x2 max pool
// (mask_pooling_layer.cu:13-26 + Pooling) on tri-plane NHWC RoI features.
#include <cuda_runtime.h>
#include <cstdint>

#include "mnc_b200.h"
#include "tri.cuh"

namespace mnc {

static inline int tri_check_launch() { return cudaGetLastError() == cudaSuccess ? MNC_OK : MNC_ERR_CUDA; }

__device__ __forceinline__ void amax_publish(float amx, unsigned int* amax) {
  if (amax == nullptr) return;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) amx = fmaxf(amx, __shfl_xor_sync(0xffffffffu, amx, o));
  if ((threadIdx.x & 31) == 0 && amx > 0.f) atomicMax(amax, __float_as_uint(amx));
}

__global__ void __launch_bounds__(256)
f32_to_tri_kernel(const float* __restrict__ in, long long n4, float scale, __half* __restrict__ h,
                  uint8_t* __restrict__ l, uint8_t* __restrict__ c, unsigned int* amax) {
  float amx = 0.f;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(in) + i);
    amx = fmaxf(amx, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
    st_tri4(h, l, c, i * 4, v, scale);
  }
  amax_publish(amx, amax);
}

__global__ void __launch_bounds__(256)
tri_to_f32_kernel(const __half* __restrict__ h, const uint8_t* __restrict__ l, long long n4,
                  float inv_scale, float* __restrict__ out) {
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float4 v = ld_tri4(h, l, i * 4);
    reinterpret_cast<float4*>(out)[i] = make_float4(v.x * inv_scale, v.y * inv_scale, v.z * inv_scale, v.w * inv_scale);
  }
}

// Is conv output row `row` (= pixel (b, y, x) of a [B][H][W] map) inside its image's extent at
// trunk level `level`?  img_hw: device int32 [B][2] input-resolution sizes (mixed-size batches).
__device__ __forceinline__ bool row_in_image(const int* img_hw, int level, int H, int W, long long row) {
  if (img_hw == nullptr) return true;
  const long long hw = static_cast<long long>(H) * W;
  const int b = static_cast<int>(row / hw);
  const int r = static_cast<int>(row - b * hw);
  const int m = (1 << level) - 1;
  return r / W < ((__ldg(img_hw + 2 * b) + m) >> level) && r % W < ((__ldg(img_hw + 2 * b + 1) + m) >> level);
}

// out[row][ch_offset + col] = act(sum_s partial[s][row][col] + bias[col]) as tri-plane; one thread
// per 4 columns.  Rows outside their image (img_hw, conv launches of mixed-size batches) are zeros.
__global__ void __launch_bounds__(256)
splitk_reduce_tri_kernel(const float* __restrict__ partial, int splits, long long split_stride,
                         long long rows, int cols, const float* __restrict__ bias, int relu,
                         float scale, __half* __restrict__ h, uint8_t* __restrict__ l,
                         uint8_t* __restrict__ c, long long out_row_stride, int out_ch_offset,
                         unsigned int* amax, const int* __restrict__ img_hw, int level, int H, int W) {
  const int c4 = cols >> 2;
  float amx = 0.f;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < rows * c4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long row = i / c4;
    const int col = static_cast<int>(i - row * c4) * 4;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 8   // loads of 8 splits in flight; the sum keeps its split order
    for (int s = 0; s < splits; ++s) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(partial + s * split_stride + row * cols + col));
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    if (bias != nullptr) {
      const float4 b = __ldg(reinterpret_cast<const float4*>(bias + col));
      acc.x += b.x; acc.y += b.y; acc.z += b.z; acc.w += b.w;
    }
    if (relu) {
      acc.x = fmaxf(acc.x, 0.f); acc.y = fmaxf(acc.y, 0.f); acc.z = fmaxf(acc.z, 0.f); acc.w = fmaxf(acc.w, 0.f);
    }
    if (!row_in_image(img_hw, level, H, W, row)) acc = make_float4(0.f, 0.f, 0.f, 0.f);
    amx = fmaxf(amx, fmaxf(fmaxf(fabsf(acc.x), fabsf(acc.y)), fmaxf(fabsf(acc.z), fabsf(acc.w))));
    st_tri4(h, l, c, row * out_row_stride + out_ch_offset + col, acc, scale);
  }
  amax_publish(amx, amax);
}

// MaskPooling + 2x2 max pool: out7[r][t][j][c] = max_{dy,dx} feat14[r][2t+dy][2j+dx][c] * mask14.
// Input and output share one exponent (|mask| <= 1 cannot grow the range): the product is formed
// on the scaled values and re-packed with scale 1.
__global__ void __launch_bounds__(256)
mask_pool_tri_kernel(const __half* __restrict__ f_h, const uint8_t* __restrict__ f_l,
                     const float* __restrict__ mask14, int C, __half* __restrict__ o_h,
                     uint8_t* __restrict__ o_l, uint8_t* __restrict__ o_c) {
  const int r = blockIdx.x, t = blockIdx.y;
  __shared__ float m[2][14];
  if (threadIdx.x < 28)
    m[threadIdx.x / 14][threadIdx.x % 14] =
        mask14[static_cast<long long>(r) * 196 + (2 * t + threadIdx.x / 14) * 14 + threadIdx.x % 14];
  __syncthreads();
  for (int c = threadIdx.x * 4; c < C; c += blockDim.x * 4) {
    for (int jp = 0; jp < 7; ++jp) {
      float4 best = make_float4(-3.402823466e+38f, -3.402823466e+38f, -3.402823466e+38f, -3.402823466e+38f);
#pragma unroll
      for (int dy = 0; dy < 2; ++dy)
#pragma unroll
        for (int dx = 0; dx < 2; ++dx) {
          const int i = 2 * t + dy, j = 2 * jp + dx;
          const float4 f = ld_tri4(f_h, f_l, ((static_cast<long long>(r) * 14 + i) * 14 + j) * C + c);
          const float mk = m[dy][j];
          best.x = fmaxf(best.x, __fmul_rn(f.x, mk));
          best.y = fmaxf(best.y, __fmul_rn(f.y, mk));
          best.z = fmaxf(best.z, __fmul_rn(f.z, mk));
          best.w = fmaxf(best.w, __fmul_rn(f.w, mk));
        }
      st_tri4(o_h, o_l, o_c, ((static_cast<long long>(r) * 7 + t) * 7 + jp) * C + c, best, 1.0f);
    }
  }
}

static inline int tri_grid(long long n, int block) {
  long long g = (n + block - 1) / block;
  if (g > 148 * 16) g = 148 * 16;
  if (g < 1) g = 1;
  return static_cast<int>(g);
}

}  // namespace mnc

using namespace mnc;

extern "C" int mnc_f32_to_tri(const float* in, long long n, float scale, void* h, void* l, void* c,
                              unsigned int* amax, void* stream) {
  if (n <= 0) return MNC_OK;
  if (n % 4 != 0 || (reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(h) |
                      reinterpret_cast<uintptr_t>(l) | reinterpret_cast<uintptr_t>(c)) % 8 != 0)
    return MNC_ERR_ARG;
  f32_to_tri_kernel<<<tri_grid(n / 4, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      in, n / 4, scale, static_cast<__half*>(h), static_cast<uint8_t*>(l), static_cast<uint8_t*>(c), amax);
  return tri_check_launch();
}

extern "C" int mnc_tri_to_f32(const void* h, const void* l, long long n, float inv_scale, float* out,
                              void* stream) {
  if (n <= 0) return MNC_OK;
  if (n % 4 != 0 || (reinterpret_cast<uintptr_t>(out) % 16) != 0) return MNC_ERR_ARG;
  tri_to_f32_kernel<<<tri_grid(n / 4, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const __half*>(h), static_cast<const uint8_t*>(l), n / 4, inv_scale, out);
  return tri_check_launch();
}

extern "C" int mnc_splitk_reduce_tri2(const float* partial, int splits, long long split_stride,
                                      long long rows, int cols, const float* bias, int relu,
                                      float scale, void* h, void* l, void* c,
                                      long long out_row_stride, int out_ch_offset,
                                      unsigned int* amax, const int* img_hw, int level, int H,
                                      int W, void* stream) {
  if (rows <= 0 || cols <= 0) return MNC_OK;
  if (img_hw != nullptr && (level < 0 || level > 16 || H <= 0 || W <= 0 ||
                            rows % (static_cast<long long>(H) * W) != 0))
    return MNC_ERR_ARG;
  if (cols % 4 != 0 || split_stride % 4 != 0 || out_row_stride % 4 != 0 || out_ch_offset % 4 != 0 ||
      reinterpret_cast<uintptr_t>(partial) % 16 != 0 ||
      (bias != nullptr && reinterpret_cast<uintptr_t>(bias) % 16 != 0))
    return MNC_ERR_ARG;
  splitk_reduce_tri_kernel<<<tri_grid(rows * (cols / 4), 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      partial, splits, split_stride, rows, cols, bias, relu, scale, static_cast<__half*>(h),
      static_cast<uint8_t*>(l), static_cast<uint8_t*>(c), out_row_stride, out_ch_offset, amax,
      img_hw, level, H, W);
  return tri_check_launch();
}

extern "C" int mnc_splitk_reduce_tri(const float* partial, int splits, long long split_stride,
                                     long long rows, int cols, const float* bias, int relu,
                                     float scale, void* h, void* l, void* c,
                                     long long out_row_stride, int out_ch_offset,
                                     unsigned int* amax, void* stream) {
  return mnc_splitk_reduce_tri2(partial, splits, split_stride, rows, cols, bias, relu, scale, h, l, c,
                                out_row_stride, out_ch_offset, amax, nullptr, 0, 1, 1, stream);
}

extern "C" int mnc_mask_pool_tri(const void* f_h, const void* f_l, const float* mask14, int R, int C,
                                 void* o_h, void* o_l, void* o_c, void* stream) {
  if (R <= 0) return MNC_OK;
  if (C % 4 != 0) return MNC_ERR_ARG;
  dim3 grid(R, 7);
  mask_pool_tri_kernel<<<grid, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const __half*>(f_h), static_cast<const uint8_t*>(f_l), mask14, C,
      static_cast<__half*>(o_h), static_cast<uint8_t*>(o_l), static_cast<uint8_t*>(o_c));
  return tri_check_launch();
}
