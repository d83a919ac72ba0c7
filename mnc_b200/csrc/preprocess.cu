// Input preparation on the device: prep_im_for_blob + im_list_to_blob
// (reference lib/utils/blob.py:17-50): uint8 BGR HWC image -> float32, minus cfg.PIXEL_MEANS,
// cv2.resize(fx = fy = scale, INTER_LINEAR), HWC -> NCHW blob.
//
// OpenCV's float INTER_LINEAR rule is restated (OpenCV is a dependency of the reference, not part
// of it): source coordinate fx = (dx + 0.5) / scale - 0.5 in double, sx = floor(fx); sx < 0 -> (0, frac 0);
// sx >= W-1 -> (W-1, frac 0); horizontal interpolation first, then vertical, in fp32.
#include <cuda_runtime.h>
#include <cstdint>

#include "mnc_b200.h"

namespace mnc {

struct LinTap {
  int i0, i1;
  float a0, a1;
};

__device__ __forceinline__ LinTap lin_tap(int d, double inv_scale, int n) {
  // the fraction is taken in double and rounded once (OpenCV 4.x resize.cpp; an fp32 coordinate
  // would lose 1e-5 of the fraction at x ~ 200 and 3e-3 of a pixel value -- measured against cv2)
  const double fd = (d + 0.5) * inv_scale - 0.5;
  int s = static_cast<int>(floor(fd));
  float f = static_cast<float>(fd - s);
  if (s < 0) {
    f = 0.f;
    s = 0;
  }
  LinTap t;
  if (s >= n - 1) {
    t.i0 = t.i1 = n - 1;
    f = 0.f;
  } else {
    t.i0 = s;
    t.i1 = s + 1;
  }
  t.a0 = 1.f - f;
  t.a1 = f;
  return t;
}

// Output pixel (x, y) of one image: 3 channels at ob, ob + plane, ob + 2 * plane.
__device__ __forceinline__ void prep_pixel(const uint8_t* __restrict__ base, int H, int W, double m0,
                                           double m1, double m2, double inv_scale, int x, int y,
                                           float* __restrict__ ob, long long plane) {
  const LinTap tx = lin_tap(x, inv_scale, W);
  const LinTap ty = lin_tap(y, inv_scale, H);
  const double means[3] = {m0, m1, m2};
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    // `im = im.astype(np.float32); im -= pixel_means`: float32(double(pixel) - mean)
    const float p00 = static_cast<float>(static_cast<double>(base[(static_cast<long long>(ty.i0) * W + tx.i0) * 3 + c]) - means[c]);
    const float p01 = static_cast<float>(static_cast<double>(base[(static_cast<long long>(ty.i0) * W + tx.i1) * 3 + c]) - means[c]);
    const float p10 = static_cast<float>(static_cast<double>(base[(static_cast<long long>(ty.i1) * W + tx.i0) * 3 + c]) - means[c]);
    const float p11 = static_cast<float>(static_cast<double>(base[(static_cast<long long>(ty.i1) * W + tx.i1) * 3 + c]) - means[c]);
    const float r0 = __fadd_rn(__fmul_rn(p00, tx.a0), __fmul_rn(p01, tx.a1));
    const float r1 = __fadd_rn(__fmul_rn(p10, tx.a0), __fmul_rn(p11, tx.a1));
    ob[static_cast<long long>(c) * plane] = __fadd_rn(__fmul_rn(r0, ty.a0), __fmul_rn(r1, ty.a1));
  }
}

// grid (ceil(out_w/128), out_h, batch); one thread per output pixel, 3 channels.
__global__ void __launch_bounds__(128)
prep_image_kernel(const uint8_t* __restrict__ img, int H, int W, double m0, double m1, double m2,
                  double inv_scale, int out_h, int out_w, float* __restrict__ out) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y;
  const int b = blockIdx.z;
  if (x >= out_w) return;
  const uint8_t* base = img + static_cast<long long>(b) * H * W * 3;
  float* ob = out + static_cast<long long>(b) * 3 * out_h * out_w + static_cast<long long>(y) * out_w + x;
  prep_pixel(base, H, W, m0, m1, m2, inv_scale, x, y, ob, static_cast<long long>(out_h) * out_w);
}

// Images of different sizes in one launch (im_list_to_blob, blob.py:17-31): image b (packed at
// byte offset off[b], h[b] x w[b] x 3) scaled into the top-left oh[b] x ow[b] of a zero-padded
// [batch][3][out_h][out_w] blob.  The per-image table travels as a kernel parameter.
constexpr int kRaggedMax = 64;
struct RaggedImages {
  long long off[kRaggedMax];
  double inv_scale[kRaggedMax];
  int h[kRaggedMax], w[kRaggedMax], oh[kRaggedMax], ow[kRaggedMax];
};

__global__ void __launch_bounds__(128)
prep_ragged_kernel(const uint8_t* __restrict__ packed, const __grid_constant__ RaggedImages t,
                   double m0, double m1, double m2, int out_h, int out_w, float* __restrict__ out) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y;
  const int b = blockIdx.z;
  if (x >= out_w) return;
  const long long plane = static_cast<long long>(out_h) * out_w;
  float* ob = out + static_cast<long long>(b) * 3 * plane + static_cast<long long>(y) * out_w + x;
  if (y < t.oh[b] && x < t.ow[b]) {
    prep_pixel(packed + t.off[b], t.h[b], t.w[b], m0, m1, m2, t.inv_scale[b], x, y, ob, plane);
  } else {
    ob[0] = 0.f;
    ob[plane] = 0.f;
    ob[2 * plane] = 0.f;
  }
}

}  // namespace mnc

extern "C" int mnc_prep_images(const unsigned char* img_bgr_hwc, int batch, int H, int W,
                               const double* pixel_means3, double scale, int out_h, int out_w,
                               float* out_nchw, void* stream) {
  if (batch <= 0 || H <= 0 || W <= 0 || out_h <= 0 || out_w <= 0 || scale <= 0) return MNC_ERR_ARG;
  dim3 grid((out_w + 127) / 128, out_h, batch);
  mnc::prep_image_kernel<<<grid, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      img_bgr_hwc, H, W, pixel_means3[0], pixel_means3[1], pixel_means3[2], 1.0 / scale, out_h,
      out_w, out_nchw);
  return cudaGetLastError() == cudaSuccess ? MNC_OK : MNC_ERR_CUDA;
}

// Host arrays: offsets[b] (bytes into `packed`), src_hw[b] = (h, w) of the uint8 BGR HWC image,
// scales[b], dst_hw[b] = (round(h * scale), round(w * scale)) <= (out_h, out_w).
extern "C" int mnc_prep_images_ragged(const unsigned char* packed, int batch, const long long* offsets,
                                      const int* src_hw, const double* scales, const int* dst_hw,
                                      const double* pixel_means3, int out_h, int out_w,
                                      float* out_nchw, void* stream) {
  if (batch <= 0 || batch > mnc::kRaggedMax || out_h <= 0 || out_w <= 0) return MNC_ERR_ARG;
  mnc::RaggedImages t;
  for (int b = 0; b < batch; ++b) {
    if (src_hw[2 * b] <= 0 || src_hw[2 * b + 1] <= 0 || !(scales[b] > 0) || offsets[b] < 0 ||
        dst_hw[2 * b] <= 0 || dst_hw[2 * b + 1] <= 0 || dst_hw[2 * b] > out_h ||
        dst_hw[2 * b + 1] > out_w)
      return MNC_ERR_ARG;
    t.off[b] = offsets[b];
    t.inv_scale[b] = 1.0 / scales[b];
    t.h[b] = src_hw[2 * b];
    t.w[b] = src_hw[2 * b + 1];
    t.oh[b] = dst_hw[2 * b];
    t.ow[b] = dst_hw[2 * b + 1];
  }
  dim3 grid((out_w + 127) / 128, out_h, batch);
  mnc::prep_ragged_kernel<<<grid, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      packed, t, pixel_means3[0], pixel_means3[1], pixel_means3[2], out_h, out_w, out_nchw);
  return cudaGetLastError() == cudaSuccess ? MNC_OK : MNC_ERR_CUDA;
}
