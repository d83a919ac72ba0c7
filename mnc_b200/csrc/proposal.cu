// Device versions of the reference's host-side Python layers on the inference path:
//   ProposalLayer.forward      lib/pylayer/proposal_layer.py:52-175  (decode / clip / min-size)
//   StageBridgeLayer.forward_test   lib/pylayer/stage_bridge_layer.py:237-255
//   Softmax (Caffe)            caffe-mnc/src/caffe/layers/softmax_layer.cu:86-120
//   im_detect tail             tools/demo.py:92-95
// The numpy code evaluates every operation separately in fp32; to reproduce it bit for bit the
// arithmetic below uses __fmul_rn/__fadd_rn/__fsub_rn (never contracted into FMA).  expf differs
// from numpy's exp by an ulp or two, which is why parity tests split "decode" (tolerance) from
// "filter / sort / NMS" (bit-exact on identical inputs).
#include <cuda_runtime.h>
#include <cmath>
#include <cstdint>

#include "mnc_b200.h"

namespace mnc {

struct Anchors {
  float v[9][4];
};

// lib/transform/anchors.py:38-102, evaluated in double like numpy, rounded half-to-even.
static void generate_anchors_host(double out[9][4]) {
  const double base_size = 16;
  const double ratios[3] = {0.5, 1, 2};
  const double scales[3] = {8, 16, 32};
  // base anchor (0,0,15,15): w = h = 16, ctr = 7.5
  const double w = base_size, h = base_size;
  const double x_ctr = 0 + 0.5 * (w - 1), y_ctr = 0 + 0.5 * (h - 1);
  const double size = w * h;
  int k = 0;
  for (int r = 0; r < 3; ++r) {
    const double size_ratio = size / ratios[r];
    const double ws = std::nearbyint(std::sqrt(size_ratio));
    const double hs = std::nearbyint(ws * ratios[r]);
    // ratio anchor
    const double rx1 = x_ctr - 0.5 * (ws - 1), ry1 = y_ctr - 0.5 * (hs - 1);
    const double rx2 = x_ctr + 0.5 * (ws - 1), ry2 = y_ctr + 0.5 * (hs - 1);
    const double rw = rx2 - rx1 + 1, rh = ry2 - ry1 + 1;
    const double rcx = rx1 + 0.5 * (rw - 1), rcy = ry1 + 0.5 * (rh - 1);
    for (int s = 0; s < 3; ++s) {
      const double sw = rw * scales[s], sh = rh * scales[s];
      out[k][0] = rcx - 0.5 * (sw - 1);
      out[k][1] = rcy - 0.5 * (sh - 1);
      out[k][2] = rcx + 0.5 * (sw - 1);
      out[k][3] = rcy + 0.5 * (sh - 1);
      ++k;
    }
  }
}

__device__ __forceinline__ float clipf(float v, float hi) { return fmaxf(fminf(v, hi), 0.f); }

// bbox_transform_inv for one box / one delta quadruple (bbox_transform.py:72-97), then
// clip_boxes (:112-118).  All fp32, one rounding per numpy operation.
__device__ __forceinline__ void decode_clip(float x1, float y1, float x2, float y2, float dx,
                                            float dy, float dw, float dh, float im_h, float im_w,
                                            float out[4]) {
  const float widths = __fadd_rn(__fsub_rn(x2, x1), 1.0f);
  const float heights = __fadd_rn(__fsub_rn(y2, y1), 1.0f);
  const float ctr_x = __fadd_rn(x1, __fmul_rn(0.5f, widths));
  const float ctr_y = __fadd_rn(y1, __fmul_rn(0.5f, heights));
  const float pred_ctr_x = __fadd_rn(__fmul_rn(dx, widths), ctr_x);
  const float pred_ctr_y = __fadd_rn(__fmul_rn(dy, heights), ctr_y);
  const float pred_w = __fmul_rn(expf(dw), widths);
  const float pred_h = __fmul_rn(expf(dh), heights);
  const float wmax = __fsub_rn(im_w, 1.0f), hmax = __fsub_rn(im_h, 1.0f);
  out[0] = clipf(__fsub_rn(pred_ctr_x, __fmul_rn(0.5f, pred_w)), wmax);
  out[1] = clipf(__fsub_rn(pred_ctr_y, __fmul_rn(0.5f, pred_h)), hmax);
  out[2] = clipf(__fadd_rn(pred_ctr_x, __fmul_rn(0.5f, pred_w)), wmax);
  out[3] = clipf(__fadd_rn(pred_ctr_y, __fmul_rn(0.5f, pred_h)), hmax);
}

// One thread per anchor t = (y*W + x)*A + a  (proposal_layer.py:96-100,111,118).
__global__ void rpn_decode_kernel(const float* __restrict__ cls, long long cls_img_stride,
                                  long long cls_ch_stride, long long cls_pix_stride,
                                  const float* __restrict__ bbox, long long bb_img_stride,
                                  long long bb_ch_stride, long long bb_pix_stride,
                                  const float* __restrict__ im_info, int H, int W, int feat_stride,
                                  float min_size, int apply_softmax, const Anchors anchors,
                                  float* __restrict__ proposals, float* __restrict__ scores,
                                  unsigned char* __restrict__ valid, const int* __restrict__ img_hw,
                                  int level) {
  const int A = 9;
  const int total = H * W * A;
  const int img = blockIdx.y;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  const int a = t % A;
  const int pix = t / A;
  const int y = pix / W, x = pix % W;
  const float* pc = cls + img * cls_img_stride + pix * cls_pix_stride;
  const float* pb = bbox + img * bb_img_stride + pix * bb_pix_stride;
  float score;
  if (apply_softmax) {
    // Caffe softmax over {bg, fg}: subtract max, exp, sum, divide (softmax_layer.cu:93-119)
    const float bg = pc[a * cls_ch_stride], fg = pc[(A + a) * cls_ch_stride];
    const float m = fmaxf(bg, fg);
    const float eb = expf(__fsub_rn(bg, m)), ef = expf(__fsub_rn(fg, m));
    score = __fdiv_rn(ef, __fadd_rn(eb, ef));
  } else {
    score = pc[(A + a) * cls_ch_stride];
  }
  const float dx = pb[(4 * a + 0) * bb_ch_stride], dy = pb[(4 * a + 1) * bb_ch_stride];
  const float dw = pb[(4 * a + 2) * bb_ch_stride], dh = pb[(4 * a + 3) * bb_ch_stride];
  // anchors are float64 integers in numpy, cast to fp32 at bbox_transform.py:72 (exact)
  const float sx = static_cast<float>(x * feat_stride), sy = static_cast<float>(y * feat_stride);
  const float ax1 = anchors.v[a][0] + sx, ay1 = anchors.v[a][1] + sy;
  const float ax2 = anchors.v[a][2] + sx, ay2 = anchors.v[a][3] + sy;
  const float im_h = im_info[img * 3 + 0], im_w = im_info[img * 3 + 1], im_s = im_info[img * 3 + 2];
  float o[4];
  decode_clip(ax1, ay1, ax2, ay2, dx, dy, dw, dh, im_h, im_w, o);
  // filter_small_boxes (bbox_transform.py:123-130) with min_size * im_info[2]
  const float ms = __fmul_rn(min_size, im_s);
  const float ws = __fadd_rn(__fsub_rn(o[2], o[0]), 1.0f);
  const float hs = __fadd_rn(__fsub_rn(o[3], o[1]), 1.0f);
  const long long oidx = static_cast<long long>(img) * total + t;
  *reinterpret_cast<float4*>(proposals + oidx * 4) = make_float4(o[0], o[1], o[2], o[3]);
  scores[oidx] = score;
  // mixed-size batch: anchors of the padded map outside this image's extent take no part
  bool inside = true;
  if (img_hw != nullptr) {
    const int m = (1 << level) - 1;
    inside = y < ((__ldg(img_hw + 2 * img) + m) >> level) && x < ((__ldg(img_hw + 2 * img + 1) + m) >> level);
  }
  valid[oidx] = (inside && ws >= ms && hs >= ms) ? 1 : 0;
}

// rois[img][k] = [batch_index, sorted_boxes[img][keep[img][k]]], zero rows past num_keep.
__global__ void write_rois_kernel(const float* __restrict__ sorted_boxes, int n_sorted,
                                  const int* __restrict__ keep, int keep_stride,
                                  const int* __restrict__ num_keep, int max_rois,
                                  int batch_index_mode, float* __restrict__ rois,
                                  int* __restrict__ roi_counts) {
  const int img = blockIdx.y;
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= max_rois) return;
  const int nk = min(num_keep[img], max_rois);
  if (k == 0 && roi_counts) roi_counts[img] = nk;
  float* r = rois + (static_cast<long long>(img) * max_rois + k) * 5;
  if (k < nk) {
    const int idx = keep[static_cast<long long>(img) * keep_stride + k];
    const float* b = sorted_boxes + (static_cast<long long>(img) * n_sorted + idx) * 4;
    r[0] = batch_index_mode ? static_cast<float>(img) : 0.f;
    r[1] = b[0];
    r[2] = b[1];
    r[3] = b[2];
    r[4] = b[3];
  } else {
    r[0] = batch_index_mode ? static_cast<float>(img) : 0.f;
    r[1] = r[2] = r[3] = r[4] = 0.f;
  }
}

// One thread per RoI: c* = first argmax over all `ncls` seg_cls_prob columns (bg allowed),
// decode the 4 deltas of class c*, clip to im_info (stage_bridge_layer.py:241-252).
__global__ void stage_bridge_kernel(const float* __restrict__ rois,
                                    const float* __restrict__ bbox_pred, int bbox_stride,
                                    const float* __restrict__ seg_cls_prob, int prob_stride,
                                    int ncls, const float* __restrict__ im_info, int rois_per_img,
                                    int total, float* __restrict__ rois_out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int img = i / rois_per_img;
  const float* r = rois + static_cast<long long>(i) * 5;
  const float* p = seg_cls_prob + static_cast<long long>(i) * prob_stride;
  int best = 0;
  float bv = p[0];
  for (int c = 1; c < ncls; ++c) {
    const float v = p[c];
    if (v > bv) {
      bv = v;
      best = c;
    }
  }
  const float* d = bbox_pred + static_cast<long long>(i) * bbox_stride + 4 * best;
  float o[4];
  decode_clip(r[1], r[2], r[3], r[4], d[0], d[1], d[2], d[3], im_info[img * 3 + 0],
              im_info[img * 3 + 1], o);
  float* ro = rois_out + static_cast<long long>(i) * 5;
  ro[0] = r[0];
  ro[1] = o[0];
  ro[2] = o[1];
  ro[3] = o[2];
  ro[4] = o[3];
}

// Row softmax (softmax_layer.cu:86-120 order of operations), one WARP per row, cols <= 64: lanes
// hold the columns (two each), the row maximum is a shuffle reduction (max is order-independent),
// the exponentials are evaluated in parallel, and the denominator is accumulated in COLUMN ORDER
// -- the order of the reference's channel-sum loop -- by every lane from shuffled values, so the
// result equals the one-thread-per-row evaluation bit for bit while the 4 launches per step drop
// from ~16 us (a serial chain of dependent global accesses) to launch latency.
__global__ void __launch_bounds__(128)
softmax_rows_kernel(const float* __restrict__ in, int in_stride, int rows, int cols,
                    float* __restrict__ out, int out_stride) {
  const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (r >= rows) return;                       // warp-uniform
  const float* x = in + static_cast<long long>(r) * in_stride;
  float* y = out + static_cast<long long>(r) * out_stride;
  const bool ok0 = lane < cols, ok1 = lane + 32 < cols;
  const float x0 = ok0 ? x[lane] : 0.f, x1 = ok1 ? x[lane + 32] : 0.f;
  const float kNegInf = __int_as_float(0xff800000);
  float m = fmaxf(ok0 ? x0 : kNegInf, ok1 ? x1 : kNegInf);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  const float e0 = ok0 ? expf(__fsub_rn(x0, m)) : 0.f;
  const float e1 = ok1 ? expf(__fsub_rn(x1, m)) : 0.f;
  float s = 0.f;
  for (int c = 0; c < cols; ++c) {
    const float v = __shfl_sync(0xffffffffu, c < 32 ? e0 : e1, c & 31);
    s = __fadd_rn(s, v);
  }
  if (ok0) y[lane] = __fdiv_rn(e0, s);
  if (ok1) y[lane + 32] = __fdiv_rn(e1, s);
}

// boxes_out[i] = clip(rois[i][1:5] / im_scale, im_shape)  -- tools/demo.py:92-95
__global__ void unscale_clip_kernel(const float* __restrict__ rois, int total, int rois_per_img,
                                    const float* __restrict__ im_scale,
                                    const float* __restrict__ im_hw, float* __restrict__ boxes) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int img = i / rois_per_img;
  const float s = im_scale[img];
  const float hmax = __fsub_rn(im_hw[img * 2 + 0], 1.0f), wmax = __fsub_rn(im_hw[img * 2 + 1], 1.0f);
  const float* r = rois + static_cast<long long>(i) * 5;
  float* b = boxes + static_cast<long long>(i) * 4;
  b[0] = clipf(__fdiv_rn(r[1], s), wmax);
  b[1] = clipf(__fdiv_rn(r[2], s), hmax);
  b[2] = clipf(__fdiv_rn(r[3], s), wmax);
  b[3] = clipf(__fdiv_rn(r[4], s), hmax);
}

// The whole im_detect tail (tools/demo.py:84-100 == TesterWrapper.py:244-260) in one launch: boxes =
// clip(rois[:, 1:5] / im_scale, original image shape) for stage 1 then stage 2, masks and scores
// concatenated in the same order, written straight into the per-step output record (the buffer
// that is copied to the host / handed to the all-gather):
//   counts[B] | boxes[B][2n][4] | scores[B][2n][ncls] | masks[B][2n][msz]      (+ valid[B][2n] u8)
// One CTA per output row.
__global__ void __launch_bounds__(128)
detect_tail_kernel(const float* __restrict__ rois, const float* __restrict__ rois_ext,
                   const float* __restrict__ mask, const float* __restrict__ mask_ext,
                   const float* __restrict__ prob, const float* __restrict__ prob_ext,
                   const int* __restrict__ roi_counts, const float* __restrict__ im_scale,
                   const float* __restrict__ im_hw, int n, int msz, int ncls,
                   float* __restrict__ counts, float* __restrict__ boxes, float* __restrict__ scores,
                   float* __restrict__ masks, unsigned char* __restrict__ valid) {
  const int img = blockIdx.y;
  const int row = blockIdx.x;            // 0 .. 2n-1: stage 1 rows then stage 2 rows
  const int stage = row >= n;
  const long long src = static_cast<long long>(img) * n + (row - stage * n);
  const long long dst = static_cast<long long>(img) * 2 * n + row;
  const float* r = (stage ? rois_ext : rois) + src * 5;
  const float* m = (stage ? mask_ext : mask) + src * msz;
  const float* p = (stage ? prob_ext : prob) + src * ncls;
  const int cnt = roi_counts[img];
  if (threadIdx.x < 4) {
    const float s = im_scale[img];
    const float lim = __fsub_rn(im_hw[img * 2 + ((threadIdx.x & 1) ? 0 : 1)], 1.0f);  // x: W-1, y: H-1
    boxes[dst * 4 + threadIdx.x] = clipf(__fdiv_rn(r[1 + threadIdx.x], s), lim);
  }
  if (threadIdx.x == 4) valid[dst] = (row - stage * n) < cnt ? 1 : 0;
  if (threadIdx.x == 5 && row == 0) counts[img] = static_cast<float>(2 * cnt);
  for (int i = threadIdx.x; i < ncls; i += blockDim.x) scores[dst * ncls + i] = p[i];
  for (int i = threadIdx.x; i < msz; i += blockDim.x) masks[dst * msz + i] = m[i];
}

// TesterWrapper._detection_forward tail (lib/caffeWrapper/TesterWrapper.py:229-234): boxes =
// rois[:,1:5] / im_scale; pred = bbox_transform_inv(boxes, deltas) for every class; clip to the
// original image.  One thread per (RoI, class).
__global__ void decode_class_boxes_kernel(const float* __restrict__ rois, int total,
                                          int rois_per_img, const float* __restrict__ bbox_pred,
                                          int bbox_stride, int ncls,
                                          const float* __restrict__ im_scale,
                                          const float* __restrict__ im_hw,
                                          float* __restrict__ out) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total * ncls) return;
  const int i = t / ncls, c = t - i * ncls;
  const int img = i / rois_per_img;
  const float s = im_scale[img];
  const float* r = rois + static_cast<long long>(i) * 5;
  const float* d = bbox_pred + static_cast<long long>(i) * bbox_stride + 4 * c;
  float o[4];
  decode_clip(__fdiv_rn(r[1], s), __fdiv_rn(r[2], s), __fdiv_rn(r[3], s), __fdiv_rn(r[4], s), d[0],
              d[1], d[2], d[3], im_hw[img * 2 + 0], im_hw[img * 2 + 1], o);
  *reinterpret_cast<float4*>(out + (static_cast<long long>(i) * ncls + c) * 4) =
      make_float4(o[0], o[1], o[2], o[3]);
}

static inline int check_launch() { return cudaGetLastError() == cudaSuccess ? MNC_OK : MNC_ERR_CUDA; }

}  // namespace mnc

using namespace mnc;

extern "C" int mnc_generate_anchors(float* out36) {
  double a[9][4];
  generate_anchors_host(a);
  for (int i = 0; i < 9; ++i)
    for (int k = 0; k < 4; ++k) out36[i * 4 + k] = static_cast<float>(a[i][k]);
  return MNC_OK;
}

extern "C" int mnc_rpn_decode2(const float* cls, long long cls_img_stride, long long cls_ch_stride,
                               long long cls_pix_stride, const float* bbox, long long bb_img_stride,
                               long long bb_ch_stride, long long bb_pix_stride,
                               const float* im_info, int batch, int H, int W, int feat_stride,
                               float min_size, int apply_softmax, float* proposals, float* scores,
                               unsigned char* valid, const int* img_hw, int level, void* stream) {
  if (level < 0 || level > 16) return MNC_ERR_ARG;
  Anchors an;
  double a[9][4];
  generate_anchors_host(a);
  for (int i = 0; i < 9; ++i)
    for (int k = 0; k < 4; ++k) an.v[i][k] = static_cast<float>(a[i][k]);
  const int total = H * W * 9;
  dim3 grid((total + 255) / 256, batch);
  rpn_decode_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      cls, cls_img_stride, cls_ch_stride, cls_pix_stride, bbox, bb_img_stride, bb_ch_stride,
      bb_pix_stride, im_info, H, W, feat_stride, min_size, apply_softmax, an, proposals, scores,
      valid, img_hw, level);
  return check_launch();
}

extern "C" int mnc_rpn_decode(const float* cls, long long cls_img_stride, long long cls_ch_stride,
                              long long cls_pix_stride, const float* bbox, long long bb_img_stride,
                              long long bb_ch_stride, long long bb_pix_stride,
                              const float* im_info, int batch, int H, int W, int feat_stride,
                              float min_size, int apply_softmax, float* proposals, float* scores,
                              unsigned char* valid, void* stream) {
  return mnc_rpn_decode2(cls, cls_img_stride, cls_ch_stride, cls_pix_stride, bbox, bb_img_stride,
                         bb_ch_stride, bb_pix_stride, im_info, batch, H, W, feat_stride, min_size,
                         apply_softmax, proposals, scores, valid, nullptr, 0, stream);
}

extern "C" int mnc_write_rois(const float* sorted_boxes, int n_sorted, const int* keep,
                              int keep_stride, const int* num_keep, int max_rois, int batch,
                              int batch_index_mode, float* rois, int* roi_counts, void* stream) {
  dim3 grid((max_rois + 127) / 128, batch);
  write_rois_kernel<<<grid, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      sorted_boxes, n_sorted, keep, keep_stride, num_keep, max_rois, batch_index_mode, rois,
      roi_counts);
  return check_launch();
}

extern "C" int mnc_stage_bridge(const float* rois, const float* bbox_pred, int bbox_stride,
                                const float* seg_cls_prob, int prob_stride, int ncls,
                                const float* im_info, int rois_per_img, int total, float* rois_out,
                                void* stream) {
  if (total <= 0) return MNC_OK;
  stage_bridge_kernel<<<(total + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      rois, bbox_pred, bbox_stride, seg_cls_prob, prob_stride, ncls, im_info, rois_per_img, total,
      rois_out);
  return check_launch();
}

extern "C" int mnc_softmax_rows(const float* in, int in_stride, int rows, int cols, float* out,
                                int out_stride, void* stream) {
  if (rows <= 0) return MNC_OK;
  if (cols <= 0 || cols > 64) return MNC_ERR_ARG;
  softmax_rows_kernel<<<(rows + 3) / 4, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      in, in_stride, rows, cols, out, out_stride);
  return check_launch();
}

extern "C" int mnc_unscale_clip(const float* rois, int total, int rois_per_img,
                                const float* im_scale, const float* im_hw, float* boxes,
                                void* stream) {
  if (total <= 0) return MNC_OK;
  unscale_clip_kernel<<<(total + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      rois, total, rois_per_img, im_scale, im_hw, boxes);
  return check_launch();
}

extern "C" int mnc_detect_tail(const float* rois, const float* rois_ext, const float* mask,
                               const float* mask_ext, const float* prob, const float* prob_ext,
                               const int* roi_counts, const float* im_scale, const float* im_hw,
                               int batch, int n, int msz, int ncls, float* counts, float* boxes,
                               float* scores, float* masks, unsigned char* valid, void* stream) {
  if (batch <= 0 || n <= 0) return MNC_OK;
  dim3 grid(2 * n, batch);
  detect_tail_kernel<<<grid, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      rois, rois_ext, mask, mask_ext, prob, prob_ext, roi_counts, im_scale, im_hw, n, msz, ncls,
      counts, boxes, scores, masks, valid);
  return check_launch();
}

extern "C" int mnc_decode_class_boxes(const float* rois, int total, int rois_per_img,
                                      const float* bbox_pred, int bbox_stride, int ncls,
                                      const float* im_scale, const float* im_hw, float* out,
                                      void* stream) {
  if (total <= 0) return MNC_OK;
  if (ncls <= 0 || bbox_stride < 4 * ncls) return MNC_ERR_ARG;
  const int n = total * ncls;
  decode_class_boxes_kernel<<<(n + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      rois, total, rois_per_img, bbox_pred, bbox_stride, ncls, im_scale, im_hw, out);
  return check_launch();
}
