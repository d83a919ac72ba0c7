// Result rendering on the device (SURVEY.md section 8f row 3): the step right after mask voting in
// tools/demo.py:153-158 and lib/utils/vis_seg.py:101-131 (_convert_pred_to_image): every kept
// instance's 21x21 mask is resized to its (rounded, clipped) box with cv2.resize INTER_LINEAR,
// binarised at cfg.BINARIZE_THRESH and painted, in list order, into an instance-id image and a
// class-id image; each box outline is then drawn into the class image with the value 150.
//
// The reference paints instance after instance over whole sub-arrays; here one thread owns one
// pixel and walks the instance list backwards, stopping at the last writer of that pixel -- the
// same result without the n read-modify-write passes over the image.
//
// cv2.resize (OpenCV, a dependency of the reference, not part of it) is restated as in
// preprocess.cu: fx = (dx + 0.5) * (src / dst) - 0.5 in double, floor, clamp (sx < 0 -> 0, frac 0;
// sx >= src - 1 -> src - 1, frac 0), horizontal pass then vertical pass in fp32.
#include <cuda_runtime.h>
#include <cstdint>

#include "mnc_b200.h"

namespace mnc {

struct InstRec {
  int x1, y1, x2, y2;  // np.round(box).astype(int), clipped to the image (vis_seg.py:106-114)
  int cls;
  int id;              // position among the painted entries of its chunk, 1-based (0: not painted)
};

__device__ __forceinline__ int box_coord(float v) { return static_cast<int>(rintf(v)); }
// voted boxes are integers already (mnc_mv_device); rintf of their fp32 copy is the same value
__device__ __forceinline__ int box_coord(int v) { return v; }

__device__ __forceinline__ void cv_tap(int d, double scale, int n, int& i0, int& i1, float& a0,
                                       float& a1) {
  const double fd = (d + 0.5) * scale - 0.5;   // fraction in double, rounded once (see preprocess.cu)
  int s = static_cast<int>(floor(fd));
  float f = static_cast<float>(fd - s);
  if (s < 0) {
    f = 0.f;
    s = 0;
  }
  if (s >= n - 1) {
    i0 = i1 = n - 1;
    f = 0.f;
  } else {
    i0 = s;
    i1 = s + 1;
  }
  a0 = 1.f - f;
  a1 = f;
}

// numpy slice [a-1 : a+1] along an axis: rows/cols {a-1, a}; empty when a == 0 (start -1 wraps to
// the last element, past the stop).
__device__ __forceinline__ bool in_edge_band(int v, int a) { return a >= 1 && (v == a - 1 || v == a); }

constexpr int kRenderChunk = 256;

// grid (ceil(max W/128), max H, batch); 128 threads, one pixel each.
// img_hw == nullptr: every image is H x W and image b starts at pixel b*H*W.  Otherwise image b is
// img_hw[b] = (H_b, W_b) starting at pixel pix_off[b] (images packed without padding); blocks
// outside their image return at once.
// scores == nullptr: the counts[b] entries are all painted, entry i as instance i+1.  Otherwise
// only the entries with scores[i] >= vis_thresh are, in order, numbered 1, 2, ... by their position
// among them (get_vis_dict, tools/demo.py:103-120, then _convert_pred_to_image).
template <typename BoxT>
__global__ void __launch_bounds__(128)
paste_instances_kernel(const BoxT* __restrict__ boxes, int box_dim, const float* __restrict__ masks,
                       const int* __restrict__ cls, const int* __restrict__ counts,
                       const float* __restrict__ scores, float vis_thresh, int max_n, int M,
                       const int* __restrict__ img_hw, const long long* __restrict__ pix_off, int H,
                       int W, float thresh, int* __restrict__ inst_img, int* __restrict__ cls_img,
                       unsigned char* __restrict__ bgr) {
  __shared__ InstRec recs[kRenderChunk];
  __shared__ int s_warp[4];
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y;
  const int b = blockIdx.z;
  long long img_off = static_cast<long long>(b) * H * W;
  if (img_hw) {
    H = img_hw[2 * b];
    W = img_hw[2 * b + 1];
    img_off = pix_off[b];
    if (y >= H || static_cast<int>(blockIdx.x * blockDim.x) >= W) return;   // block-uniform
  }
  const int n = min(counts[b], max_n);
  const BoxT* pboxes = boxes + static_cast<long long>(b) * max_n * box_dim;
  const float* pmasks = masks + static_cast<long long>(b) * max_n * M * M;
  const int* pcls = cls + static_cast<long long>(b) * max_n;
  const float* pscores = scores ? scores + static_cast<long long>(b) * max_n : nullptr;
  int kept_total = n;
  if (pscores) {
    kept_total = 0;
    for (int base = 0; base < n; base += blockDim.x) {
      const int i = base + threadIdx.x;
      kept_total += __syncthreads_count(i < n && pscores[i] >= vis_thresh);
    }
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

  int inst_val = 0, cls_val = 0;
  bool inst_done = false, cls_done = false;
  int kept_after = 0;   // painted entries in [hi, n)
  // chunks from the end of the list towards its start
  for (int hi = n; hi > 0; hi -= kRenderChunk) {
    const int lo = max(hi - kRenderChunk, 0);
    __syncthreads();
    // two rounds of 128 entries (kRenderChunk = 2 * blockDim.x): every thread takes part in both
    int kept_chunk = 0;
    for (int i = lo + threadIdx.x; i < lo + kRenderChunk; i += blockDim.x) {
      const bool in = i < hi;
      const bool keep = in && (!pscores || pscores[i] >= vis_thresh);
      const unsigned bal = __ballot_sync(0xffffffffu, keep);
      if (lane == 0) s_warp[warp] = __popc(bal);
      __syncthreads();
      int id = kept_chunk + __popc(bal & ((2u << lane) - 1u));   // inclusive count in the chunk
      for (int w = 0; w < warp; ++w) id += s_warp[w];
      kept_chunk += s_warp[0] + s_warp[1] + s_warp[2] + s_warp[3];
      __syncthreads();
      if (!in) continue;
      const BoxT* bx = pboxes + static_cast<long long>(i) * box_dim;
      InstRec r;
      r.x1 = min(max(box_coord(bx[0]), 0), W - 1);
      r.y1 = min(max(box_coord(bx[1]), 0), H - 1);
      r.x2 = min(max(box_coord(bx[2]), 0), W - 1);
      r.y2 = min(max(box_coord(bx[3]), 0), H - 1);
      r.cls = pcls[i];
      r.id = id;
      if (!keep) r.x2 = r.x1 - 1;   // filtered out: an empty box paints nothing
      recs[i - lo] = r;
    }
    const int id_base = kept_total - kept_after - kept_chunk;   // painted entries before lo
    kept_after += kept_chunk;
    __syncthreads();
    const bool all_done = (x >= W) || (inst_done && cls_done);
    if (__syncthreads_and(all_done)) break;
    if (x >= W) continue;
    for (int i = hi - 1; i >= lo && !(inst_done && cls_done); --i) {
      const InstRec r = recs[i - lo];
      const int bw = r.x2 - r.x1 + 1, bh = r.y2 - r.y1 + 1;
      if (bw <= 0 || bh <= 0) continue;  // cv2.resize would reject an empty size; nothing painted
      const bool in_x = x >= r.x1 && x <= r.x2, in_y = y >= r.y1 && y <= r.y2;
      // outline, drawn after this instance's mask (vis_seg.py:123-126)
      if (!cls_done) {
        const bool edge = (in_y && (in_edge_band(x, r.x1) || in_edge_band(x, r.x2))) ||
                          (in_x && (in_edge_band(y, r.y1) || in_edge_band(y, r.y2)));
        if (edge) {
          cls_val = 150;
          cls_done = true;
        }
      }
      if (!(in_x && in_y)) continue;
      int x0, x1i, y0, y1i;
      float ax0, ax1, ay0, ay1;
      cv_tap(x - r.x1, static_cast<double>(M) / bw, M, x0, x1i, ax0, ax1);
      cv_tap(y - r.y1, static_cast<double>(M) / bh, M, y0, y1i, ay0, ay1);
      const float* m = pmasks + static_cast<long long>(i) * M * M;
      const float r0 = __fadd_rn(__fmul_rn(m[y0 * M + x0], ax0), __fmul_rn(m[y0 * M + x1i], ax1));
      const float r1 = __fadd_rn(__fmul_rn(m[y1i * M + x0], ax0), __fmul_rn(m[y1i * M + x1i], ax1));
      const float v = __fadd_rn(__fmul_rn(r0, ay0), __fmul_rn(r1, ay1));
      if (v >= thresh) {
        if (!inst_done) {
          inst_val = id_base + r.id;
          inst_done = true;
        }
        if (!cls_done) {
          cls_val = r.cls;
          cls_done = true;
        }
      }
    }
  }
  if (x >= W) return;
  const long long o = img_off + static_cast<long long>(y) * W + x;
  if (inst_img) inst_img[o] = inst_val;
  if (cls_img) cls_img[o] = cls_val;
  if (bgr) {
    // _get_voc_color_map (vis_seg.py:133-148): bit j of each colour channel comes from bits
    // 3j, 3j+1, 3j+2 of the class id, most significant first; stored BGR as demo.py:163 does.
    int cid = cls_val & 255, r = 0, g = 0, bl = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      r |= (cid & 1) << (7 - j);
      g |= ((cid >> 1) & 1) << (7 - j);
      bl |= ((cid >> 2) & 1) << (7 - j);
      cid >>= 3;
    }
    bgr[o * 3 + 0] = static_cast<unsigned char>(bl);
    bgr[o * 3 + 1] = static_cast<unsigned char>(g);
    bgr[o * 3 + 2] = static_cast<unsigned char>(r);
  }
}

// Binarised, box-sized masks packed one after another (voc_eval.py:249-251 resizes every
// prediction this way before mask_overlap): out[offset[i] + dy * bw + dx] = resized >= thresh.
// grid (ceil(max_area/256), n).
__global__ void __launch_bounds__(256)
binarize_masks_kernel(const int* __restrict__ rboxes, const float* __restrict__ masks, int M,
                      float thresh, const long long* __restrict__ offsets,
                      unsigned char* __restrict__ out) {
  const int i = blockIdx.y;
  const int x1 = rboxes[i * 4 + 0], y1 = rboxes[i * 4 + 1];
  const int bw = rboxes[i * 4 + 2] - x1 + 1, bh = rboxes[i * 4 + 3] - y1 + 1;
  if (bw <= 0 || bh <= 0) return;
  const float* m = masks + static_cast<long long>(i) * M * M;
  for (long long p = blockIdx.x * blockDim.x + threadIdx.x; p < static_cast<long long>(bw) * bh;
       p += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int dx = static_cast<int>(p % bw), dy = static_cast<int>(p / bw);
    int x0, x1i, y0, y1i;
    float ax0, ax1, ay0, ay1;
    cv_tap(dx, static_cast<double>(M) / bw, M, x0, x1i, ax0, ax1);
    cv_tap(dy, static_cast<double>(M) / bh, M, y0, y1i, ay0, ay1);
    const float r0 = __fadd_rn(__fmul_rn(m[y0 * M + x0], ax0), __fmul_rn(m[y0 * M + x1i], ax1));
    const float r1 = __fadd_rn(__fmul_rn(m[y1i * M + x0], ax0), __fmul_rn(m[y1i * M + x1i], ax1));
    const float v = __fadd_rn(__fmul_rn(r0, ay0), __fmul_rn(r1, ay1));
    out[offsets[i] + p] = v >= thresh ? 1 : 0;
  }
}

}  // namespace mnc

extern "C" int mnc_paste_instances(const float* boxes, int box_dim, const float* masks,
                                   const int* cls, const int* counts, int batch, int max_n,
                                   int mask_size, int H, int W, float thresh, int* inst_img,
                                   int* cls_img, unsigned char* bgr, void* stream) {
  if (batch <= 0 || max_n < 0 || box_dim < 4 || mask_size <= 0 || H <= 0 || W <= 0)
    return MNC_ERR_ARG;
  dim3 grid((W + 127) / 128, H, batch);
  mnc::paste_instances_kernel<float><<<grid, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      boxes, box_dim, masks, cls, counts, nullptr, 0.f, max_n, mask_size, nullptr, nullptr, H, W,
      thresh, inst_img, cls_img, bgr);
  return cudaGetLastError() == cudaSuccess ? MNC_OK : MNC_ERR_CUDA;
}

extern "C" int mnc_paste_voted_ragged(const int* n_res, const float* res_score, const int* res_class,
                                      const int* result_box, const float* result_mask, int batch,
                                      int max_results, int mask_size, const int* img_hw,
                                      const long long* pix_off, int max_h, int max_w,
                                      float vis_thresh, float thresh, int* inst_img, int* cls_img,
                                      unsigned char* bgr, void* stream) {
  if (batch <= 0 || max_results < 0 || mask_size <= 0 || max_h <= 0 || max_w <= 0 || !n_res ||
      !res_score || !img_hw || !pix_off)
    return MNC_ERR_ARG;
  dim3 grid((max_w + 127) / 128, max_h, batch);
  mnc::paste_instances_kernel<int><<<grid, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      result_box, 4, result_mask, res_class, n_res, res_score, vis_thresh, max_results, mask_size,
      img_hw, pix_off, max_h, max_w, thresh, inst_img, cls_img, bgr);
  return cudaGetLastError() == cudaSuccess ? MNC_OK : MNC_ERR_CUDA;
}

extern "C" int mnc_binarize_masks(const int* rboxes, const float* masks, int n, int mask_size,
                                  float thresh, const long long* offsets, int max_area,
                                  unsigned char* out, void* stream) {
  if (n < 0 || mask_size <= 0) return MNC_ERR_ARG;
  if (n == 0 || max_area <= 0) return MNC_OK;
  int gx = (max_area + 255) / 256;
  if (gx > 1024) gx = 1024;
  mnc::binarize_masks_kernel<<<dim3(gx, n), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      rboxes, masks, mask_size, thresh, offsets, out);
  return cudaGetLastError() == cudaSuccess ? MNC_OK : MNC_ERR_CUDA;
}
