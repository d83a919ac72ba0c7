/*
 * mnc_b200 -- C-ABI of the B200-native MNC (Multi-task Network Cascades) inference hot path.
 *
 * Every entry point is `extern "C"`, takes plain pointers / sizes / a `cudaStream_t` passed as
 * `void*`, and returns an `int` status (MNC_OK == 0).  No torch types cross this boundary.
 *
 * Two families:
 *   (1) reference-compatible HOST-pointer entry points that replace the reference's own native
 *       functions one-for-one (`_nms`, `_mv`; caller-owned host buffers, synchronous):
 *         mnc_nms_host   <- lib/nms/gpu_nms.hpp:1-2     (void _nms(...),  lib/nms/nms_kernel.cu:91-144)
 *         mnc_mv_host    <- lib/nms/gpu_mv.hpp:1-4      (void _mv(...),   lib/nms/mv_kernel.cu:242-348)
 *         mnc_bbox_overlaps_host <- lib/utils/bbox.pyx:15-55 (utils.cython_bbox.bbox_overlaps)
 *   (2) DEVICE-pointer, stream-ordered entry points that replace the Caffe layers' Forward_gpu on
 *       the path (each cites the layer it replaces).  These are what the host-side Python layer
 *       mirror (mnc_b200/lib/...) and the batched engine (mnc_b200/engine.py) call.
 *
 * Unless stated otherwise: fp32 tensors are NCHW as in Caffe blobs; "split" tensors are NHWC
 * stored as two bf16 planes (hi, lo) with x ~= hi + lo (see DESIGN.md, "Data layout in HBM").
 */
#ifndef MNC_B200_H_
#define MNC_B200_H_

#ifdef __cplusplus
extern "C" {
#endif

#define MNC_OK 0
#define MNC_ERR_ARG 1    /* invalid argument / unsupported shape */
#define MNC_ERR_CUDA 2   /* a CUDA runtime call or launch failed (see mnc_last_cuda_error) */
#define MNC_ERR_DRIVER 3 /* cuTensorMapEncodeTiled unavailable or failed */
#define MNC_ERR_NOGPU 4  /* no CUDA device visible */

/* Library identity / diagnostics. */
int mnc_abi_version(void);
const char* mnc_last_cuda_error(void);
int mnc_device_count(void);

/* ---------------------------------------------------------------------------------------------
 * Tensor-core implicit GEMM: 3x3/pad1/stride1 convolution (taps == 9) or inner product / 1x1
 * convolution (taps == 1) with fused bias + ReLU.
 * Replaces Convolution (caffe-mnc/src/caffe/layers/cudnn_conv_layer.cu:11-54, conv_layer.cu:8-23)
 * and InnerProduct (caffe-mnc/src/caffe/layers/inner_product_layer.cu:21-27) Forward_gpu.
 *   a_hi/a_lo : bf16 [batch][H][W][Cin] planes (inner product: batch=1, H=1, W=rows, Cin=K)
 *   w_hi/w_lo : bf16 [Cout][taps*Cin] planes, K index = tap*Cin + c, tap = ky*3+kx
 *   out_mode 0: out0/out1 = bf16 hi/lo planes; 1: out0 = fp32 (out1 ignored);
 *            2: (conv only) hi/lo planes of the 2x2/2 ceil-mode max-pooled output
 *               [batch][ceil(H/2)][ceil(W/2)][..] -- Pooling fused into the epilogue
 *               (pooling_layer.cu:11-47, pooling_layer.cpp:90-93)
 *   output element (pixel p, channel c) at p*out_pix_stride + out_ch_offset + c
 *   split_k > 1 (fp32 mode only): partial sums go to plane s at s*split_stride; finish with
 *   mnc_splitk_reduce.  bn: Cout tile (0 = auto, 64/128/256).  max_ctas: 0 = one CTA per SM.
 */
int mnc_igemm_tc(const void* a_hi, const void* a_lo, int batch, int H, int W, int Cin,
                 const void* w_hi, const void* w_lo, int Cout, int taps, const float* bias,
                 int relu, int out_mode, void* out0, void* out1, long long out_pix_stride,
                 int out_ch_offset, int split_k, long long split_stride, int bn, int max_ctas,
                 void* stream);

/* General form of mnc_igemm_tc (same layers replaced: cudnn_conv_layer.cu:11-54 / conv_layer.cu:8-23 +
 * im2col.cu:9-39, inner_product_layer.cu:21-27, relu_layer.cu:9-14, pooling_layer.cu:11-47).
 * in_fmt 0: split-bf16 operands (a0 = hi, a1 = lo, a2 unused; w0 = hi, w1 = lo) -- 3 bf16 MMAs per
 *   k slice.  in_fmt 1 ("precision mode 1"): tri-plane operands: a0 = fp16(x * 2^ea), a1 = e4m3 of
 *   the fp16 residual * 2^6, a2 = e4m3(x * 2^ea * 2^-5); w0 = fp16(w * 2^ew), w1 = e4m3(w * 2^ew *
 *   2^-6), w2 = e4m3 of the residual * 2^5.  X.W * 2^(ea+ew) = a0.w0 + a1.w1 + a2.w2: one fp16
 *   product plus two FP8 products (kind::f8f6f4, twice the rate), 2 tensor-work units per MAC.
 * out_mode 0 / 2: split-bf16 (out0, out1); 1: fp32 (out0); 4 / 5: tri-plane activation (out0 fp16,
 *   out1 residual, out2 copy) with scale out_scale = 2^e; 2 and 5 fuse the 2x2 ceil-mode max pool.
 * acc_scale: accumulator -> true value (2^-(ea+ew) for tri-plane operands, 1 otherwise).
 * amax: optional device word receiving atomicMax(|output|) as float bits (scale calibration). */
int mnc_igemm_tc2(int in_fmt, const void* a0, const void* a1, const void* a2, int batch, int H,
                  int W, int Cin, const void* w0, const void* w1, const void* w2, int Cout, int taps,
                  const float* bias, int relu, int out_mode, void* out0, void* out1, void* out2,
                  long long out_pix_stride, int out_ch_offset, int split_k, long long split_stride,
                  int bn, int max_ctas, float acc_scale, float out_scale, unsigned int* amax,
                  void* stream);

/* Mixed-size batches.  Image b of the batch fills the top-left corner of the zero-padded blob;
 * img_hw is a DEVICE int32 [batch][2] array of the images' sizes at input resolution (blob rows
 * and columns of image b before any pooling), and `level` the number of 2x2 ceil-mode pools
 * between the input and this launch (0 = conv1_x ... 4 = conv5_x / RPN), so that image b covers
 * ((h + 2^level - 1) >> level, (w + 2^level - 1) >> level) of the launch's map.  img_hw lives in
 * device memory, so these entry points check only `level` (MNC_ERR_ARG outside 0..16) and do NOT
 * validate the sizes: the CALLER owns that check and must reject, on the host before uploading,
 * any size < 1 or larger than the blob (the Python layer does so in engine.check_extents).  Invalid
 * sizes give wrong results but never an out-of-map access: the kernels clamp every extent to the
 * map (the RoI warps to [1, map]).  img_hw == NULL is the whole-blob launch of the entry point
 * without the suffix.
 *
 * mnc_igemm_tc3: mnc_igemm_tc2 whose outputs outside their image are exact zeros (out_mode 0 / 4);
 * with the fused pool (2 / 5) pixels outside the image take no part in a window and pooled pixels
 * outside the image's level + 1 extent are zeros.  Running maxima (amax) count pixels inside. */
int mnc_igemm_tc3(int in_fmt, const void* a0, const void* a1, const void* a2, int batch, int H,
                  int W, int Cin, const void* w0, const void* w1, const void* w2, int Cout, int taps,
                  const float* bias, int relu, int out_mode, void* out0, void* out1, void* out2,
                  long long out_pix_stride, int out_ch_offset, int split_k, long long split_stride,
                  int bn, int max_ctas, float acc_scale, float out_scale, unsigned int* amax,
                  const int* img_hw, int level, void* stream);
/* Split-K reductions of a conv launch over a [batch][H][W] map (rows = batch*H*W) with the rows
 * outside their image written as zeros. */
int mnc_splitk_reduce2(const float* partial, int splits, long long split_stride, long long rows,
                       int cols, const float* bias, int relu, int out_mode, void* out0, void* out1,
                       long long out_row_stride, int out_ch_offset, const int* img_hw, int level,
                       int H, int W, void* stream);
int mnc_splitk_reduce_tri2(const float* partial, int splits, long long split_stride, long long rows,
                           int cols, const float* bias, int relu, float scale, void* h, void* l,
                           void* c, long long out_row_stride, int out_ch_offset, unsigned int* amax,
                           const int* img_hw, int level, int H, int W, void* stream);
/* conv1_1 (level 0) of a mixed-size batch. */
int mnc_conv1_1_tc3(const float* data_nchw, int batch, int H, int W, const void* w_stacked,
                    const float* bias, int out_mode, void* out0, void* out1, void* out2,
                    float out_scale, unsigned int* amax, const int* img_hw, void* stream);
/* Proposal decode: anchors outside their image's extent are marked invalid. */
int mnc_rpn_decode2(const float* cls, long long cls_img_stride, long long cls_ch_stride,
                    long long cls_pix_stride, const float* bbox, long long bb_img_stride,
                    long long bb_ch_stride, long long bb_pix_stride, const float* im_info, int batch,
                    int H, int W, int feat_stride, float min_size, int apply_softmax,
                    float* proposals, float* scores, unsigned char* valid, const int* img_hw,
                    int level, void* stream);
/* RoI warps: samples are bounded and clamped by the extent of the RoI's image (roi[0]); the map's
 * row stride stays W.  Not combined with the A/B kernel forms (set_walk / set_rows): MNC_ERR_ARG. */
int mnc_roi_warp_split2(const float* feat_nhwc, int C, int H, int W, const float* rois, int R,
                        int sub, float spatial_scale, void* o14_hi, void* o14_lo, void* o7_hi,
                        void* o7_lo, const int* img_hw, int level, void* stream);
int mnc_roi_warp_tri2(const float* feat_nhwc, int C, int H, int W, const float* rois, int R, int sub,
                      float spatial_scale, float scale, void* o14_h, void* o14_l, void* o14_c,
                      void* o7_h, void* o7_l, void* o7_c, const int* img_hw, int level, void* stream);

/* Tri-plane helpers.  fp32 -> (fp16 h, e4m3 l, e4m3 c) with scale 2^e and back (h + l / 2^6) *
 * inv_scale; n % 4 == 0. */
int mnc_f32_to_tri(const float* in, long long n, float scale, void* h, void* l, void* c,
                   unsigned int* amax, void* stream);
int mnc_tri_to_f32(const void* h, const void* l, long long n, float inv_scale, float* out, void* stream);
/* mnc_splitk_reduce with a tri-plane result. */
int mnc_splitk_reduce_tri(const float* partial, int splits, long long split_stride, long long rows,
                          int cols, const float* bias, int relu, float scale, void* h, void* l,
                          void* c, long long out_row_stride, int out_ch_offset, unsigned int* amax,
                          void* stream);
/* MaskPooling (mask_pooling_layer.cu:13-26) + 2x2 max pool on tri-plane NHWC RoI features
 * (R,14,14,C) x mask14 (R,196) -> (R,7,7,C), same exponent in and out. */
int mnc_mask_pool_tri(const void* f_h, const void* f_l, const float* mask14, int R, int C, void* o_h,
                      void* o_l, void* o_c, void* stream);
/* mnc_roi_warp_split (ROIWarping roi_warping_layer.cu:67-107 + the 2x2 pools) with tri-plane
 * outputs scaled by `scale`. */
int mnc_roi_warp_tri(const float* feat_nhwc, int C, int H, int W, const float* rois, int R, int sub,
                     float spatial_scale, float scale, void* o14_h, void* o14_l, void* o14_c,
                     void* o7_h, void* o7_l, void* o7_c, void* stream);

/* Thread-block-cluster size of mnc_igemm_tc launches: 2 (default) = CTA pairs (cta_group::2): one
 * M = 256 MMA per instruction, each CTA holds its 128 pixel rows and half of the weight tile;
 * 1 = single-CTA 128-row tiles. */
int mnc_igemm_set_cluster(int cluster_size);
/* A/B switch: CTA pairs (cta_group::2, M = 256) in the halo kernel's precision mode 1 (default on). */
int mnc_igemm_set_halo_pair(int on);
/* K elements per pipeline stage: 64 (SWIZZLE_128B), 32 (SWIZZLE_64B, twice the stages) or
 * 0 = default (64; the 192-wide Cout tile always uses 32).  bn also accepts 192. */
int mnc_igemm_set_block_k(int bk);
/* out_mode 0 epilogue: 1 (default) = stage tiles in shared memory and write them with TMA bulk
 * tensor stores; 0 = per-thread 16-byte global stores. */
int mnc_igemm_set_tma_store(int on);
/* 3x3 convolutions with Cout tiles <= 128: 1 (default) = halo kernel (one TMA box of the pixel
 * tile + border feeds all 9 filter taps through shifted shared-memory descriptors);
 * 0 = per-tap activation loads. */
int mnc_igemm_set_halo(int on);

/* Same contract as mnc_igemm_tc on the fp32 SIMT pipes (exact fp32 FMA on hi+lo operands).
 * Not on the product path: it is the on-device cross-check for the tensor-core kernel. */
int mnc_igemm_simt(const void* a_hi, const void* a_lo, int batch, int H, int W, int Cin,
                   const void* w_hi, const void* w_lo, int Cout, int taps, const float* bias,
                   int relu, int out_mode, void* out0, void* out1, long long out_pix_stride,
                   int out_ch_offset, void* stream);

/* out = act(sum_s partial[s] + bias); rows x cols fp32 partial planes -> split bf16 or fp32. */
int mnc_splitk_reduce(const float* partial, int splits, long long split_stride, long long rows,
                      int cols, const float* bias, int relu, int out_mode, void* out0, void* out1,
                      long long out_row_stride, int out_ch_offset, void* stream);

/* conv1_1: 3 -> Cout(64) 3x3/pad1 + bias + ReLU on the fp32 NCHW input blob `data`
 * (test.prototxt:19-43), written as split NHWC.  weight fp32 [Cout][3][3][3] (Caffe order). */
int mnc_conv1_1(const float* data_nchw, int batch, int H, int W, const float* weight,
                const float* bias, int Cout, void* out_hi, void* out_lo, void* stream);
/* The same layer on the tensor cores (what the engine uses; the fp32 FMA form above stays as the
 * cross-check).  w_stacked: bf16 [128][32], rows 0..63 / 64..127 = hi / lo plane of
 * weight.reshape(64, 27) (k = c*9 + ky*3 + kx), columns 27..31 zero.  Cout is 64. */
int mnc_conv1_1_tc(const float* data_nchw, int batch, int H, int W, const void* w_stacked,
                   const float* bias, void* out_hi, void* out_lo, void* stream);
/* General form: out_mode 0 = split-bf16 (out0 hi, out1 lo), 4 = tri-plane (out0 fp16, out1 e4m3
 * residual, out2 e4m3 copy; values scaled by out_scale, a power of two).  amax (optional, device)
 * receives atomicMax of |output| as float bits. */
int mnc_conv1_1_tc2(const float* data_nchw, int batch, int H, int W, const void* w_stacked,
                    const float* bias, int out_mode, void* out0, void* out1, void* out2,
                    float out_scale, unsigned int* amax, void* stream);

/* 2x2 stride-2 ceil-mode max pooling on split NHWC (pooling_layer.cu:11-47, pooling_layer.cpp:90-93). */
int mnc_maxpool2x2_split(const void* in_hi, const void* in_lo, int batch, int H, int W, int C,
                         void* out_hi, void* out_lo, void* stream);

/* split NHWC -> fp32 NCHW (blob view of an internal activation) and back. */
int mnc_split_to_nchw(const void* in_hi, const void* in_lo, int batch, int H, int W, int C,
                      float* out_nchw, void* stream);
int mnc_nchw_to_split(const float* in_nchw, int batch, int C, int H, int W, void* out_hi,
                      void* out_lo, void* stream);
/* fp32 [rows][cols] row-major -> split planes (and back). */
int mnc_f32_to_split(const float* in, long long n, void* out_hi, void* out_lo, void* stream);
int mnc_split_to_f32(const void* in_hi, const void* in_lo, long long n, float* out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * NMS.  mnc_nms_host is the drop-in for the reference's `_nms` (lib/nms/gpu_nms.hpp:1-2,
 * lib/nms/nms_kernel.cu:91-144): caller-owned HOST buffers, boxes already sorted by score
 * (descending), keep_out holds >= boxes_num ints, suppression when IoU > thresh (strict, :71),
 * synchronous.  Differences: returns a status instead of printing CUDA errors (:12-19); the
 * suppression matrix stays on the device (only the keep list crosses PCIe).
 */
int mnc_nms_host(int* keep_out, int* num_out, const float* boxes_host, int boxes_num,
                 int boxes_dim, float nms_overlap_thresh, int device_id);
/* nms.gpu_nms.gpu_nms (lib/nms/gpu_nms.pyx:16-31) in one call: UNSORTED dets (n x dim, dim >= 5,
 * score in column 4) in host memory -> keep_out = indices of the kept rows in score order
 * (`order[keep]`), *num_out their number.  Sort (score descending, ties by ascending index), gather,
 * NMS and scan run on the device. */
int mnc_gpu_nms_host(int* keep_out, int* num_out, const float* dets_host, int n, int dim,
                     float nms_overlap_thresh, int device_id);

/* Device form, batched over `problems` independent box lists (images x classes):
 *   boxes + p*problem_stride : n_max x box_stride floats (x1,y1,x2,y2,...), score-sorted
 *   counts[p] (device, may be NULL = n_max) : number of valid boxes of problem p
 *   keep_out + p*keep_stride : kept positions (into the sorted list), num_out[p] of them,
 *   stopping after max_keep (<= 0: no limit).  workspace: mnc_nms_workspace_bytes(n_max, problems). */
long long mnc_nms_workspace_bytes(int n_max, int problems);
int mnc_nms_sorted(const float* boxes, int box_stride, long long problem_stride, const int* counts,
                   int n_max, int problems, float thresh, int max_keep, void* workspace,
                   int* keep_out, int keep_stride, int* num_out, void* stream);
/* When max_keep is small against n_max (n_max >= 1024, max_keep <= 2048, 4*max_keep <= n_max: the
 * ProposalLayer's 6000 -> 300, lib/pylayer/proposal_layer.py:147-152) mnc_nms_sorted runs a capped
 * greedy NMS that never builds the suppression matrix (candidates walked in blocks of 64 against
 * the kept boxes held in shared memory; workspace unused) -- same keep list.
 * mnc_nms_set_lazy(mode): 2 (default) = a thread-block cluster of 8 CTAs per problem, 1 = one CTA
 * per problem, 0 = always the mask + scan pair (cross-check / A-B switch); returns the previous
 * mode. */
int mnc_nms_set_lazy(int on);
/* number of kernels mnc_nms_sorted launches for these sizes (1: capped form, 2: mask + scan) */
int mnc_nms_sorted_launches(int n_max, int max_keep);

/* `scores.argsort()[::-1]` (lib/pylayer/proposal_layer.py:139, lib/nms/gpu_nms.pyx:25-26) with the
 * tie rule (score desc, index asc).  Problem p reads keys at
 * keys + (p / inner)*outer_stride + (p % inner)*inner_stride + i*key_stride, i < n; entries with
 * valid[p*n + i] == 0 are dropped (valid may be NULL).  order[p*n + rank] = i, n_valid[p] = count. */
int mnc_rank_sort_desc(const float* keys, long long outer_stride, long long inner_stride, int inner,
                       int key_stride, const unsigned char* valid, int n, int problems, int* order,
                       int* n_valid, void* stream);
/* Same ordering, but only the k best entries are produced: order[prob][0..min(n_valid, k)) and
 * n_out[prob] = min(n_valid, k) -- what `scores.argsort()[::-1][:pre_nms_topN]`
 * (lib/pylayer/proposal_layer.py:139-142) consumes.  Radix select + sort of the selection in one
 * CTA per problem; returns MNC_ERR_ARG when n / k exceed its shared-memory budget
 * (8*pow2(k) + 4*n <= 200 KB), in which case use mnc_rank_sort_desc. */
int mnc_topk_sort_desc(const float* keys, long long outer_stride, long long inner_stride, int inner,
                       int key_stride, const unsigned char* valid, int n, int problems, int k,
                       int* order, int order_stride, int* n_out, void* stream);
/* dst[p][k][0..3] = src[(p / inner)][order[p*order_stride + k]][0..3], k < min(counts[p], n_out);
 * out_counts[p] = that minimum. */
int mnc_gather_boxes(const float* src, int src_stride, long long src_outer_stride, int inner,
                     const int* order, int order_stride, const int* counts, int n_out, int problems,
                     float* dst, int* out_counts, void* stream);

/* ---------------------------------------------------------------------------------------------
 * ProposalLayer pieces (lib/pylayer/proposal_layer.py:52-175), StageBridgeLayer.forward_test
 * (lib/pylayer/stage_bridge_layer.py:237-255), Caffe Softmax (softmax_layer.cu:86-120) and the
 * im_detect tail (tools/demo.py:92-95), all on device.
 */
int mnc_generate_anchors(float* out36); /* lib/transform/anchors.py:38-49, 9x4 */
/* Element (img, ch, pixel) of cls at cls + img*img_stride + ch*ch_stride + pixel*pix_stride
 * (so both NCHW blobs and the engine's NHWC buffer work); channels [bg a0..a8 | fg a0..a8]
 * (test.prototxt:440-462) and [4a..4a+3]; apply_softmax: cls holds logits.
 * Outputs per image: proposals [H*W*9][4], scores [H*W*9], valid [H*W*9] (min-size filter). */
int mnc_rpn_decode(const float* cls, long long cls_img_stride, long long cls_ch_stride,
                   long long cls_pix_stride, const float* bbox, long long bb_img_stride,
                   long long bb_ch_stride, long long bb_pix_stride, const float* im_info, int batch,
                   int H, int W, int feat_stride, float min_size, int apply_softmax,
                   float* proposals, float* scores, unsigned char* valid, void* stream);
int mnc_write_rois(const float* sorted_boxes, int n_sorted, const int* keep, int keep_stride,
                   const int* num_keep, int max_rois, int batch, int batch_index_mode, float* rois,
                   int* roi_counts, void* stream);
int mnc_stage_bridge(const float* rois, const float* bbox_pred, int bbox_stride,
                     const float* seg_cls_prob, int prob_stride, int ncls, const float* im_info,
                     int rois_per_img, int total, float* rois_out, void* stream);
int mnc_softmax_rows(const float* in, int in_stride, int rows, int cols, float* out,
                     int out_stride, void* stream);
int mnc_unscale_clip(const float* rois, int total, int rois_per_img, const float* im_scale,
                     const float* im_hw, float* boxes, void* stream);
/* The im_detect tail (tools/demo.py:84-100) in one launch, into the per-step output record:
 * counts[B] (valid detections, as float), boxes[B][2n][4] = clip(rois[:,1:5] / im_scale, image),
 * scores[B][2n][ncls], masks[B][2n][msz] -- stage 1 rows, then stage 2 rows -- and valid[B][2n]. */
int mnc_detect_tail(const float* rois, const float* rois_ext, const float* mask, const float* mask_ext,
                    const float* prob, const float* prob_ext, const int* roi_counts,
                    const float* im_scale, const float* im_hw, int batch, int n, int msz, int ncls,
                    float* counts, float* boxes, float* scores, float* masks, unsigned char* valid,
                    void* stream);

/* ---------------------------------------------------------------------------------------------
 * The three MNC Caffe layers, Forward_gpu contract (fp32 NCHW device blobs):
 *   ROIWarping  roi_warping_layer.cu:110-122 : feat (B,C,H,W), rois (R,5) -> out (R,C,ph,pw)
 *   MaskResize  mask_resize_layer.cu:76-84   : in (N,C,ih,iw) -> out (N,C,oh,ow)
 *   MaskPooling mask_pooling_layer.cu:29-41  : feat (N,C,H,W), mask (N,1,H,W) -> out (N,C,H,W)
 */
int mnc_roi_warp_nchw(const float* feat, int C, int H, int W, const float* rois, int R,
                      int pooled_h, int pooled_w, float spatial_scale, float* out, void* stream);
/* ROIWarping 28x28 / 14x14 kernel choice (all bit-identical; scripts/gpu_roi_stage_ab.py measures them):
 * 2 (default) = row walk (a warp per output plane keeps the two live feature rows in registers:
 * ~1.5 loads per output); 1 = RoI window staged in shared memory (28x28 only; 4-byte cp.async,
 * channel pairs interleaved, packed fp32x2 arithmetic); 0 = per-tap gathers through L1 (round-1
 * kernel; other pooled sizes always use it).  Returns the previous value. */
int mnc_roi_warp_set_stage(int on);
/* Launch shape of the row-walk kernel: threads per CTA (multiple of 32, <= 256) and channels per
 * CTA (default 128 / 32: every warp of the CTA owns planes; scripts/gpu_roi_walk_shape_ab.py). */
int mnc_roi_warp_set_walk_shape(int threads, int channels_per_cta);
int mnc_roi_warp_set_walk_planes14(int planes);   /* 14x14 row walk: planes per lane, 4 (default) or 8 */
/* Fused engine form (mnc_roi_warp_split / mnc_roi_warp_tri): 0 (default) = per-cell gathers,
 * 1 = row walk (bit-identical outputs, 2.5x fewer loads, measured no faster:
 * scripts/gpu_roi_rows_ab.py).  Returns the previous value. */
int mnc_roi_warp_set_rows(int on);
int mnc_mask_resize_nchw(const float* in, int N, int C, int in_h, int in_w, int out_h, int out_w,
                         float* out, void* stream);
int mnc_mask_pool_nchw(const float* feat, const float* mask, int N, int C, int H, int W,
                       float* out, void* stream);
/* Fused engine forms on split NHWC: RoI warp (+2x2 max when sub == 2) to [R][14][14][C] plus the
 * 7x7 box pool [R][7][7][C]; sigmoid + 21->14 mask resize; mask pooling + 2x2 max. */
int mnc_roi_warp_split(const float* feat_nhwc /* fp32 [B][H][W][C] */, int C, int H, int W,
                       const float* rois, int R, int sub, float spatial_scale, void* o14_hi,
                       void* o14_lo, void* o7_hi, void* o7_lo, void* stream);
/* Kernel choice for mnc_roi_warp_split: 0 (default) = one gather of 4 taps per sample, 1 =
 * column-walking kernel (separable bilinear, taps cached in registers; 2.4x fewer loads but
 * measured 1.2-1.5x slower: serial dependence per thread, scripts/gpu_roi_warp_ab.py).  Returns the previous setting.
 * For A/B measurement (scripts/microbench.py). */
int mnc_roi_warp_set_walk(int on);
int mnc_sigmoid_mask_resize(const float* logits, int stride, int R, int mask_size, int out_size,
                            float* mask_proposal, float* mask_resized, void* stream);
int mnc_mask_pool_split(const void* f_hi, const void* f_lo, const float* mask14, int R, int C,
                        void* o_hi, void* o_lo, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Mask voting.  mnc_mv_host is the drop-in for the reference's `_mv` (lib/nms/gpu_mv.hpp:1-4,
 * lib/nms/mv_kernel.cu:242-348): HOST buffers, candidate_start holds END offsets (:101-102),
 * outputs result_num x mask_size^2 floats and result_num x 4 ints [x1,y1,x2,y2]; synchronous.
 * Differences: returns a status; honours device_id; needs no nb*H*W render buffer.
 * mnc_bbox_overlaps_host: utils.cython_bbox.bbox_overlaps (lib/utils/bbox.pyx:15-55), float64.
 */
int mnc_mv_host(const float* all_boxes, const float* all_masks, int all_boxes_num,
                const int* candidate_inds, const int* candidate_start,
                const float* candidate_weights, int candidate_num, int image_height,
                int image_width, int box_dim, int mask_size, int result_num,
                float* finalize_output_mask, int* finalize_output_box, int device_id);
int mnc_bbox_overlaps_host(const double* boxes, int N, const double* query, int K, double* out);

/* Device pipeline of gpu_mask_voting (lib/transform/mask_transform.py:213-286), batched:
 * after per-class rank sort + NMS (mnc_rank_sort_desc / mnc_gather_boxes / mnc_nms_sorted with
 * problems = batch*(ncls-1)), vote_select picks the global threshold and enumerates results,
 * vote_candidates builds the (inds, weights) lists, mv_device renders/aggregates/resizes.
 * mv_device's bbox_ws: int32 workspace of batch*max_results*4 + batch entries. */
int mnc_vote_select(const float* scores, int nb, int ncls, const int* order, const int* keep,
                    int keep_stride, const int* num_keep, int max_per_image, int max_results,
                    int batch, int* res_box_idx, int* res_class, float* res_score, int* n_res,
                    int* class_bar, int* overflow, void* stream);
int mnc_vote_candidates(const float* boxes, const float* scores,
                        const unsigned char* box_valid /* [batch][nb], NULL = all */, int nb,
                        int ncls, const int* res_box_idx, const int* res_class, const int* n_res,
                        int max_results, int batch, double iou_thresh, int* cand_inds,
                        float* cand_weights, int* cand_begin, int* cand_end, void* stream);
int mnc_mv_device(const float* boxes, const float* masks, int nb, int box_dim, int mask_size,
                  const int* cand_inds, const float* cand_weights, long long cand_img_stride,
                  const int* cand_begin, const int* cand_end, const int* n_res, int max_results,
                  int batch, const int* im_hw, int* bbox_ws, float* out_mask, int* out_box,
                  void* stream);
/* mv_device finds each result's tight box in two passes (every 6th pixel of every 6th row, then
 * exactly the pixels outside the box the first pass found): same boxes as one full sweep of the
 * region.  mnc_mv_set_two_pass(0) selects the single sweep (cross-check / A-B switch); returns the
 * previous setting.  mnc_mv_device_launches(): kernels per mnc_mv_device call (5 / 4). */
int mnc_mv_set_two_pass(int on);
int mnc_mv_device_launches(void);
/* A/B knob: pixel stride of the coarse pass and CTAs per result of the coarse / border pass
 * (defaults 6, 2, 16: the best of the shapes measured, scripts/gpu_mv_shape_ab.py). */
int mnc_mv_set_shape(int stride, int chunks_coarse, int chunks_border);

/* ---------------------------------------------------------------------------------------------
 * Input preparation on the device (SURVEY.md section 8f, "next" row 1): prep_im_for_blob +
 * im_list_to_blob (lib/utils/blob.py:17-50).  img: uint8 BGR [batch][H][W][3] (device);
 * pixel_means3: HOST doubles (cfg.PIXEL_MEANS, lib/mnc_config.py:20); out: fp32
 * [batch][3][out_h][out_w] with out = cv2.resize(float32(img) - means, fx=fy=scale, INTER_LINEAR).
 * out_h/out_w = round(H*scale), round(W*scale) as cv2 computes them. */
int mnc_prep_images(const unsigned char* img_bgr_hwc, int batch, int H, int W,
                    const double* pixel_means3, double scale, int out_h, int out_w,
                    float* out_nchw, void* stream);
/* Images of different sizes in one launch (im_list_to_blob, lib/utils/blob.py:17-31): image b,
 * uint8 BGR HWC of src_hw[b] = (h, w) at byte offset offsets[b] of the DEVICE buffer `packed`, is
 * prepared as mnc_prep_images does with scale scales[b] into the top-left dst_hw[b] (= its rounded
 * scaled size) of the [batch][3][out_h][out_w] blob; every other blob element is written as 0.
 * offsets, src_hw, scales, dst_hw: HOST arrays; batch <= 64. */
int mnc_prep_images_ragged(const unsigned char* packed, int batch, const long long* offsets,
                           const int* src_hw, const double* scales, const int* dst_hw,
                           const double* pixel_means3, int out_h, int out_w, float* out_nchw,
                           void* stream);

/* ---------------------------------------------------------------------------------------------
 * Result rendering (SURVEY.md section 8f, "next" row 3): _convert_pred_to_image
 * (lib/utils/vis_seg.py:101-131, called from tools/demo.py:153-158) for a batch of images.
 * boxes [batch][max_n][box_dim] (x1,y1,x2,y2[,score]; rounded half-to-even and clipped inside),
 * masks [batch][max_n][M][M], cls [batch][max_n] class ids, counts [batch] valid instances
 * (painted in list order).  inst_img / cls_img: int32 [batch][H][W] (either may be NULL); bgr:
 * optional uint8 [batch][H][W][3] = _get_voc_color_map()[cls_img][::-1] (vis_seg.py:133-148,
 * demo.py:160-164).  All device pointers. */
int mnc_paste_instances(const float* boxes, int box_dim, const float* masks, const int* cls,
                        const int* counts, int batch, int max_n, int mask_size, int H, int W,
                        float thresh, int* inst_img, int* cls_img, unsigned char* bgr,
                        void* stream);

/* The same rendering straight from the outputs of batched mask voting (mnc_vote_select +
 * mnc_mv_device), for images of different sizes in one launch: get_vis_dict (tools/demo.py:103-120)
 * then _convert_pred_to_image per image.  n_res [batch], res_score / res_class [batch][max_results],
 * result_box int32 [batch][max_results][4], result_mask [batch][max_results][M][M]; of the first
 * n_res[b] results of image b those with res_score >= vis_thresh are painted, in order, the k-th of
 * them as instance k.  img_hw int32 [batch][2] = (H_b, W_b); image b occupies pixels
 * [pix_off[b], pix_off[b] + H_b*W_b) of inst_img / cls_img (int32, either may be NULL) and of bgr
 * (uint8, 3 bytes a pixel, optional), packed without padding.  max_h / max_w: the largest H_b / W_b
 * (launch shape).  thresh: the mask binarisation threshold (cfg.BINARIZE_THRESH).  Equal, bit for
 * bit, to selecting those results and calling mnc_paste_instances image by image.  All device
 * pointers. */
int mnc_paste_voted_ragged(const int* n_res, const float* res_score, const int* res_class,
                           const int* result_box, const float* result_mask, int batch,
                           int max_results, int mask_size, const int* img_hw,
                           const long long* pix_off, int max_h, int max_w, float vis_thresh,
                           float thresh, int* inst_img, int* cls_img, unsigned char* bgr,
                           void* stream);

/* cv2.resize(mask, (bw, bh)) >= thresh for n predictions at once, as the AP^r evaluator does per
 * prediction (lib/utils/voc_eval.py:249-251).  rboxes int32 [n][4] already rounded; out is one
 * packed uint8 buffer, prediction i occupying bw_i*bh_i bytes (row-major) at offsets[i];
 * max_area = max_i bw_i*bh_i.  All device pointers. */
int mnc_binarize_masks(const int* rboxes, const float* masks, int n, int mask_size, float thresh,
                       const long long* offsets, int max_area, unsigned char* out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Sibling test graphs (SURVEY.md section 8f, "next" row 4).
 * mnc_roi_pool_nchw: ROIPoolingLayer::Forward_gpu (caffe-mnc/src/caffe/layers/
 * roi_pooling_layer.cu:17-105): fp32 NCHW feat [B][C][H][W], rois [R][5] -> out
 * [R][C][pooled_h][pooled_w], argmax (int32, same shape; may be NULL).  Empty bins give 0 / -1.
 * mnc_roi_pool_split / mnc_roi_sample_split: engine forms on the fp32 NHWC feature copy ->
 * split-bf16 rows [R][P][P][C] (ROIPooling, and ROIWarping roi_warping_layer.cu:67-107 without a
 * pool after it, as faster_rcnn_end2end/test.prototxt:479-490 uses it). */
/* _detection_forward tail (lib/caffeWrapper/TesterWrapper.py:229-234): for every RoI and class,
 * bbox_transform_inv(rois[:,1:5] / im_scale, bbox_pred[:, 4c:4c+4]) clipped to the image.
 * out [total][ncls][4]; im_scale [batch]; im_hw [batch][2] (original image size). */
int mnc_decode_class_boxes(const float* rois, int total, int rois_per_img, const float* bbox_pred,
                           int bbox_stride, int ncls, const float* im_scale, const float* im_hw,
                           float* out, void* stream);
int mnc_roi_pool_nchw(const float* feat, int C, int H, int W, const float* rois, int R,
                      int pooled_h, int pooled_w, float spatial_scale, float* out, int* argmax,
                      void* stream);
int mnc_roi_pool_split(const float* feat_nhwc, int C, int H, int W, const float* rois, int R,
                       int pooled, float spatial_scale, void* o_hi, void* o_lo, void* stream);
int mnc_roi_sample_split(const float* feat_nhwc, int C, int H, int W, const float* rois, int R,
                         int pooled, float spatial_scale, void* o_hi, void* o_lo, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MNC_B200_H_ */
