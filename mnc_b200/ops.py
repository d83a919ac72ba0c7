"""Device-tensor wrappers over the non-dense C-ABI entry points (include/mnc_b200.h).

All arguments are CUDA torch tensors; everything is launched on torch's current stream.  PyTorch is
only the allocator / stream provider here: every computation happens in libmnc_b200.so.
"""
import ctypes

import torch

from ._lib import lib, ptr, cur_stream, check, c_int, c_ll, c_float
from .dense import img_hw_arg

c_double = ctypes.c_double
lib.mnc_nms_workspace_bytes.restype = ctypes.c_longlong


def _i32(*shape, device):
    return torch.empty(shape, dtype=torch.int32, device=device)


# ----------------------------------------------------------------------------- sort / NMS
def rank_sort_desc(keys, n, problems, outer_stride, inner_stride=0, inner=1, key_stride=1,
                   valid=None):
    """-> (order int32 [problems, n], n_valid int32 [problems])."""
    dev = keys.device
    order = _i32(problems, n, device=dev)
    n_valid = _i32(problems, device=dev)
    check(lib.mnc_rank_sort_desc(ptr(keys), c_ll(outer_stride), c_ll(inner_stride), c_int(inner),
                                 c_int(key_stride), ptr(valid), c_int(n), c_int(problems),
                                 ptr(order), ptr(n_valid), cur_stream()), "mnc_rank_sort_desc")
    return order, n_valid


def topk_sort_desc(keys, n, problems, k, outer_stride, inner_stride=0, inner=1, key_stride=1,
                   valid=None):
    """The k best entries in (key desc, index asc) order.
    -> (order int32 [problems, min(k, n)], n_out int32 [problems])."""
    dev = keys.device
    kk = min(k, n)
    order = _i32(problems, kk, device=dev)
    n_out = _i32(problems, device=dev)
    check(lib.mnc_topk_sort_desc(ptr(keys), c_ll(outer_stride), c_ll(inner_stride), c_int(inner),
                                 c_int(key_stride), ptr(valid), c_int(n), c_int(problems), c_int(kk),
                                 ptr(order), c_int(kk), ptr(n_out), cur_stream()),
          "mnc_topk_sort_desc")
    return order, n_out


def gather_boxes(src, src_stride, src_outer_stride, inner, order, counts, n_out, problems):
    """-> (sorted boxes fp32 [problems, n_out, 4], counts int32 [problems])."""
    dev = src.device
    dst = torch.zeros((problems, n_out, 4), dtype=torch.float32, device=dev)
    out_counts = _i32(problems, device=dev)
    check(lib.mnc_gather_boxes(ptr(src), c_int(src_stride), c_ll(src_outer_stride), c_int(inner),
                               ptr(order), c_int(order.shape[1]), ptr(counts), c_int(n_out),
                               c_int(problems), ptr(dst), ptr(out_counts), cur_stream()),
          "mnc_gather_boxes")
    return dst, out_counts


_nms_ws = {}


def nms_sorted(boxes, counts, thresh, max_keep, per_stream=False):
    """boxes fp32 [problems, n_max, 4] score-sorted; counts int32 [problems] or None.
    per_stream: a workspace of its own for the current stream, for callers that run on several
    streams at once.  -> (keep int32 [problems, max_keep], num int32 [problems])."""
    problems, n_max, stride = boxes.shape
    dev = boxes.device
    nbytes = lib.mnc_nms_workspace_bytes(c_int(n_max), c_int(problems))
    key = (dev, nbytes) + ((torch.cuda.current_stream(dev).cuda_stream,) if per_stream else ())
    ws = _nms_ws.get(key)
    if ws is None:
        # one workspace per size, kept: a captured CUDA graph (MNCEngine.detect_graphed) holds the
        # address of the workspace it was captured with and replays into it
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        _nms_ws[key] = ws
    mk = max_keep if max_keep > 0 else n_max
    keep = _i32(problems, mk, device=dev)
    num = _i32(problems, device=dev)
    check(lib.mnc_nms_sorted(ptr(boxes), c_int(stride), c_ll(n_max * stride), ptr(counts),
                             c_int(n_max), c_int(problems), c_float(thresh), c_int(mk), ptr(ws),
                             ptr(keep), c_int(mk), ptr(num), cur_stream()), "mnc_nms_sorted",
          launches=lib.mnc_nms_sorted_launches(c_int(n_max), c_int(mk)))
    return keep, num


DEFAULT_NMS_MODE = 2


def nms_set_lazy(mode):
    """A/B and cross-check switch of the capped NMS mnc_nms_sorted picks when max_keep << n:
    3 = thread-block cluster, 256-candidate rounds; 2 = cluster, 64-candidate rounds; 1 = one CTA
    per problem; 0 / False = always the suppression-matrix pair (nms_mask + nms_scan); True = the
    library default.  Returns the previous mode (int)."""
    mode = DEFAULT_NMS_MODE if mode is True else (0 if mode is False else int(mode))
    return int(lib.mnc_nms_set_lazy(c_int(mode)))


# ----------------------------------------------------------------------------- proposal pieces
def generate_anchors():
    import numpy as np
    out = np.zeros((9, 4), dtype=np.float32)
    check(lib.mnc_generate_anchors(ptr(out)), "mnc_generate_anchors")
    return out


def rpn_decode(cls, bbox, im_info, batch, H, W, layout, apply_softmax, feat_stride=16,
               min_size=16.0, img_hw=None, level=4):
    """layout 'nchw': cls (B,18,H,W), bbox (B,36,H,W); 'nhwc': one buffer (B,H,W,Cpad) where
    channels [0,18) are cls and [18,54) bbox (then `bbox` is ignored).  img_hw: image sizes of a
    mixed-size batch (device int32 (B, 2), input resolution; the map is `level` pools below it):
    anchors outside their image are invalid."""
    dev = cls.device
    total = H * W * 9
    proposals = torch.empty((batch, total, 4), dtype=torch.float32, device=dev)
    scores = torch.empty((batch, total), dtype=torch.float32, device=dev)
    valid = torch.empty((batch, total), dtype=torch.uint8, device=dev)
    if layout == "nchw":
        ci, cc, cp = 18 * H * W, H * W, 1
        bi, bc, bp = 36 * H * W, H * W, 1
        bptr = ptr(bbox)
    else:
        cpad = cls.shape[-1]
        ci, cc, cp = H * W * cpad, 1, cpad
        bi, bc, bp = ci, cc, cp
        bptr = ctypes.c_void_p(cls.data_ptr() + 18 * 4)
    args = (ptr(cls), c_ll(ci), c_ll(cc), c_ll(cp), bptr, c_ll(bi), c_ll(bc), c_ll(bp), ptr(im_info),
            c_int(batch), c_int(H), c_int(W), c_int(feat_stride), c_float(min_size),
            c_int(int(apply_softmax)), ptr(proposals), ptr(scores), ptr(valid))
    if img_hw is None:
        check(lib.mnc_rpn_decode(*args, cur_stream()), "mnc_rpn_decode")
    else:
        check(lib.mnc_rpn_decode2(*args, ptr(img_hw_arg(img_hw, batch)), c_int(level), cur_stream()),
              "mnc_rpn_decode2")
    return proposals, scores, valid


def write_rois(sorted_boxes, keep, num_keep, max_rois, batch_index_mode):
    batch, n_sorted, _ = sorted_boxes.shape
    dev = sorted_boxes.device
    rois = torch.empty((batch, max_rois, 5), dtype=torch.float32, device=dev)
    counts = _i32(batch, device=dev)
    check(lib.mnc_write_rois(ptr(sorted_boxes), c_int(n_sorted), ptr(keep), c_int(keep.shape[1]),
                             ptr(num_keep), c_int(max_rois), c_int(batch),
                             c_int(int(batch_index_mode)), ptr(rois), ptr(counts), cur_stream()),
          "mnc_write_rois")
    return rois, counts


def proposals_from_rpn(cls, bbox, im_info, batch, H, W, layout, apply_softmax, pre_nms_top_n=6000,
                       post_nms_top_n=300, nms_thresh=0.7, min_size=16.0, batch_index_mode=True,
                       return_intermediate=False, img_hw=None, level=4):
    """Whole ProposalLayer.forward on device (lib/pylayer/proposal_layer.py:52-175).  img_hw /
    level: image sizes of a mixed-size batch (rpn_decode)."""
    proposals, scores, valid = rpn_decode(cls, bbox, im_info, batch, H, W, layout, apply_softmax,
                                          min_size=min_size, img_hw=img_hw, level=level)
    total = H * W * 9
    n_sorted = min(pre_nms_top_n, total) if pre_nms_top_n > 0 else total
    if 8 * (1 << max(n_sorted - 1, 1).bit_length()) + 4 * total <= 200 * 1024:
        order, n_valid = topk_sort_desc(scores, total, batch, n_sorted, outer_stride=total, valid=valid)
    else:   # beyond the select kernel's shared-memory budget: sort everything
        order, n_valid = rank_sort_desc(scores, total, batch, outer_stride=total, valid=valid)
    sorted_boxes, counts = gather_boxes(proposals, 4, total * 4, 1, order, n_valid, n_sorted, batch)
    keep, num = nms_sorted(sorted_boxes, counts, nms_thresh, post_nms_top_n)
    rois, roi_counts = write_rois(sorted_boxes, keep, num, post_nms_top_n, batch_index_mode)
    if return_intermediate:
        return rois, roi_counts, dict(proposals=proposals, scores=scores, valid=valid, order=order,
                                      n_valid=n_valid, sorted_boxes=sorted_boxes, counts=counts,
                                      keep=keep, num=num)
    return rois, roi_counts


def stage_bridge(rois, bbox_pred, seg_cls_prob, im_info, rois_per_img):
    """rois [T,5], bbox_pred [T,>=84] (row stride = bbox_pred.stride(0)), seg_cls_prob [T,21]."""
    total = rois.shape[0]
    out = torch.empty_like(rois)
    check(lib.mnc_stage_bridge(ptr(rois), ptr(bbox_pred), c_int(bbox_pred.stride(0)),
                               ptr(seg_cls_prob), c_int(seg_cls_prob.stride(0)),
                               c_int(seg_cls_prob.shape[1]), ptr(im_info), c_int(rois_per_img),
                               c_int(total), ptr(out), cur_stream()), "mnc_stage_bridge")
    return out


def softmax_rows(x, cols=None, out=None):
    rows = x.shape[0]
    cols = cols or x.shape[1]
    if out is None:
        out = torch.empty((rows, cols), dtype=torch.float32, device=x.device)
    check(lib.mnc_softmax_rows(ptr(x), c_int(x.stride(0)), c_int(rows), c_int(cols), ptr(out),
                               c_int(out.stride(0)), cur_stream()), "mnc_softmax_rows")
    return out


def unscale_clip(rois, rois_per_img, im_scale, im_hw):
    total = rois.shape[0]
    boxes = torch.empty((total, 4), dtype=torch.float32, device=rois.device)
    check(lib.mnc_unscale_clip(ptr(rois), c_int(total), c_int(rois_per_img), ptr(im_scale),
                               ptr(im_hw), ptr(boxes), cur_stream()), "mnc_unscale_clip")
    return boxes


def record_layout(B, n, msz=441, ncls=21):
    """Offsets (in floats) of the sections of the per-step output record and its length."""
    o_boxes = (B + 3) // 4 * 4
    o_scores = o_boxes + B * 2 * n * 4
    o_masks = o_scores + B * 2 * n * ncls
    return o_boxes, o_scores, o_masks, o_masks + B * 2 * n * msz


def record_views(rec, B, n, msz=441, ncls=21):
    ob, os_, om, end = record_layout(B, n, msz, ncls)
    side = int(round(msz ** 0.5))
    return (rec[:B], rec[ob:os_].view(B, 2 * n, 4), rec[os_:om].view(B, 2 * n, ncls),
            rec[om:end].view(B, 2 * n, 1, side, side))


def vote_record_layout(B, R, M=21):
    """Offsets (in 4-byte elements) of the sections of a mask-voting result record and its length:
    n_res[B] | overflow | class[B][R] | score[B][R] | box[B][R][4] | mask[B][R][M*M].  Integer
    sections hold int32 bit patterns; every section starts on a 16-byte boundary."""
    up = lambda v: (v + 3) // 4 * 4
    o_over = up(B)
    o_class = up(o_over + 1)
    o_score = o_class + up(B * R)
    o_box = o_score + up(B * R)
    o_mask = o_box + B * R * 4
    return o_over, o_class, o_score, o_box, o_mask, o_mask + B * R * M * M


def vote_record_views(rec, B, R, M=21):
    """Views of a record of `vote_record_layout(B, R, M)` elements (4-byte dtype; device or host):
    the keys of the dict `mask_voting` returns that the record holds, each in its dtype."""
    oo, oc, os_, ob, om, end = vote_record_layout(B, R, M)
    i32, f32 = rec[:end].view(torch.int32), rec[:end].view(torch.float32)
    return dict(n_res=i32[:B], overflow=i32[oo:oo + 1], res_class=i32[oc:oc + B * R].view(B, R),
                res_score=f32[os_:os_ + B * R].view(B, R), result_box=i32[ob:om].view(B, R, 4),
                result_mask=f32[om:end].view(B, R, 1, M, M))


def detect_tail(o, B, n, im_scale, im_hw, rec, valid):
    """im_detect tail into the record buffer `rec` (fp32, record_layout(B, n)[3] floats) and
    `valid` (uint8 [B, 2n]).  Returns (counts, boxes, scores, masks) views of rec."""
    msz = o["mask_proposal"].shape[-1] * o["mask_proposal"].shape[-2]
    ncls = o["seg_cls_prob"].shape[-1]
    counts, boxes, scores, masks = record_views(rec, B, n, msz, ncls)
    check(lib.mnc_detect_tail(ptr(o["rois"]), ptr(o["rois_ext"]), ptr(o["mask_proposal"]),
                              ptr(o["mask_proposal_ext"]), ptr(o["seg_cls_prob"]),
                              ptr(o["seg_cls_prob_ext"]), ptr(o["roi_counts"]), ptr(im_scale),
                              ptr(im_hw), c_int(B), c_int(n), c_int(msz), c_int(ncls), ptr(counts),
                              ptr(boxes), ptr(scores), ptr(masks), ptr(valid), cur_stream()),
          "mnc_detect_tail")
    return counts, boxes, scores, masks


def decode_class_boxes(rois, bbox_pred, rois_per_img, im_scale, im_hw, ncls=21):
    """-> (R, ncls*4) fp32: per-class decoded boxes in original-image coordinates, clipped."""
    R = rois.shape[0]
    out = torch.empty((R, ncls * 4), dtype=torch.float32, device=rois.device)
    check(lib.mnc_decode_class_boxes(ptr(rois), c_int(R), c_int(rois_per_img), ptr(bbox_pred),
                                     c_int(bbox_pred.stride(0)), c_int(ncls), ptr(im_scale),
                                     ptr(im_hw), ptr(out), cur_stream()), "mnc_decode_class_boxes")
    return out


# ----------------------------------------------------------------------------- RoI / mask layers
def roi_warp_nchw(feat, rois, pooled_h, pooled_w, spatial_scale=0.0625, out=None):
    B, C, H, W = feat.shape
    R = rois.shape[0]
    if out is None:
        out = torch.empty((R, C, pooled_h, pooled_w), dtype=torch.float32, device=feat.device)
    check(lib.mnc_roi_warp_nchw(ptr(feat), c_int(C), c_int(H), c_int(W), ptr(rois), c_int(R),
                                c_int(pooled_h), c_int(pooled_w), c_float(spatial_scale), ptr(out),
                                cur_stream()), "mnc_roi_warp_nchw")
    return out


def mask_resize_nchw(x, out_h, out_w):
    N, C, ih, iw = x.shape
    out = torch.empty((N, C, out_h, out_w), dtype=torch.float32, device=x.device)
    check(lib.mnc_mask_resize_nchw(ptr(x), c_int(N), c_int(C), c_int(ih), c_int(iw), c_int(out_h),
                                   c_int(out_w), ptr(out), cur_stream()), "mnc_mask_resize_nchw")
    return out


def mask_pool_nchw(feat, mask, out=None):
    N, C, H, W = feat.shape
    if mask.shape != (N, 1, H, W):
        raise ValueError("MaskPooling: mask must be (N,1,H,W) matching feat "
                         "(mask_pooling_layer.cpp:20-29)")
    if out is None:
        out = torch.empty_like(feat)
    check(lib.mnc_mask_pool_nchw(ptr(feat), ptr(mask), c_int(N), c_int(C), c_int(H), c_int(W),
                                 ptr(out), cur_stream()), "mnc_mask_pool_nchw")
    return out


def roi_warp_split(feat, C, H, W, rois, sub, out14, out7, spatial_scale=0.0625, img_hw=None, level=4):
    """feat fp32 NHWC [B,H,W,C]; rois [R,5]; out14 split [2,R,14,14,C]; out7 split [2,R,7,7,C].
    img_hw / level: image sizes of a mixed-size batch; samples are bounded by the RoI's image."""
    R = rois.shape[0]
    assert feat.dtype == torch.float32
    args = (ptr(feat), c_int(C), c_int(H), c_int(W), ptr(rois), c_int(R), c_int(sub),
            c_float(spatial_scale), ptr(out14[0]), ptr(out14[1]), ptr(out7[0]), ptr(out7[1]))
    if img_hw is None:
        check(lib.mnc_roi_warp_split(*args, cur_stream()), "mnc_roi_warp_split")
    else:
        check(lib.mnc_roi_warp_split2(*args, ptr(img_hw_arg(img_hw, feat.shape[0])), c_int(level),
                                      cur_stream()), "mnc_roi_warp_split2")


def roi_warp_tri(feat, C, H, W, rois, sub, out14, out7, exp, spatial_scale=0.0625, img_hw=None,
                 level=4):
    """roi_warp_split with tri-plane outputs (mnc_b200.dense.Tri) written with exponent `exp`."""
    R = rois.shape[0]
    assert feat.dtype == torch.float32
    out14.exp = out7.exp = int(exp)
    args = (ptr(feat), c_int(C), c_int(H), c_int(W), ptr(rois), c_int(R), c_int(sub),
            c_float(spatial_scale), c_float(2.0 ** exp), ptr(out14.h), ptr(out14.l), ptr(out14.c),
            ptr(out7.h), ptr(out7.l), ptr(out7.c))
    if img_hw is None:
        check(lib.mnc_roi_warp_tri(*args, cur_stream()), "mnc_roi_warp_tri")
    else:
        check(lib.mnc_roi_warp_tri2(*args, ptr(img_hw_arg(img_hw, feat.shape[0])), c_int(level),
                                    cur_stream()), "mnc_roi_warp_tri2")


def mask_pool_tri(feat14, mask14, R, C, out7):
    """MaskPooling + 2x2 max pool on tri-plane features; the output takes the input's exponent."""
    out7.exp = feat14.exp
    check(lib.mnc_mask_pool_tri(ptr(feat14.h), ptr(feat14.l), ptr(mask14), c_int(R), c_int(C),
                                ptr(out7.h), ptr(out7.l), ptr(out7.c), cur_stream()), "mnc_mask_pool_tri")


def sigmoid_mask_resize(logits, R, mask_size=21, out_size=14):
    dev = logits.device
    mp = torch.empty((R, 1, mask_size, mask_size), dtype=torch.float32, device=dev)
    mr = torch.empty((R, 1, out_size, out_size), dtype=torch.float32, device=dev)
    check(lib.mnc_sigmoid_mask_resize(ptr(logits), c_int(logits.stride(0)), c_int(R),
                                      c_int(mask_size), c_int(out_size), ptr(mp), ptr(mr),
                                      cur_stream()), "mnc_sigmoid_mask_resize")
    return mp, mr


def mask_pool_split(feat14, mask14, R, C, out7):
    check(lib.mnc_mask_pool_split(ptr(feat14[0]), ptr(feat14[1]), ptr(mask14), c_int(R), c_int(C),
                                  ptr(out7[0]), ptr(out7[1]), cur_stream()), "mnc_mask_pool_split")


def roi_pool_nchw(feat, rois, pooled_h, pooled_w, spatial_scale=0.0625, out=None, argmax=None):
    """ROIPoolingLayer forward (roi_pooling_layer.cu:17-105) on fp32 NCHW device tensors."""
    B, C, H, W = feat.shape
    R = rois.shape[0]
    if out is None:
        out = torch.empty((R, C, pooled_h, pooled_w), dtype=torch.float32, device=feat.device)
    check(lib.mnc_roi_pool_nchw(ptr(feat), c_int(C), c_int(H), c_int(W), ptr(rois), c_int(R),
                                c_int(pooled_h), c_int(pooled_w), c_float(spatial_scale), ptr(out),
                                ptr(argmax), cur_stream()), "mnc_roi_pool_nchw")
    return out


def roi_pool_split(feat, C, H, W, rois, pooled, out, spatial_scale=0.0625):
    """feat fp32 NHWC [B,H,W,C]; rois [R,5]; out split [2,R,P,P,C] (ROIPooling)."""
    check(lib.mnc_roi_pool_split(ptr(feat), c_int(C), c_int(H), c_int(W), ptr(rois),
                                 c_int(rois.shape[0]), c_int(pooled), c_float(spatial_scale),
                                 ptr(out[0]), ptr(out[1]), cur_stream()), "mnc_roi_pool_split")


def roi_sample_split(feat, C, H, W, rois, pooled, out, spatial_scale=0.0625):
    """feat fp32 NHWC [B,H,W,C]; rois [R,5]; out split [2,R,P,P,C] (ROIWarping, no pool after)."""
    check(lib.mnc_roi_sample_split(ptr(feat), c_int(C), c_int(H), c_int(W), ptr(rois),
                                   c_int(rois.shape[0]), c_int(pooled), c_float(spatial_scale),
                                   ptr(out[0]), ptr(out[1]), cur_stream()), "mnc_roi_sample_split")


# ----------------------------------------------------------------------------- mask voting
class VotingOverflow(RuntimeError):
    pass


def default_vote_cap(max_per_image):
    """Result slots per image a voting call starts with (more only after an overflow)."""
    return max(128, max_per_image + 28)


def mask_voting(boxes, masks, scores, im_hw, max_per_image=100, nms_thresh=0.3, iou_thresh=0.5,
                max_results=128, box_valid=None, out=None):
    """Batched device pipeline of gpu_mask_voting (lib/transform/mask_transform.py:213-286).
    boxes [B,nb,4] fp32, masks [B,nb,1,M,M] fp32, scores [B,nb,ncls] fp32, im_hw [B,2] int32.
    box_valid: optional uint8 [B,nb]; rows with 0 are padding and take no part.
    out: optional `vote_record_views(rec, B, max_results, M)`; the results are written there (one
    record, one copy to the host) instead of into fresh tensors.
    Returns dict of device tensors: n_res [B], class_bar [B,ncls-1], res_score [B,max_results],
    res_class, result_mask [B,max_results,1,M,M], result_box [B,max_results,4] int32, plus the
    candidate lists."""
    B, nb, ncls = scores.shape
    M = masks.shape[-1]
    dev = boxes.device
    nprob = B * (ncls - 1)
    # per-class score sort: problem p = (img, c-1); keys at scores[img, :, c]
    valid_p = None
    if box_valid is not None:
        valid_p = box_valid.view(B, 1, nb).expand(B, ncls - 1, nb).contiguous()
    order, n_valid = rank_sort_desc(scores[:, :, 1:], nb, nprob, outer_stride=nb * ncls,
                                    inner_stride=1, inner=ncls - 1, key_stride=ncls, valid=valid_p)
    sorted_boxes, counts = gather_boxes(boxes, 4, nb * 4, ncls - 1, order, n_valid, nb, nprob)
    # two pipelined batches vote at once on two streams (Detector.im_segment_stream)
    keep, num = nms_sorted(sorted_boxes, counts, nms_thresh, min(max_per_image, nb), per_stream=True)
    res_idx = _i32(B, max_results, device=dev)
    class_bar = _i32(B, ncls - 1, device=dev)
    if out is None:
        res_cls = _i32(B, max_results, device=dev)
        res_score = torch.zeros((B, max_results), dtype=torch.float32, device=dev)
        n_res = _i32(B, device=dev)
        overflow = torch.zeros(1, dtype=torch.int32, device=dev)
        out_mask = torch.zeros((B, max_results, 1, M, M), dtype=torch.float32, device=dev)
        out_box = torch.zeros((B, max_results, 4), dtype=torch.int32, device=dev)
    else:
        if out["res_score"].shape != (B, max_results) or out["result_mask"].shape[-1] != M:
            raise ValueError("mask_voting: out= views of another shape")
        res_cls, res_score, n_res, overflow = out["res_class"], out["res_score"], out["n_res"], out["overflow"]
        out_mask, out_box = out["result_mask"], out["result_box"]
        for t in (res_score, overflow, out_mask, out_box):
            t.zero_()
    check(lib.mnc_vote_select(ptr(scores), c_int(nb), c_int(ncls), ptr(order), ptr(keep),
                              c_int(keep.shape[1]), ptr(num), c_int(max_per_image),
                              c_int(max_results), c_int(B), ptr(res_idx), ptr(res_cls),
                              ptr(res_score), ptr(n_res), ptr(class_bar), ptr(overflow),
                              cur_stream()), "mnc_vote_select")
    cand_inds = _i32(B, max_results, nb, device=dev)
    cand_w = torch.empty((B, max_results, nb), dtype=torch.float32, device=dev)   # lists only; gaps unread
    cand_begin = _i32(B, max_results, device=dev)
    cand_end = _i32(B, max_results, device=dev)
    check(lib.mnc_vote_candidates(ptr(boxes), ptr(scores), ptr(box_valid), c_int(nb), c_int(ncls),
                                  ptr(res_idx),
                                  ptr(res_cls), ptr(n_res), c_int(max_results), c_int(B),
                                  c_double(iou_thresh), ptr(cand_inds), ptr(cand_w),
                                  ptr(cand_begin), ptr(cand_end), cur_stream()),
          "mnc_vote_candidates")
    bbox_ws = _i32(B * max_results * 4 + B, device=dev)   # tight boxes + per-image range flag
    check(lib.mnc_mv_device(ptr(boxes), ptr(masks), c_int(nb), c_int(4), c_int(M), ptr(cand_inds),
                            ptr(cand_w), c_ll(max_results * nb), ptr(cand_begin), ptr(cand_end),
                            ptr(n_res), c_int(max_results), c_int(B), ptr(im_hw), ptr(bbox_ws),
                            ptr(out_mask), ptr(out_box), cur_stream()), "mnc_mv_device",
          launches=lib.mnc_mv_device_launches())
    return dict(n_res=n_res, class_bar=class_bar, res_score=res_score, res_class=res_cls,
                res_box_idx=res_idx, result_mask=out_mask, result_box=out_box,
                cand_inds=cand_inds, cand_weights=cand_w, cand_begin=cand_begin, cand_end=cand_end,
                overflow=overflow, order=order, keep=keep, num_keep=num)


def mv_set_two_pass(on):
    """A/B and cross-check switch of mnc_mv_device: False = one full sweep of each result's region
    instead of the coarse pass + exact border pass.  Returns the previous setting."""
    return bool(lib.mnc_mv_set_two_pass(c_int(1 if on else 0)))


def mask_voting_checked(boxes, masks, scores, im_hw, max_per_image=100, box_valid=None, **kw):
    """mask_voting that never truncates: the reference keeps EVERY kept row whose score ties the
    global threshold (mask_transform.py:258), so when more rows tie than `max_results` has slots
    the device reports it and the call is repeated with room (one host read of a 4-byte flag)."""
    cap = kw.pop("max_results", default_vote_cap(max_per_image))
    nb = boxes.shape[1]
    while True:
        r = mask_voting(boxes, masks, scores, im_hw, max_per_image=max_per_image, max_results=cap,
                        box_valid=box_valid, **kw)
        if int(r["overflow"].item()) == 0:
            return r
        if cap >= nb * (scores.shape[2] - 1):
            raise VotingOverflow("mask voting overflow at max_results = %d" % cap)
        cap = min(2 * cap, nb * (scores.shape[2] - 1))


# ----------------------------------------------------------------------------- input preparation
PIXEL_MEANS = (102.9801, 115.9465, 122.7717)   # cfg.PIXEL_MEANS, lib/mnc_config.py:20


def im_scale_for(shape, target_size=600, max_size=1000):
    """Scale rule of prep_im_for_blob (lib/utils/blob.py:41-46)."""
    import numpy as np
    im_size_min = min(shape[0], shape[1])
    im_size_max = max(shape[0], shape[1])
    im_scale = float(target_size) / float(im_size_min)
    if np.round(im_scale * im_size_max) > max_size:
        im_scale = float(max_size) / float(im_size_max)
    return im_scale


def prep_images(images_u8, scale, out=None, pixel_means=PIXEL_MEANS):
    """images_u8: uint8 CUDA tensor [B,H,W,3] (BGR).  -> fp32 [B,3,round(H*s),round(W*s)]."""
    import numpy as np
    B, H, W, _ = images_u8.shape
    out_h, out_w = int(np.rint(H * scale)), int(np.rint(W * scale))
    if out is None:
        out = torch.empty((B, 3, out_h, out_w), dtype=torch.float32, device=images_u8.device)
    means = (ctypes.c_double * 3)(*pixel_means)
    check(lib.mnc_prep_images(ptr(images_u8), c_int(B), c_int(H), c_int(W), means,
                              ctypes.c_double(scale), c_int(out_h), c_int(out_w), ptr(out),
                              cur_stream()), "mnc_prep_images")
    return out


def blob_size_for(shape, scale):
    """(rows, cols) of an image of `shape` (H, W, ...) in the blob at `scale` (cv2's rounding)."""
    import numpy as np
    return int(np.rint(shape[0] * scale)), int(np.rint(shape[1] * scale))


def prep_images_ragged(packed_u8, offsets, src_hw, scales, out_h, out_w, out=None,
                       pixel_means=PIXEL_MEANS):
    """Images of different sizes in one launch (`im_list_to_blob` of `prep_im_for_blob` outputs):
    packed_u8 a uint8 CUDA tensor holding image b (BGR HWC, src_hw[b]) at byte offsets[b]; image b
    is prepared with scales[b] into the top-left corner of a zero-padded fp32 (B,3,out_h,out_w)
    blob.  offsets / src_hw / scales: host sequences.  -> (blob, dst_hw int32 numpy (B, 2))."""
    import numpy as np
    B = len(scales)
    dst = np.array([blob_size_for(hw, s) for hw, s in zip(src_hw, scales)], dtype=np.int32).reshape(B, 2)
    if out is None:
        out = torch.empty((B, 3, out_h, out_w), dtype=torch.float32, device=packed_u8.device)
    off = np.ascontiguousarray(offsets, dtype=np.int64)
    shw = np.ascontiguousarray(src_hw, dtype=np.int32).reshape(B, 2)
    sc = np.ascontiguousarray(scales, dtype=np.float64)
    if (shw.astype(np.int64).prod(axis=1) * 3 + off > packed_u8.numel()).any():
        raise ValueError("prep_images_ragged: an image lies outside the packed buffer")
    means = (ctypes.c_double * 3)(*pixel_means)
    check(lib.mnc_prep_images_ragged(ptr(packed_u8), c_int(B), ptr(off), ptr(shw), ptr(sc), ptr(dst),
                                     means, c_int(out_h), c_int(out_w), ptr(out), cur_stream()),
          "mnc_prep_images_ragged")
    return out, dst


# ----------------------------------------------------------------------------- result rendering
def paste_instances(boxes, masks, cls, counts, H, W, thresh=0.4, want_bgr=False):
    """Batched `_convert_pred_to_image` (lib/utils/vis_seg.py:101-131).  boxes [B,n,>=4] fp32,
    masks [B,n,(1,)M,M] fp32, cls [B,n] int32, counts [B] int32 -- device tensors, instances in
    painting order.  -> inst_img, cls_img int32 [B,H,W] (+ uint8 BGR [B,H,W,3] colour image)."""
    B, n, box_dim = boxes.shape
    M = masks.shape[-1]
    dev = boxes.device
    boxes = boxes.contiguous().float()
    masks = masks.contiguous().float()
    cls = cls.contiguous().to(torch.int32)
    counts = counts.contiguous().to(torch.int32)
    inst = torch.empty((B, H, W), dtype=torch.int32, device=dev)
    clsi = torch.empty((B, H, W), dtype=torch.int32, device=dev)
    bgr = torch.empty((B, H, W, 3), dtype=torch.uint8, device=dev) if want_bgr else None
    check(lib.mnc_paste_instances(ptr(boxes), c_int(box_dim), ptr(masks), ptr(cls), ptr(counts),
                                  c_int(B), c_int(n), c_int(M), c_int(H), c_int(W), c_float(thresh),
                                  ptr(inst), ptr(clsi), ptr(bgr), cur_stream()),
          "mnc_paste_instances")
    return (inst, clsi, bgr) if want_bgr else (inst, clsi)


def paste_voted_ragged(vote, img_hw, pix_off, max_hw, inst, cls, bgr, vis_thresh=0.5, thresh=0.4):
    """`select_for_display` + `paste_instances` for images of different sizes in one launch,
    straight from the outputs of `mask_voting` (its dict, or `vote_record_views` of its record).
    img_hw: device int32 (B, 2) image sizes; pix_off: device int64 (B,) first pixel of each image
    in the packed outputs; max_hw: host (max H, max W).  inst, cls int32 and bgr uint8 device
    tensors of P, P and 3P elements, P = sum of H_b * W_b (inst / cls may be None): image b is
    written to pixels [pix_off[b], pix_off[b] + H_b * W_b)."""
    score = vote["res_score"]
    B, R = score.shape
    M = vote["result_mask"].shape[-1]
    check(lib.mnc_paste_voted_ragged(ptr(vote["n_res"]), ptr(score), ptr(vote["res_class"]),
                                     ptr(vote["result_box"]), ptr(vote["result_mask"]), c_int(B),
                                     c_int(R), c_int(M), ptr(img_hw), ptr(pix_off),
                                     c_int(int(max_hw[0])), c_int(int(max_hw[1])),
                                     c_float(vis_thresh), c_float(thresh), ptr(inst), ptr(cls),
                                     ptr(bgr), cur_stream()), "mnc_paste_voted_ragged")


def select_for_display(vote, vis_thresh=0.5):
    """`get_vis_dict` (tools/demo.py:103-120) on the device: keep voted results with
    score >= vis_thresh, order preserved (results are class-major, as the reference's loops
    visit them).  vote: the dict `mask_voting` returns.  -> boxes [B,R,4] fp32, masks, cls, counts."""
    n_res, score = vote["n_res"], vote["res_score"]
    B, R = score.shape
    live = (torch.arange(R, device=score.device)[None, :] < n_res[:, None]) & (score >= vis_thresh)
    perm = torch.sort((~live).to(torch.int8), dim=1, stable=True).indices
    boxes = torch.gather(vote["result_box"].float(), 1, perm[:, :, None].expand(B, R, 4))
    M = vote["result_mask"].shape[-1]
    masks = torch.gather(vote["result_mask"].view(B, R, M * M), 1, perm[:, :, None].expand(B, R, M * M))
    cls = torch.gather(vote["res_class"], 1, perm)
    return boxes, masks.view(B, R, M, M), cls, live.sum(dim=1).to(torch.int32)


def binarize_masks(rboxes, masks, thresh=0.4):
    """cv2.resize(mask, box size) >= thresh for every prediction (lib/utils/voc_eval.py:249-251).
    rboxes int32 [n,4] (rounded boxes), masks fp32 [n,M,M], both on the device.
    -> (packed uint8 device tensor, offsets int64 host array of n+1 entries)."""
    import numpy as np
    n = rboxes.shape[0]
    M = masks.shape[-1]
    rb = rboxes.contiguous().to(torch.int32)
    hb = rb.cpu().numpy().astype(np.int64)
    areas = np.maximum(hb[:, 2] - hb[:, 0] + 1, 0) * np.maximum(hb[:, 3] - hb[:, 1] + 1, 0)
    offsets = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(areas, out=offsets[1:])
    out = torch.empty((max(int(offsets[-1]), 1),), dtype=torch.uint8, device=rboxes.device)
    d_off = torch.from_numpy(offsets[:-1].copy()).to(rboxes.device)
    check(lib.mnc_binarize_masks(ptr(rb), ptr(masks.contiguous().float()), c_int(n), c_int(M),
                                 c_float(thresh), ptr(d_off), c_int(int(areas.max()) if n else 0),
                                 ptr(out), cur_stream()), "mnc_binarize_masks")
    return out, offsets
