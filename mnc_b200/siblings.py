"""The two sibling test graphs of the reference that run on the same kernels as the 5-stage net
(SURVEY.md section 8f row 4):

* `FasterRCNNEngine` -- models/VGG16/faster_rcnn_end2end/test.prototxt: trunk, RPN, ProposalLayer,
  ROIWarping 7x7 (:479-490), fc6/fc7 (Dropout = identity in TEST phase), cls_score + Softmax,
  bbox_pred.  Caller: TesterWrapper._detection_forward (lib/caffeWrapper/TesterWrapper.py:215-237).
* `CFMEngine` -- models/VGG16/cfm/test.prototxt: trunk on an image pyramid; rois (with pyramid level)
  and 14x14 binary masks are INPUTS; ROIPooling 7x7 -> fc6/fc7; ROIPooling 14x14 -> MaskPooling ->
  2x2 max pool -> fc6_mask/fc7_mask; fc6_maskest/mask_pred/Sigmoid on the un-masked 14x14 feature;
  Concat -> cls_score / seg_cls_score / bbox_pred.  Caller: TesterWrapper.cfm_network_forward
  (:336-414).

Both reuse MNCEngine's trunk, implicit-GEMM inner products and buffers; the only new device code
is ROIPooling and the pool-free ROIWarping (csrc/roi_ops.cu).
"""
import torch

from . import ops
from .engine import MNCEngine, ROIS_PER_IMAGE, NUM_CLASSES, MASK_SIZE


class FasterRCNNEngine(MNCEngine):
    DEFAULT_PRECISION = "bf16x3"   # RoI producers of this graph write split-bf16 features

    def forward(self, data, im_info, keep_intermediate=False, extents=None):
        """-> rois (B*300,5), roi_counts (B,), cls_prob (B*300,21), bbox_pred (B*300,84)."""
        if extents is not None:
            raise NotImplementedError("mixed-size batches: the 5-stage MNCEngine only")
        B = data.shape[0]
        conv5_3, H5, W5, c5f, rois, roi_counts, res, _ = self.rpn_rois(data, im_info, keep_intermediate)
        c5, fc = self.c5, self.fc
        R = B * ROIS_PER_IMAGE
        pool5 = self._split_buf("box7", R, 7, 7, c5)
        ops.roi_sample_split(c5f, c5, H5, W5, rois, 7, pool5)
        h6 = self._split_buf("h6", R, fc)
        h7 = self._split_buf("h7", R, fc)
        self._linear(pool5, R, 49 * c5, self.fc6[0], fc, self.fc6[1], True, out=h6, key="fc6")
        self._linear(h6, R, fc, self.fc7[0], fc, self.fc7[1], True, out=h7, key="fc7")
        heads = torch.empty((R, 128), dtype=torch.float32, device=self.device)
        self._linear(h7, R, fc, self.cls_heads[0], 105, self.cls_heads[1], False, out_f32=heads,
                     out_stride=128, key="cls")
        out = dict(rois=rois, roi_counts=roi_counts, cls_prob=ops.softmax_rows(heads[:, 0:21], 21),
                   bbox_pred=heads[:, 21:105])
        if keep_intermediate:
            out["_pool5"] = pool5.clone()
            out["_conv5_3"] = conv5_3.clone()
            out["_proposal"] = res[2]
        return out

    def detect(self, data, im_info, im_hw, im_scale, extents=None):
        """forward + `_detection_forward` tail (TesterWrapper.py:226-237): per RoI 21 class scores
        and 21 decoded, clipped boxes.  -> scores (B,300,21), pred_boxes (B,300,84), valid."""
        if extents is not None:
            raise NotImplementedError("mixed-size batches: the 5-stage MNCEngine only")
        B = data.shape[0]
        o = self.forward(data, im_info)
        n = ROIS_PER_IMAGE
        pred = ops.decode_class_boxes(o["rois"], o["bbox_pred"], n, im_scale, im_hw)
        ar = torch.arange(n, device=self.device, dtype=torch.int32).view(1, n)
        valid = (ar < o["roi_counts"].view(B, 1)).to(torch.uint8)
        return o["cls_prob"].view(B, n, NUM_CLASSES), pred.view(B, n, 4 * NUM_CLASSES), valid, o


class CFMEngine(MNCEngine):
    DEFAULT_PRECISION = "bf16x3"

    def forward(self, data, rois, masks, keep_intermediate=False, extents=None):
        """data fp32 (S,3,H,W) image pyramid; rois fp32 (R,5) [level,x1,y1,x2,y2] in the level's
        scaled coordinates; masks fp32 (R,1,14,14).  -> mask_prob (R,1,21,21), seg_cls_prob,
        cls_prob (R,21), bbox_pred (R,84)."""
        if extents is not None:
            raise NotImplementedError("mixed-size batches: the 5-stage MNCEngine only")
        S = data.shape[0]
        R = rois.shape[0]
        conv5_3, H5, W5 = self.trunk(data)
        c5f = self.conv5_f32(conv5_3, S, H5, W5)
        c5, fc, me = self.c5, self.fc, self.me
        rois = rois.contiguous().float()
        box7 = self._split_buf("box7", R, 7, 7, c5)
        ops.roi_pool_split(c5f, c5, H5, W5, rois, 7, box7)
        feat14 = self._split_buf("feat14", R, 14, 14, c5)
        ops.roi_pool_split(c5f, c5, H5, W5, rois, 14, feat14)
        join = self._split_buf("join", R, 2 * fc)
        h6 = self._split_buf("h6", R, fc)
        self._linear(box7, R, 49 * c5, self.fc6[0], fc, self.fc6[1], True, out=h6, key="fc6")
        self._linear(h6, R, fc, self.fc7[0], fc, self.fc7[1], True, out=join, out_stride=2 * fc,
                     out_ch_offset=fc, key="fc7")
        m7 = self._split_buf("m7", R, 7, 7, c5)
        ops.mask_pool_split(feat14, masks.contiguous().float(), R, c5, m7)
        self._linear(m7, R, 49 * c5, self.fc6_mask[0], fc, self.fc6_mask[1], True, out=h6, key="fc6")
        self._linear(h6, R, fc, self.fc7_mask[0], fc, self.fc7_mask[1], True, out=join,
                     out_stride=2 * fc, out_ch_offset=0, key="fc7")
        h_me = self._split_buf("h_me", R, me)
        self._linear(feat14, R, 196 * c5, self.fc6_maskest[0], me, self.fc6_maskest[1], True,
                     out=h_me, key="me", block_k=32)
        logits = self._f32_buf("mask_logits_cfm", R, 448)
        self._linear(h_me, R, me, self.mask_pred[0], 441, self.mask_pred[1], False,
                     out_f32=logits, out_stride=448, key="mp")
        mask_prob, _ = ops.sigmoid_mask_resize(logits, R, MASK_SIZE, 14)
        heads = torch.empty((R, 128), dtype=torch.float32, device=self.device)
        self._linear(join, R, 2 * fc, self.cls_heads[0], 126, self.cls_heads[1], False,
                     out_f32=heads, out_stride=128, key="cls")
        out = dict(mask_prob=mask_prob, cls_prob=ops.softmax_rows(heads[:, 0:21], 21),
                   seg_cls_prob=ops.softmax_rows(heads[:, 21:42], 21), bbox_pred=heads[:, 42:126],
                   seg_cls_score=heads[:, 21:42])
        if keep_intermediate:
            out["_box7"] = box7.clone()
            out["_feat14"] = feat14.clone()
            out["_m7"] = m7.clone()
            out["_conv5_3"] = conv5_3.clone()
            out["_mask_logits"] = logits.clone()
        return out
