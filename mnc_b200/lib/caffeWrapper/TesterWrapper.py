"""Dataset-level result collection -- mirror of the reference's lib/caffeWrapper/TesterWrapper.py
for the segmentation task (`get_result` :46-67, `get_segmentation_result` :149-214,
`_segmentation_forward` :239-260): run every image of an imdb through the 5-stage net + mask
voting, keep [class][image] arrays, write `res_boxes.pkl` / `res_masks.pkl`, hand them to
`imdb.evaluate_segmentation`.

The reference walks the images one by one (batch 1).  Here images are bucketed by size and sent
through the batched engine (`Detector.im_detect_images` + device mask voting), `max_batch` at a
time; results are stored by image index, so the output structure is the reference's.

The sibling tasks ride on the same class (SURVEY.md section 8f row 4): `det` (Faster R-CNN test
net, `get_detection_result` :85-143) and `cfm` (`get_cfm_result` / `cfm_network_forward`
:286-414, multi-scale pyramid with externally supplied mask proposals).

`imdb` is duck-typed as in the reference: `image_index`, `num_classes`, `image_path_at(i)`,
`evaluate_segmentation(all_boxes, all_masks, output_dir)` / `evaluate_detections(all_boxes,
output_dir)`; optional `image_at(i)` returning a BGR uint8 array bypasses cv2.imread,
`proposals_at(i)` supplies the CFM proposals, `output_dir` overrides the default output location.
"""
import heapq
import os
import pickle

import numpy as np
import torch

from mnc_b200 import ops
from mnc_b200.api import Detector, unpack_voting
from mnc_config import cfg
from nms.nms_wrapper import apply_nms_mask_single


class TesterWrapper(object):
    def __init__(self, test_prototxt, imdb, test_model, task_name, max_batch=8, device=None):
        from caffe.net import load_weights
        from mnc_b200.siblings import FasterRCNNEngine, CFMEngine
        self.device = torch.device(device or "cuda:%d" % cfg.GPU_ID)
        weights, self.kind = load_weights(test_prototxt, test_model, return_kind=True)
        want = {"seg": "mnc_5stage", "det": "faster_rcnn", "cfm": "cfm"}.get(task_name)
        if want is None:
            raise NotImplementedError("task name only support 'det', 'seg' and 'cfm'")
        if want != self.kind:
            raise ValueError("task '%s' runs the %s graph, got the %s graph" % (task_name, want, self.kind))
        self.max_batch = max_batch
        if self.kind == "mnc_5stage":
            self.detector = Detector(weights, device=self.device, max_batch=max_batch)
        else:
            with torch.cuda.device(self.device):
                self.engine = (FasterRCNNEngine if self.kind == "faster_rcnn" else CFMEngine)(
                    weights, device=self.device)
        self.name = (os.path.splitext(os.path.basename(test_model))[0]
                     if isinstance(test_model, str) else "mnc_5stage")
        self.imdb = imdb
        self.output_dir = getattr(imdb, "output_dir", None) or os.path.join("output", self.name)
        self.task_name = task_name
        self.num_images = len(self.imdb.image_index)
        self.num_classes = self.imdb.num_classes
        self.max_per_set = 40 * self.num_images     # :39
        self.max_per_image = 100                    # :41
        os.makedirs(self.output_dir, exist_ok=True)

    # ------------------------------------------------------------------ :46-67
    def get_result(self):
        det_file = os.path.join(self.output_dir, "res_boxes.pkl")
        seg_file = os.path.join(self.output_dir, "res_masks.pkl")
        if self.task_name == "det":
            return self.get_detection_result()
        if os.path.isfile(det_file) and os.path.isfile(seg_file):
            with open(det_file, "rb") as f:
                seg_box = pickle.load(f)
            with open(seg_file, "rb") as f:
                seg_mask = pickle.load(f)
        else:
            seg_box, seg_mask = (self.get_segmentation_result() if self.task_name == "seg"
                                 else self.get_cfm_result())
            with open(det_file, "wb") as f:
                pickle.dump(seg_box, f, pickle.HIGHEST_PROTOCOL)
            with open(seg_file, "wb") as f:
                pickle.dump(seg_mask, f, pickle.HIGHEST_PROTOCOL)
        return self.imdb.evaluate_segmentation(seg_box, seg_mask, self.output_dir)

    def _read(self, i):
        if hasattr(self.imdb, "image_at"):
            return np.ascontiguousarray(self.imdb.image_at(i))
        import cv2
        return cv2.imread(self.imdb.image_path_at(i))

    def _buckets(self):
        """image indices grouped by image size, each group cut into engine batches."""
        by_shape = {}
        for i in range(self.num_images):
            by_shape.setdefault(self._read(i).shape, []).append(i)
        mb = self.max_batch
        for idx in by_shape.values():
            for s in range(0, len(idx), mb):
                yield idx[s:s + mb]

    # ------------------------------------------------------------------ :85-143 (task 'det')
    def _detection_forward_batch(self, ims):
        """Batched `_detection_forward` (:215-237) on equally sized uint8 images.
        -> scores (B,300,21), pred_boxes (B,300,84), valid (B,300) host arrays."""
        B, H, W = ims.shape[:3]
        dev = self.device
        scale = ops.im_scale_for((H, W), cfg.TEST.SCALES[0], cfg.TRAIN.MAX_SIZE)
        out_h, out_w = int(np.rint(H * scale)), int(np.rint(W * scale))
        with torch.cuda.device(dev):
            data = ops.prep_images(torch.from_numpy(ims).to(dev), scale)
            info = torch.tensor([[out_h, out_w, scale]] * B, dtype=torch.float32, device=dev)
            hw = torch.tensor([[H, W]] * B, dtype=torch.float32, device=dev)
            sc = torch.full((B,), scale, dtype=torch.float32, device=dev)
            scores, pred, valid, _ = self.engine.detect_checked(data, info, hw, sc)
            return scores.cpu().numpy(), pred.cpu().numpy(), valid.cpu().numpy().astype(bool)

    def _detection_forward(self, im):
        scores, pred, valid = self._detection_forward_batch(np.ascontiguousarray(im)[None])
        return scores[0][valid[0]], pred[0][valid[0]]

    def get_detection_result(self):
        nc, ni = self.num_classes, self.num_images
        book = _ClassBook(nc, self.max_per_set, self.max_per_image)
        all_boxes = [[[] for _ in range(ni)] for _ in range(nc)]
        for batch in self._buckets():
            scores, pred, valid = self._detection_forward_batch(np.stack([self._read(i) for i in batch]))
            for b, i in enumerate(batch):
                sc, bx = scores[b][valid[b]], pred[b][valid[b]]
                for j in range(1, nc):
                    inds = book.select(j, sc[:, j])
                    all_boxes[j][i] = np.hstack((bx[inds, j * 4:(j + 1) * 4], sc[inds, j][:, None])) \
                        .astype(np.float32, copy=False)
        for j in range(1, nc):
            for i in range(ni):
                keep = np.where(all_boxes[j][i][:, -1] > book.thresh[j])[0]
                all_boxes[j][i] = all_boxes[j][i][keep, :]
        with open(os.path.join(self.output_dir, "detections.pkl"), "wb") as f:
            pickle.dump(all_boxes, f, pickle.HIGHEST_PROTOCOL)
        from nms.nms_wrapper import apply_nms
        nms_dets = apply_nms(all_boxes, cfg.TEST.NMS)
        return self.imdb.evaluate_detections(nms_dets, self.output_dir)

    # ------------------------------------------------------------------ :286-414 (task 'cfm')
    def cfm_network_forward(self, im_i):
        """Multi-scale CFM forward for image `im_i` with the imdb's object proposals
        (`imdb.proposals_at(i)` -> boxes (n,4), masks (n,h,w); the reference reads them from the
        MCG .mat cache, :338-343).  -> masks (n,1,21,21), boxes (n,4), seg scores (n,21)."""
        import cv2
        from transform.bbox_transform import filter_small_boxes
        from utils.blob import prep_im_for_blob_cfm, pred_rois_for_blob
        im = self._read(im_i)
        boxes, masks = self.imdb.proposals_at(im_i)
        keep = filter_small_boxes(boxes, min_size=16)
        boxes, masks = boxes[keep, :], masks[keep, :, :]
        S = cfg.TEST.CFM_INPUT_MASK_SIZE
        # proposal masks to the CFM input size (:346-350): input preparation, host cv2 as upstream
        masks = np.stack([cv2.resize(m.astype(np.float64), (S, S)) for m in masks]) if len(masks) \
            else np.zeros((0, S, S))
        if cfg.TEST.USE_TOP_K_MCG:
            k = min(boxes.shape[0], cfg.TEST.USE_TOP_K_MCG)
            boxes, masks = boxes[:k, :], masks[:k, :, :]
        _, im_scale_factors = prep_im_for_blob_cfm(im, cfg.TEST.SCALES)
        orig_boxes = boxes.copy()
        boxes = pred_rois_for_blob(boxes, im_scale_factors)
        group = cfg.TEST.GROUP_SCALE
        res_boxes = np.zeros((0, 4), dtype=np.float32)
        res_masks = np.zeros((0, 1, cfg.MASK_SIZE, cfg.MASK_SIZE), dtype=np.float32)
        res_scores = np.zeros((0, self.num_classes), dtype=np.float32)
        dev = self.device
        for it, lo in enumerate(range(0, len(cfg.TEST.SCALES), group)):
            hi = min(lo + group, len(cfg.TEST.SCALES))
            inds = np.where((boxes[:, 0] >= lo) & (boxes[:, 0] < hi))[0]
            if len(inds) == 0:
                continue
            max_rois = cfg.TEST.MAX_ROIS_GPU[it]
            b_scale, m_scale = boxes[inds, :].copy(), masks[inds, :, :]
            b_scale[:, 0] -= b_scale[:, 0].min()
            data, _ = prep_im_for_blob_cfm(im, cfg.TEST.SCALES[lo:hi])
            with torch.cuda.device(dev):
                d_data = torch.from_numpy(np.ascontiguousarray(data, dtype=np.float32)).to(dev)
                for s in range(0, b_scale.shape[0], max_rois):
                    rois = b_scale[s:s + max_rois].astype(np.float32, copy=False)
                    m_in = (m_scale[s:s + max_rois].reshape(-1, 1, S, S).astype(np.float32)
                            >= cfg.BINARIZE_THRESH).astype(np.float32)
                    o = self.engine.run_checked(
                        self.engine.forward, d_data, torch.from_numpy(np.ascontiguousarray(rois)).to(dev),
                        torch.from_numpy(m_in).to(dev))
                    res_masks = np.vstack((res_masks, o["mask_prob"].cpu().numpy().reshape(
                        -1, 1, cfg.MASK_SIZE, cfg.MASK_SIZE)))
                    res_scores = np.vstack((res_scores, o["seg_cls_prob"].cpu().numpy()))
            res_boxes = np.vstack((res_boxes, orig_boxes[inds, :]))
        return res_masks, res_boxes, res_scores

    def get_cfm_result(self):
        nc, ni = self.num_classes, self.num_images
        book = _ClassBook(nc, self.max_per_set, self.max_per_image)
        all_boxes = [[[] for _ in range(ni)] for _ in range(nc)]
        all_masks = [[[] for _ in range(ni)] for _ in range(nc)]
        for i in range(ni):
            masks, boxes, seg_scores = self.cfm_network_forward(i)
            for j in range(1, nc):
                inds = book.select(j, seg_scores[:, j])
                dets = np.hstack((boxes[inds, :], seg_scores[inds, j][:, None])).astype(np.float32, copy=False)
                all_boxes[j][i], all_masks[j][i] = apply_nms_mask_single(
                    dets, masks[inds, :].astype(np.float32, copy=False), cfg.TEST.NMS)
        for j in range(1, nc):
            for i in range(ni):
                if len(all_boxes[j][i]) == 0:
                    continue
                keep = np.where(all_boxes[j][i][:, -1] > book.thresh[j])[0]
                all_boxes[j][i] = all_boxes[j][i][keep, :]
                all_masks[j][i] = all_masks[j][i][keep]
        return all_boxes, all_masks

    # ------------------------------------------------------------------ :149-214
    def get_segmentation_result(self):
        nc, ni = self.num_classes, self.num_images
        book = _ClassBook(nc, self.max_per_set, self.max_per_image)
        all_boxes = [[[] for _ in range(ni)] for _ in range(nc)]
        all_masks = [[[] for _ in range(ni)] for _ in range(nc)]
        det = self.detector
        for batch in self._buckets():
            ims = np.stack([self._read(i) for i in batch])
            H, W = ims.shape[1:3]
            if cfg.TEST.USE_MASK_MERGE:
                if not cfg.TEST.USE_GPU_MASK_MERGE:
                    raise NotImplementedError("cpu_mask_voting is off the GPU path (out of scope)")
                per_image = self._vote_batch(ims)
                for i, (result_mask, result_box) in zip(batch, per_image):
                    for j in range(1, nc):
                        all_boxes[j][i] = result_box[j - 1]
                        all_masks[j][i] = result_mask[j - 1]
            else:
                boxes, masks, scores, valid, _ = det.im_detect_images(ims)
                for b, i in enumerate(batch):
                    ok = valid[b].astype(bool)
                    bx, mk, sc = boxes[b][ok], masks[b][ok], scores[b][ok]
                    for j in range(1, nc):
                        inds = book.select(j, sc[:, j])
                        dets = np.hstack((bx[inds], sc[inds, j][:, None])).astype(np.float32, copy=False)
                        all_boxes[j][i], all_masks[j][i] = apply_nms_mask_single(
                            dets, mk[inds].astype(np.float32, copy=False), cfg.TEST.NMS)
        for j in range(1, nc):
            for i in range(ni):
                if len(all_boxes[j][i]) == 0:
                    continue
                inds = np.where(all_boxes[j][i][:, -1] > book.thresh[j])[0]
                all_boxes[j][i] = all_boxes[j][i][inds, :]
                all_masks[j][i] = all_masks[j][i][inds]
        return all_boxes, all_masks

    def _vote_batch(self, ims):
        """forward + gpu_mask_voting for one batch of equally sized images (Detector.im_segment).
        -> per image (list_mask, list_box) in the format `gpu_mask_voting` returns
        (mask_transform.py:270-286)."""
        res = self.detector.im_segment(ims, max_per_image=self.max_per_image)
        return [unpack_voting(r, self.num_classes) for r in res]


class _ClassBook(object):
    """The adaptive per-class score threshold of the reference's result loops (:95-124,:163-186,
    :300-320): per image keep the `max_per_image` best rows above the class threshold; a min-heap
    of all kept scores raises the threshold once more than `max_per_set` have been collected."""

    def __init__(self, num_classes, max_per_set, max_per_image):
        self.thresh = -np.inf * np.ones(num_classes)
        self.heaps = [[] for _ in range(num_classes)]
        self.max_per_set, self.max_per_image = max_per_set, max_per_image

    def select(self, j, scores_j):
        inds = np.where(scores_j > self.thresh[j])[0]
        inds = inds[np.argsort(-scores_j[inds])[:self.max_per_image]]
        heap = self.heaps[j]
        for val in scores_j[inds]:
            heapq.heappush(heap, val)
        if len(heap) > self.max_per_set:
            while len(heap) > self.max_per_set:
                heapq.heappop(heap)
            self.thresh[j] = heap[0]
        return inds
