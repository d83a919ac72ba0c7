"""Oracle == REFERENCE, on fixtures the reference's own Python produced (tests/golden/ref_*.npz, made
by scripts/make_ref_fixtures.py from /root/reference: ProposalLayer.forward, StageBridgeLayer /
MaskLayer forward, bbox_transform, anchors, gpu_mask_voting, prep_im_for_blob, demo.im_detect, the
cythonized bbox_overlaps, the real cfg).  Bit-exact unless stated.  CPU only; the CUDA path is held
to the same fixtures in tests/test_gpu_ref_fixtures.py, and the native calls the reference made
while producing them were replayed through its real CUDA extensions (tests/test_ref_pin.py)."""
import os
import zlib

import numpy as np
import pytest

from oracle import oracle as O

G = os.path.join(os.path.dirname(__file__), "golden")


def load(name):
    return np.load(os.path.join(G, name), allow_pickle=False)


def test_cfg_constants():
    c = load("ref_cfg.npz")
    assert np.array_equal(c["PIXEL_MEANS"], O.CFG.PIXEL_MEANS)
    for k_ref, k in (("BINARIZE_THRESH", "BINARIZE_THRESH"), ("MASK_SIZE", "MASK_SIZE"),
                     ("TEST_NMS", "TEST_NMS"), ("RPN_NMS_THRESH", "RPN_NMS_THRESH"),
                     ("RPN_PRE_NMS_TOP_N", "RPN_PRE_NMS_TOP_N"), ("RPN_POST_NMS_TOP_N", "RPN_POST_NMS_TOP_N"),
                     ("RPN_MIN_SIZE", "RPN_MIN_SIZE"), ("MASK_MERGE_IOU_THRESH", "MASK_MERGE_IOU_THRESH"),
                     ("MASK_MERGE_NMS_THRESH", "MASK_MERGE_NMS_THRESH"), ("TEST_MAX_SIZE", "TEST_MAX_SIZE")):
        assert c[k_ref] == getattr(O.CFG, k), k
    assert tuple(c["TEST_SCALES"]) == O.CFG.TEST_SCALES
    assert c["TRAIN_MAX_SIZE"] == O.CFG.TEST_MAX_SIZE      # demo.py:59 passes cfg.TRAIN.MAX_SIZE
    assert bool(c["USE_GPU_NMS"]) and bool(c["USE_GPU_MASK_MERGE"])


def test_anchors_and_bbox_transforms():
    f = load("ref_bbox.npz")
    assert np.array_equal(f["anchors"], O.generate_anchors())
    for tag in ("a", "b"):
        pred = O.bbox_transform_inv(f["boxes_" + tag], f["deltas_" + tag])
        assert pred.dtype == f["pred_" + tag].dtype and np.array_equal(pred, f["pred_" + tag])
        clipped, keep = O.clip_boxes(pred, np.array([600, 1000], np.float32))
        assert np.array_equal(clipped, f["clipped_" + tag]) and np.array_equal(keep, f["clip_keep_" + tag])
        assert np.array_equal(O.filter_small_boxes(clipped[:, :4], 16 * 1.6), f["small_keep_" + tag])
    e = O.bbox_transform_inv(np.zeros((0, 4), np.float32), np.zeros((0, 84), np.float32))
    assert e.shape == f["pred_empty"].shape
    ov = O.bbox_overlaps(f["ov_boxes"], f["ov_boxes"][::3].copy())
    assert np.array_equal(ov, f["ov"])        # float64, == the reference's cythonized bbox.pyx


def test_proposal_layer_forward():
    f = load("ref_proposal.npz")
    for tag in f["cases"]:
        rois, mid = O.proposal_layer_forward(f["prob_" + tag], f["deltas_" + tag], f["im_info_" + tag],
                                             return_intermediate=True)
        want = f["rois_" + tag]
        assert rois.shape == want.shape and rois.dtype == np.float32, tag
        assert np.array_equal(rois, want), tag
        assert np.array_equal(mid["keep_filter"], f["ind_after_filter_" + tag])
        assert np.array_equal(mid["order"], f["ind_after_sort_" + tag])
        assert np.array_equal(mid["nms_keep"], f["proposal_index_" + tag])


def test_stage_bridge_and_mask_layer():
    f = load("ref_stage_bridge.npz")
    for tag in ("a", "b"):
        got = O.stage_bridge_forward(f["rois_" + tag], f["bbox_pred_" + tag], f["prob_" + tag],
                                     f["im_info_" + tag])
        assert got.dtype == np.float32 and np.array_equal(got, f["rois_ext_" + tag])
    assert np.array_equal(O.mask_layer_forward(f["mask_output"]), f["mask_proposal"])


def voting_case(f, tag):
    masks = (f["masks_q4096_" + tag].astype(np.float32) / np.float32(4096.0)).astype(np.float32)
    H, W = (int(v) for v in f["hw_" + tag])
    return f["boxes_" + tag], masks, f["scores_" + tag], H, W


@pytest.mark.parametrize("tag", ["a", "b", "c"])
def test_gpu_mask_voting_host_logic(tag):
    f = load("ref_voting.npz")
    boxes, masks, scores, H, W = voting_case(f, tag)
    for c in range(1, 21):     # the 20 nms() calls of mask_transform.py:233-234
        dets = np.hstack((boxes.astype(np.float32), scores[:, c:c + 1]))
        assert np.array_equal(np.asarray(O.nms(dets, O.CFG.MASK_MERGE_NMS_THRESH)),
                              f["nms_keep_%s_c%d" % (tag, c)]), c
    for variant, np2 in (("np1", False), ("np2", True)):
        inds, start, weights, cscores, class_bar = O.mask_voting_candidates(boxes, scores, 21, 100, numpy2=np2)
        sfx = "_%s_%s" % (tag, variant)
        assert np.array_equal(inds, f["cand_inds" + sfx])
        assert np.array_equal(start, f["cand_start" + sfx])
        assert np.array_equal(weights, f["cand_weights" + sfx]), variant
        lm, lb = O.gpu_mask_voting(masks, boxes, scores, 21, 100, W, H, numpy2=np2)
        assert np.array_equal(np.array([len(b) for b in lb]), f["class_counts" + sfx])
        assert np.array_equal(np.vstack(lb), f["result_box" + sfx])
        assert np.array_equal(np.concatenate(lm, 0), f["result_mask" + sfx])
    # the two numpy rules differ only in the weights, by the rounding of a float32 running sum
    w1, w2 = f["cand_weights_%s_np1" % tag], f["cand_weights_%s_np2" % tag]
    assert np.all(np.abs(w1 - w2) <= 2e-6 * np.maximum(w1, w2))


def tail_case(f, tag):
    seed, H, W, crc = (int(v) for v in f["im_seed_shape_crc_" + tag])
    im = np.random.default_rng(seed).integers(0, 256, size=(H, W, 3), dtype=np.uint8)
    assert zlib.crc32(im.tobytes()) == crc
    blobs = {"rois": f["rois_" + tag], "rois_ext": f["rois_ext_" + tag],
             "mask_proposal": f["mask_" + tag], "mask_proposal_ext": f["mask_ext_" + tag],
             "seg_cls_prob": f["prob_" + tag], "seg_cls_prob_ext": f["prob_ext_" + tag]}
    return im, blobs


def test_prep_and_im_detect_tail():
    f = load("ref_prep_tail.npz")
    for tag in f["cases"]:
        im, blobs = tail_case(f, tag)
        x, scale = O.prep_im_for_blob(im)
        assert scale == float(f["scale_" + tag])
        data = np.ascontiguousarray(x[np.newaxis].transpose(0, 3, 1, 2))
        assert np.array_equal(np.array(data.shape), f["data_shape_" + tag])
        assert np.array_equal(data[0, :, ::37, ::41], f["data_probe_" + tag])
        assert data.astype(np.float64).sum() == float(f["data_sum_" + tag])
        info = f["im_info_" + tag]
        assert info.dtype == np.float32
        assert np.array_equal(info, np.array([[data.shape[2], data.shape[3], scale]], np.float32))
        boxes, masks, scores = O.im_detect_tail(blobs, im.shape, scale, numpy2=True)
        want = f["out_boxes_" + tag]
        assert boxes.dtype == want.dtype and np.array_equal(boxes, want), tag
        assert np.array_equal(masks, f["out_masks_" + tag]) and np.array_equal(scores, f["out_scores_" + tag])
        b1, _, _ = O.im_detect_tail(blobs, im.shape, scale, numpy2=False)   # numpy-1.x rule: fp32 divide
        assert b1.dtype == np.float32
        assert np.all(np.abs(b1.astype(np.float64) - want) <= np.spacing(np.maximum(np.abs(b1), 1e-30)))
        # some box must actually hit the original-image border, or the clip is untested
        assert (want[:, 2] == im.shape[1] - 1).any() and (want[:, 3] == im.shape[0] - 1).any()


def roi_pool_cpu_inputs():
    rng = np.random.default_rng(7)
    feat = rng.standard_normal((2, 24, 38, 63)).astype(np.float32)
    R = 80
    x1, y1 = rng.uniform(0, 950, R), rng.uniform(0, 560, R)
    rois = np.stack([rng.integers(0, 2, R), x1, y1, np.minimum(x1 + rng.uniform(0, 600, R), 999),
                     np.minimum(y1 + rng.uniform(0, 600, R), 599)], 1).astype(np.float32)
    return feat, rois


def test_reference_roi_pooling_cpu_forward():
    """The reference's own ROIPoolingLayer::Forward_cpu (roi_pooling_layer.cpp:46-132, compiled
    unmodified; its output stored as a digest in ref_pin.npz by scripts/make_ref_pin_golden.py):
    oracle == reference."""
    from tests import util
    g = load("ref_pin.npz")
    feat, rois = roi_pool_cpu_inputs()
    for P in (7, 14):
        assert util.digest(O.roi_pool(feat, rois, P, P)) == g["roi_pool_cpu%d" % P].item()
