#!/usr/bin/env python
"""Run the original project's own kernels -- lib/nms/{nms,mv}_kernel.cu and the ROIWarping /
MaskResize / MaskPooling / ROIPooling Caffe layers, compiled unmodified into oracle/_ref/ by
`make -C oracle ref` (default and -fmad=false builds) -- on the inputs of tests/test_ref_pin.py and
tests/test_ref_fixtures.py, and store what they return in tests/golden/ref_pin.npz.  Needs a GPU
and oracle/_ref/; the tests that read the file need neither.

  python scripts/make_ref_pin_golden.py [OUT.npz]

Integer results (keep lists, boxes) are stored in full; float results compared bit for bit are
stored as tests.util.digest; float results held to a tolerance as tests.util.sample_idx elements
(`<key>_idx`, `<key>_val`)."""
import ctypes
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tests import util  # noqa: E402
from tests import test_ref_pin as T  # noqa: E402
from tests.test_ref_fixtures import load, voting_case, roi_pool_cpu_inputs  # noqa: E402

REF = os.path.join(ROOT, "oracle", "_ref")
p = T._p


def lib(name):
    return ctypes.CDLL(os.path.join(REF, name))


def main(out):
    nms, nms_nf = lib("libmnc_ref.so"), lib("libmnc_ref_nofma.so")
    lay, lay_nf = lib("libmnc_ref_layers.so"), lib("libmnc_ref_layers_nofma.so")
    g = {}

    def sample(key, a):
        idx = util.sample_idx(a.size)
        g[key + "_idx"] = idx.astype(np.int32)
        g[key + "_val"] = a.ravel()[idx]

    def ref_nms(dets, thresh):
        keep = np.zeros(dets.shape[0], dtype=np.int32)
        num = ctypes.c_int(0)
        nms._Z4_nmsPiS_PKfiifi(p(keep), ctypes.byref(num), p(dets), dets.shape[0], dets.shape[1],
                               ctypes.c_float(thresh), 0)
        return keep[:num.value]

    def ref_mv(so, boxes, masks, inds, start, w, H, W):
        k = len(start)
        rm = np.zeros((k, 1, 21, 21), dtype=np.float32)
        rb = np.zeros((k, 4), dtype=np.int32)
        so._Z3_mvPKfS0_iPKiS2_S0_iiiiiiPfPii(p(boxes), p(masks), boxes.shape[0], p(inds), p(start), p(w),
                                             len(inds), H, W, 4, 21, k, p(rm), p(rb), 0)
        return rm, rb

    for n, thresh, seed in T.NMS_CASES:
        g["nms_keep_%d_%d" % (n, seed)] = ref_nms(T.nms_sorted_dets(n, seed), thresh)

    boxes, masks, inds, start, w, H, W = T.mv_inputs()
    rm, rb = ref_mv(nms, boxes, masks, inds, start, w, H, W)
    rm_nf, rb_nf = ref_mv(nms_nf, boxes, masks, inds, start, w, H, W)
    sample("mv_mask", rm)
    g["mv_box"], g["mv_box_nofma"], g["mv_mask_nofma"] = rb, rb_nf, util.digest(rm_nf)

    f = load("ref_native_calls.npz")
    for tag in f["cases"]:
        g["replay_keep_" + tag] = util.digest(T.gpu_nms(ref_nms, f["dets_" + tag], float(f["thresh_" + tag])))
    v = load("ref_voting.npz")
    for tag in ("a", "b", "c"):
        boxes, masks, scores, H, W = voting_case(v, tag)
        for c in range(1, 21):
            dets = np.hstack((boxes.astype(np.float32), scores[:, c:c + 1]))
            g["replay_nms_%s_c%d" % (tag, c)] = util.digest(T.gpu_nms(ref_nms, dets, 0.3))
        for variant in ("np1", "np2"):
            sfx = "_%s_%s" % (tag, variant)
            args = (boxes, masks, v["cand_inds" + sfx], v["cand_start" + sfx], v["cand_weights" + sfx], H, W)
            rm, rb = ref_mv(nms, *args)
            rm_nf, rb_nf = ref_mv(nms_nf, *args)
            sample("replay_mask" + sfx, rm)
            g["replay_box" + sfx], g["replay_box_nofma" + sfx] = util.digest(rb), util.digest(rb_nf)
            g["replay_mask_nofma" + sfx] = util.digest(rm_nf)

    for P in T.WARP_SIZES:
        feat, rois = T._warp_inputs(120, seed=P)
        B, C, Hf, Wf = feat.shape
        for so, sfx in ((lay, ""), (lay_nf, "_nofma")):
            o = np.zeros((rois.shape[0], C, P, P), np.float32)
            assert so.ref_roi_warp(p(feat), B, C, Hf, Wf, p(rois), rois.shape[0], P, P, ctypes.c_float(0.0625), p(o)) == 0
            if sfx:
                g["warp%d_nofma" % P] = util.digest(o)
            else:
                sample("warp%d" % P, o)
                g["warp%d_zero" % P] = util.digest(o == 0)

    m, feat, mask = T.mask_inputs()
    for oh, ow in T.RESIZE_SIZES:
        for so, sfx in ((lay, ""), (lay_nf, "_nofma")):
            o = np.zeros((m.shape[0], 1, oh, ow), np.float32)
            assert so.ref_mask_resize(p(m), m.shape[0], 1, 21, 21, oh, ow, p(o)) == 0
            if sfx:
                g["resize%dx%d_nofma" % (oh, ow)] = util.digest(o)
            else:
                sample("resize%dx%d" % (oh, ow), o)
    o = np.zeros_like(feat)
    assert lay.ref_mask_pool(p(feat), p(mask), *feat.shape, p(o)) == 0
    g["mask_pool"] = util.digest(o)

    for P in T.POOL_SIZES:
        feat, rois = T._warp_inputs(100, seed=40 + P)
        B, C, Hf, Wf = feat.shape
        for use_gpu, dev in ((1, "gpu"), (0, "cpu")):
            o = np.zeros((rois.shape[0], C, P, P), np.float32)
            assert lay.ref_roi_pool(p(feat), B, C, Hf, Wf, p(rois), rois.shape[0], P, P, ctypes.c_float(0.0625),
                                    use_gpu, p(o)) == 0
            g["roi_pool%d_%s" % (P, dev)] = util.digest(o)

    feat, rois = roi_pool_cpu_inputs()
    for P in (7, 14):
        o = np.zeros((rois.shape[0], feat.shape[1], P, P), np.float32)
        assert lay.ref_roi_pool(p(feat), *feat.shape, p(rois), rois.shape[0], P, P, ctypes.c_float(0.0625), 0,
                                p(o)) == 0
        g["roi_pool_cpu%d" % P] = util.digest(o)

    np.savez_compressed(out, **g)
    print("wrote %s (%d entries, %d bytes)" % (out, len(g), os.path.getsize(out)))


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden", "ref_pin.npz"))
