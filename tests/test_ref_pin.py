"""Pin the oracle AND the CUDA path against the original project's own kernels: lib/nms/nms_kernel.cu,
lib/nms/mv_kernel.cu and the ROIWarping / MaskResize / MaskPooling / ROIPooling Caffe layers,
compiled unmodified (oracle/Makefile `ref`, default and -fmad=false builds) and run on a B200 by
scripts/make_ref_pin_golden.py on the inputs built here.  What they returned is stored in
tests/golden/ref_pin.npz (integer results in full, float results compared bit for bit as
util.digest, float results held to a tolerance as a fixed sample of elements), so the comparison
needs neither the original project nor its binaries."""
import ctypes
import functools
import os

import numpy as np
import pytest

from tests import util

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_pin.npz")

NMS_CASES = [(600, 0.3, 1), (6000, 0.7, 2), (10000, 0.7, 10)]
WARP_SIZES = [28, 14, 7]
RESIZE_SIZES = [(14, 14), (7, 9), (21, 21), (28, 28)]
POOL_SIZES = [7, 14]


@functools.lru_cache(maxsize=None)
def _golden():
    return dict(np.load(GOLDEN, allow_pickle=False))


def _want(key):
    g = _golden()
    return g[key].item() if g[key].ndim == 0 else g[key]


def _sampled(got, key):
    """(got at the stored sample positions, the reference's values there)."""
    g = _golden()
    return np.asarray(got).ravel()[g[key + "_idx"]], g[key + "_val"]


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _cuda_nms(sorted_dets, thresh):
    from mnc_b200._lib import lib, check
    n = sorted_dets.shape[0]
    keep = np.zeros(n, dtype=np.int32)
    num = ctypes.c_int(0)
    check(lib.mnc_nms_host(_p(keep), ctypes.byref(num), _p(sorted_dets), n, sorted_dets.shape[1],
                           ctypes.c_float(thresh), 0), "mnc_nms_host")
    return keep[:num.value]


def _cuda_mv(boxes, masks, inds, start, w, H, W):
    from mnc_b200._lib import lib, check
    k = len(start)
    rm = np.zeros((k, 1, 21, 21), dtype=np.float32)
    rb = np.zeros((k, 4), dtype=np.int32)
    check(lib.mnc_mv_host(_p(boxes), _p(masks), boxes.shape[0], _p(inds), _p(start), _p(w), len(inds), H,
                          W, 4, 21, k, _p(rm), _p(rb), 0), "mnc_mv_host")
    return rm, rb


def nms_sorted_dets(n, seed):
    from oracle import oracle as O
    boxes = util.random_boxes(n, seed=seed)
    scores = util.tie_free_scores(n, seed=seed + 1)
    dets = np.hstack([boxes, scores[:, None]]).astype(np.float32)
    return np.ascontiguousarray(dets[O.order_desc(scores)])


@pytest.mark.parametrize("n,thresh,seed", NMS_CASES)
def test_nms_three_way(n, thresh, seed):
    """reference `_nms` == oracle orc_nms == mnc_nms_host, float boxes, no margin nudging."""
    from oracle import oracle as O
    sorted_dets = nms_sorted_dets(n, seed)
    keep_ref = _want("nms_keep_%d_%d" % (n, seed))
    assert np.array_equal(_cuda_nms(sorted_dets, thresh), keep_ref), "CUDA path differs from reference _nms"
    assert np.array_equal(O.nms_sorted(sorted_dets, thresh), keep_ref), "oracle differs from reference _nms"


def _voting_inputs(nb, H, W, seed):
    rng = np.random.default_rng(seed)
    boxes = util.random_boxes(nb, seed=seed, width=W, height=H, smin=12, smax=min(H, W) * 0.8)
    masks = (1.0 / (1.0 + np.exp(-rng.normal(0, 2, size=(nb, 1, 21, 21))))).astype(np.float32)
    logits = rng.normal(0, 1, size=(nb, 21))
    scores = (np.exp(logits) / np.exp(logits).sum(1, keepdims=True)).astype(np.float32)
    return boxes, masks, scores


def mv_inputs():
    """gpu_mask_voting's candidate lists on a small image, so that the reference's nb*H*W render
    buffer stays small."""
    from oracle import oracle as O
    nb, H, W = 120, 150, 200
    boxes, masks, scores = _voting_inputs(nb, H, W, seed=21)
    inds, start, weights, _, _ = O.mask_voting_candidates(boxes, scores, 21, 100)
    return boxes, masks, inds, start, weights, H, W


def test_mv_three_way():
    """reference `_mv` vs oracle orc_mv vs mnc_mv_host."""
    from oracle import oracle as O
    boxes, masks, inds, start, weights, H, W = mv_inputs()
    assert len(start) > 10
    rb_ref = _want("mv_box")
    rm_o, rb_o = O.mv(boxes, masks, inds, start, weights, H, W)
    rm, rb = _cuda_mv(boxes, masks, inds, start, weights, H, W)
    # boxes: int-exact unless an aggregate value sits within an ulp of 0.4 (FMA contraction);
    # allow no mismatch on this seeded input
    assert np.array_equal(rb_o, rb_ref), "oracle boxes differ from reference _mv"
    assert np.array_equal(rb, rb_ref), "CUDA boxes differ from reference _mv"
    # mask values: the reference binary contracts a*b+c into FMA, the C oracle does not
    assert util.rel_err(*_sampled(rm_o, "mv_mask")) < 1e-4
    assert util.rel_err(*_sampled(rm, "mv_mask")) < 1e-4
    # ... and with contraction off (-fmad=false build of the same source) the reference equals the
    # oracle bit for bit
    assert np.array_equal(_want("mv_box_nofma"), rb_o) and util.digest(rm_o) == _want("mv_mask_nofma")


# ------------------------------------------------------------------------------------------------
# Replay of the native calls the reference's Python made while scripts/make_ref_fixtures.py produced
# tests/golden/ref_*.npz.  There (no GPU) `gpu_nms` was answered by the reference's py_cpu_nms.py
# and `mv` by the C oracle; the reference's REAL CUDA extensions (`_nms`, `_mv`, compiled
# unmodified) reproduced the recorded outputs from the recorded inputs -- which closes the chain
# fixture == reference-with-its-own-extensions -- and the CUDA path must reproduce them too.
def gpu_nms(nms_sorted, dets, thresh):
    """lib/nms/gpu_nms.pyx:16-31 around an `_nms`-like nms_sorted(sorted_dets, thresh) -> keep."""
    order = dets[:, 4].argsort()[::-1]
    sorted_dets = np.ascontiguousarray(dets[order, :])
    return order[nms_sorted(sorted_dets, thresh)]


def test_recorded_native_calls_replay():
    from tests.test_ref_fixtures import load, voting_case
    f = load("ref_native_calls.npz")
    for tag in f["cases"]:                        # ProposalLayer.forward -> nms(dets, 0.7)
        want = _want("replay_keep_" + tag)
        assert util.digest(f["keep_" + tag]) == want, tag
        assert util.digest(gpu_nms(_cuda_nms, f["dets_" + tag], float(f["thresh_" + tag]))) == want, tag
    v = load("ref_voting.npz")
    for tag in ("a", "b", "c"):
        boxes, masks, scores, H, W = voting_case(v, tag)
        for c in range(1, 21):                    # gpu_mask_voting -> nms(dets, 0.3) per class
            dets = np.hstack((boxes.astype(np.float32), scores[:, c:c + 1]))
            want = _want("replay_nms_%s_c%d" % (tag, c))
            assert util.digest(v["nms_keep_%s_c%d" % (tag, c)]) == want, (tag, c)
            assert util.digest(gpu_nms(_cuda_nms, dets, 0.3)) == want, (tag, c)
        for variant in ("np1", "np2"):            # gpu_mask_voting -> mv(...)
            sfx = "_%s_%s" % (tag, variant)
            box_ref = _want("replay_box" + sfx)
            assert util.digest(v["result_box" + sfx][:, :4].astype(np.int32)) == box_ref, (tag, variant)
            # the reference binary contracts a*b+c into FMA, the C oracle that recorded the masks
            # does not: values agree to fp32 rounding of one product, not bit for bit
            assert util.rel_err(*_sampled(v["result_mask" + sfx], "replay_mask" + sfx)) < 1e-4
            # same source, -fmad=false: bit for bit
            assert _want("replay_box_nofma" + sfx) == box_ref
            assert _want("replay_mask_nofma" + sfx) == util.digest(v["result_mask" + sfx])
            rm, rb = _cuda_mv(boxes, masks, v["cand_inds" + sfx], v["cand_start" + sfx],
                              v["cand_weights" + sfx], H, W)
            assert util.digest(rb) == box_ref, (tag, variant)
            assert util.rel_err(*_sampled(rm, "replay_mask" + sfx)) < 1e-4


# ------------------------------------------------------------------------------------------------
# The reference's Caffe layers for this path, compiled UNMODIFIED (.cu kernels and .cpp
# LayerSetUp/Reshape, class declarations from the reference's own headers) against the Caffe-runtime
# stand-in oracle/ref_stub into oracle/_ref/libmnc_ref_layers.so: reference == oracle == CUDA path.
def _warp_inputs(R, seed, B=2, C=24, H=38, W=63):
    rng = np.random.default_rng(seed)
    feat = np.maximum(rng.standard_normal((B, C, H, W)), 0).astype(np.float32)
    x1, y1 = rng.uniform(0, 16 * W - 17, R), rng.uniform(0, 16 * H - 17, R)
    rois = np.stack([rng.integers(0, B, R), x1, y1, np.minimum(x1 + rng.uniform(16, 600, R), 16 * W - 1),
                     np.minimum(y1 + rng.uniform(16, 600, R), 16 * H - 1)], 1).astype(np.float32)
    edge = np.array([[0, 0, 0, 0, 0],                       # degenerate: one sample point
                     [0, 0, 0, 16 * W - 1, 16 * H - 1],     # whole map
                     [1, 16 * W - 9, 16 * H - 9, 16 * W - 1, 16 * H - 1],   # bottom-right corner
                     [0, 8, 8, 8, 300], [1, 8, 8, 300, 8],  # zero width / zero height after rounding
                     [0, 500, 300, 400, 200],               # inverted (end < start): clamped to 0 size
                     [1, 7.99, 24.0, 600.5, 424.01]], dtype=np.float32)   # .5 rounding cases
    return feat, np.vstack([edge, rois]).astype(np.float32)


@pytest.mark.parametrize("P", WARP_SIZES)
def test_roi_warping_three_way(P):
    """ROIWarpingLayer::Forward_gpu (roi_warping_layer.cu:67-122) == oracle == mnc_roi_warp_nchw."""
    import torch
    from oracle import oracle as O
    from mnc_b200 import ops
    feat, rois = _warp_inputs(120, seed=P)
    assert np.abs(_want("warp%d_val" % P)).max() > 0
    orc = O.roi_warp(feat, rois, P, P)
    got = ops.roi_warp_nchw(torch.from_numpy(feat).cuda(), torch.from_numpy(rois).cuda(), P, P).cpu().numpy()
    # nvcc fuses `start + p * bin` and the 4-tap sum of the reference source into FMAs; a 1-ulp
    # sample coordinate moves a value by ~1e-5 of the map's range.  The oracle and our kernel keep
    # every operation separately rounded, and equal the reference compiled with -fmad=false bit
    # for bit.
    assert util.rel_err(*_sampled(orc, "warp%d" % P)) < 2e-5, "oracle differs from reference ROIWarping"
    assert util.rel_err(*_sampled(got, "warp%d" % P)) < 2e-5, "CUDA path differs from reference ROIWarping"
    assert util.digest(orc == 0) == _want("warp%d_zero" % P)      # out-of-map samples in the same places
    nofma = _want("warp%d_nofma" % P)
    assert util.digest(orc) == nofma, "oracle != reference ROIWarping built with -fmad=false"
    assert util.digest(got) == nofma, "CUDA path != reference ROIWarping built with -fmad=false"


def mask_inputs():
    rng = np.random.default_rng(5)
    m = rng.uniform(0, 1, size=(37, 1, 21, 21)).astype(np.float32)
    feat = rng.standard_normal((37, 24, 14, 14)).astype(np.float32)
    mask = rng.uniform(0, 1, size=(37, 1, 14, 14)).astype(np.float32)
    return m, feat, mask


def test_mask_resize_and_pooling_three_way():
    """MaskResizeLayer / MaskPoolingLayer Forward_gpu (mask_resize_layer.cu:57-84,
    mask_pooling_layer.cu:13-41) == oracle == mnc_mask_resize_nchw / mnc_mask_pool_nchw."""
    import torch
    from oracle import oracle as O
    from mnc_b200 import ops
    m, feat, mask = mask_inputs()
    for oh, ow in RESIZE_SIZES:
        key = "resize%dx%d" % (oh, ow)
        orc = O.mask_resize(m, oh, ow)
        got = ops.mask_resize_nchw(torch.from_numpy(m).cuda(), oh, ow).cpu().numpy()
        assert util.rel_err(*_sampled(orc, key)) < 2e-6 and util.rel_err(*_sampled(got, key)) < 2e-6
        assert util.digest(orc) == _want(key + "_nofma") and util.digest(got) == _want(key + "_nofma")
    got = ops.mask_pool_nchw(torch.from_numpy(feat).cuda(), torch.from_numpy(mask).cuda()).cpu().numpy()
    assert util.digest(O.mask_pool(feat, mask)) == _want("mask_pool")      # one multiply: bit-exact
    assert util.digest(got) == _want("mask_pool")


@pytest.mark.parametrize("P", POOL_SIZES)
def test_roi_pooling_three_way(P):
    """ROIPoolingLayer Forward_gpu and Forward_cpu (roi_pooling_layer.cu:17-92, .cpp:46-132) ==
    oracle == mnc_roi_pool_nchw (max over integer bins: bit-exact)."""
    import torch
    from oracle import oracle as O
    from mnc_b200 import ops
    feat, rois = _warp_inputs(100, seed=40 + P)
    want = _want("roi_pool%d_gpu" % P)
    assert _want("roi_pool%d_cpu" % P) == want
    assert util.digest(O.roi_pool(feat, rois, P, P)) == want
    got = ops.roi_pool_nchw(torch.from_numpy(feat).cuda(), torch.from_numpy(rois).cuda(), P, P).cpu().numpy()
    assert util.digest(got) == want
