"""Detector.im_segment / im_segment_stream: raw images (one size, or a list of sizes) to voted
instances and rendered label images, against the reference's flow built from the mirrored
functions (`im_detect` -> `gpu_mask_voting` per image -> `get_vis_dict` ->
`_convert_pred_to_image`), and the ragged, score-filtered rendering kernel
(mnc_paste_voted_ragged) against `select_for_display` + `paste_instances` per image."""
import functools
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

DEMO = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "demo")


@pytest.fixture
def pinned_split(monkeypatch):
    from mnc_b200.engine import MNCEngine
    monkeypatch.setattr(MNCEngine, "_pick_split", lambda self, *a, **k: 1)


@functools.lru_cache(maxsize=None)
def _weights(arch="TINY_ARCH"):
    from mnc_b200 import weights as Wt
    return Wt.make_weights(getattr(Wt, arch))


def _mix():
    """The two demo images (landscape 375x500 / 500x333 class sizes) and seeded images of both
    orientations: sizes differ in both dimensions."""
    import cv2
    from oracle import oracle as O
    demo = [cv2.imread(os.path.join(DEMO, n + ".jpg")) for n in ("2008_000533", "2008_001602")]
    return demo + [O.synthetic_image(i, h, w) for i, (h, w) in
                   enumerate([(375, 500), (500, 333), (480, 640)])]


def _reference_vote(boxes, masks, scores, valid, b, im):
    import mnc_b200.lib as L
    L.install()
    from transform.mask_transform import gpu_mask_voting
    ok = valid[b].astype(bool)
    return gpu_mask_voting(masks[b][ok], boxes[b][ok], scores[b][ok], 21, 100, im.shape[1], im.shape[0])


def _assert_equals_reference(res, rm, rb):
    from mnc_b200.api import unpack_voting
    list_mask, list_box = unpack_voting(res)
    n = 0
    for j in range(20):
        assert np.array_equal(list_box[j], np.asarray(rb[j], np.float32).reshape(-1, 5)), j
        assert np.array_equal(list_mask[j], np.asarray(rm[j], np.float32).reshape(-1, 1, 21, 21)), j
        n += len(list_box[j])
    assert n == len(res["scores"])
    return n


def _assert_same(a, b, keys=("boxes", "scores", "classes", "masks", "scale")):
    for k in keys:
        assert np.array_equal(np.asarray(a[k]), np.asarray(b[k])), k


def test_uniform_batch_equals_detect_then_reference_voting():
    from oracle import oracle as O
    from mnc_b200.api import Detector
    det = Detector(_weights(), max_batch=8)
    ims = np.stack([O.synthetic_image(i, 375, 500) for i in range(3)])
    res = det.im_segment(ims)
    boxes, masks, scores, valid, scale = [np.array(o, copy=True) for o in det.im_detect_images(ims)]
    assert len(res) == 3
    total = 0
    for b, r in enumerate(res):
        assert r["boxes"].dtype == np.int32 and r["classes"].dtype == np.int32
        assert r["scores"].dtype == np.float32 and r["masks"].shape == (len(r["scores"]), 21, 21)
        assert r["scale"] == scale and "inst" not in r
        total += _assert_equals_reference(r, *_reference_vote(boxes, masks, scores, valid, b, ims[b]))
    assert total > 0


@pytest.mark.parametrize("arch", ["TINY_ARCH", "FULL_ARCH"])
def test_mixed_batch_equals_detect_mixed_and_each_image_alone(arch, pinned_split):
    from mnc_b200.api import Detector
    det = Detector(_weights(arch), max_batch=8)
    ims = _mix()
    res = det.im_segment(ims)
    boxes, masks, scores, valid, scales = [np.array(o, copy=True) for o in det.im_detect_mixed(ims)]
    total = 0
    for b, (r, im) in enumerate(zip(res, ims)):
        assert r["scale"] == scales[b]
        total += _assert_equals_reference(r, *_reference_vote(boxes, masks, scores, valid, b, im))
        _assert_same(r, det.im_segment([im])[0])
    assert total > 0


def _vote_dict(r, dev="cuda"):
    """One image's im_segment result as the (B = 1) device dict `select_for_display` takes."""
    k = len(r["scores"])
    R = max(k, 1)
    d = dict(n_res=torch.tensor([k], dtype=torch.int32),
             res_score=torch.zeros((1, R)), res_class=torch.zeros((1, R), dtype=torch.int32),
             result_box=torch.zeros((1, R, 4), dtype=torch.int32), result_mask=torch.zeros((1, R, 1, 21, 21)))
    d["res_score"][0, :k] = torch.from_numpy(r["scores"])
    d["res_class"][0, :k] = torch.from_numpy(r["classes"])
    d["result_box"][0, :k] = torch.from_numpy(r["boxes"])
    d["result_mask"][0, :k, 0] = torch.from_numpy(r["masks"])
    return {key: v.to(dev) for key, v in d.items()}


def _display_reference(vote, H, W, vis_thresh):
    from mnc_b200 import ops
    vb, vm, vc, cnt = ops.select_for_display(vote, vis_thresh=vis_thresh)
    inst, cls, bgr = ops.paste_instances(vb, vm, vc, cnt, H, W, want_bgr=True)
    return inst[0].cpu().numpy(), cls[0].cpu().numpy(), bgr[0].cpu().numpy()


@pytest.mark.parametrize("vis_thresh", [0.0, 0.5, 1.01])
def test_render_of_mixed_batch_equals_select_and_paste_per_image(vis_thresh):
    import mnc_b200.lib as L
    L.install()
    from utils.vis_seg import get_vis_dict, _convert_pred_to_image
    from mnc_b200.api import Detector, unpack_voting
    det = Detector(_weights(), max_batch=8)
    ims = _mix()
    plain = det.im_segment(ims)
    res = det.im_segment(ims, render=True, vis_thresh=vis_thresh)
    drawn = 0
    for r, p, im in zip(res, plain, ims):
        H, W = im.shape[:2]
        _assert_same(r, p)                                   # vis_thresh filters the drawing only
        assert r["inst"].shape == r["cls"].shape == (H, W) and r["bgr"].shape == (H, W, 3)
        assert r["inst"].dtype == r["cls"].dtype == np.int32 and r["bgr"].dtype == np.uint8
        inst, cls, bgr = _display_reference(_vote_dict(r), H, W, vis_thresh)
        assert np.array_equal(r["inst"], inst) and np.array_equal(r["cls"], cls)
        assert np.array_equal(r["bgr"], bgr)
        # and the reference's demo flow on the per-class lists
        list_mask, list_box = unpack_voting(r)
        pred = get_vis_dict(list_box, list_mask, "x", ["c%d" % i for i in range(20)], vis_thresh=vis_thresh)
        w_inst, w_cls = _convert_pred_to_image(W, H, pred)
        assert np.array_equal(r["inst"], w_inst) and np.array_equal(r["cls"], w_cls)
        drawn += int(r["inst"].max())
    if vis_thresh == 0.0:
        assert drawn > 0
    if vis_thresh > 1:
        assert drawn == 0


def _hand_built_votes(sizes, n_res, R=40, seed=5):
    """Voting outputs of len(sizes) images: boxes integer, many touching or crossing the image
    border, scores uniform in [0, 1) (some exactly 0.5), classes 1..20."""
    rng = np.random.default_rng(seed)
    B = len(sizes)
    box = np.zeros((B, R, 4), np.int32)
    for b, (H, W) in enumerate(sizes):
        x1, y1 = rng.integers(-10, W, R), rng.integers(-10, H, R)
        box[b] = np.stack([x1, y1, x1 + rng.integers(0, W // 2 + 2, R), y1 + rng.integers(0, H // 2 + 2, R)], 1)
        box[b, :4] = [[0, 0, W - 1, H - 1], [0, 5, 20, H - 1], [W - 30, 0, W - 1, 25], [W - 9, H - 9, W + 5, H + 3]]
    score = rng.uniform(0, 1, (B, R)).astype(np.float32)
    score[:, 5] = 0.5
    vote = dict(n_res=torch.tensor(n_res, dtype=torch.int32),
                res_score=torch.from_numpy(score),
                res_class=torch.from_numpy(rng.integers(1, 21, (B, R)).astype(np.int32)),
                result_box=torch.from_numpy(box),
                result_mask=torch.from_numpy((1 / (1 + np.exp(-rng.normal(0, 2, (B, R, 1, 21, 21))))).astype(np.float32)))
    return {k: v.cuda() for k, v in vote.items()}


@pytest.mark.parametrize("vis_thresh", [0.0, 0.5, 1.01])
def test_ragged_paste_kernel_equals_select_and_paste_per_image(vis_thresh):
    """Images of different widths and heights (one tiny, one taller than wide), one with no
    results; boxes touching and crossing the border; a score equal to the threshold."""
    from mnc_b200 import ops
    sizes = [(375, 500), (500, 333), (21, 33), (130, 700)]
    n_res = [40, 0, 17, 33]
    vote = _hand_built_votes(sizes, n_res)
    hw = torch.tensor(sizes, dtype=torch.int32).cuda()
    pix = [h * w for h, w in sizes]
    off = np.concatenate([[0], np.cumsum(pix)[:-1]]).astype(np.int64)
    P = sum(pix)
    inst = torch.full((P,), -1, dtype=torch.int32, device="cuda")
    cls = torch.full((P,), -1, dtype=torch.int32, device="cuda")
    bgr = torch.full((3 * P,), 7, dtype=torch.uint8, device="cuda")
    ops.paste_voted_ragged(vote, hw, torch.from_numpy(off).cuda(), (500, 700), inst, cls, bgr, vis_thresh=vis_thresh)
    inst, cls, bgr = inst.cpu().numpy(), cls.cpu().numpy(), bgr.cpu().numpy()
    for b, (H, W) in enumerate(sizes):
        one = {k: v[b:b + 1] for k, v in vote.items()}
        w_inst, w_cls, w_bgr = _display_reference(one, H, W, vis_thresh)
        o = off[b]
        assert np.array_equal(inst[o:o + H * W].reshape(H, W), w_inst), b
        assert np.array_equal(cls[o:o + H * W].reshape(H, W), w_cls), b
        assert np.array_equal(bgr[3 * o:3 * (o + H * W)].reshape(H, W, 3), w_bgr), b
        kept = int((vote["res_score"][b, :n_res[b]] >= vis_thresh).sum())
        assert w_inst.max() <= kept
        if n_res[b] == 0 or vis_thresh > 1:
            assert not w_inst.any() and not w_cls.any()


def test_stream_equals_blocking_calls_and_recomputes_a_batch_out_of_range():
    from oracle import oracle as O
    from tests.test_gpu_mixed_sizes import _low_contrast
    from mnc_b200.api import Detector
    w = _weights()
    ims = _mix()
    arr = np.stack([O.synthetic_image(10 + i, 375, 500) for i in range(2)])
    arr2 = O.synthetic_image(20, 480, 640)[None]
    seq = [ims, arr, ims[:3], arr2, list(reversed(ims))]
    det = Detector(w, max_batch=8)
    got = [r for r in det.im_segment_stream(seq, render=True, vis_thresh=0.0)]
    assert len(got) == len(seq)
    for batch, g in zip(seq, got):
        want = det.im_segment(batch, render=True, vis_thresh=0.0)
        assert len(g) == len(want)
        for a, b in zip(g, want):
            _assert_same(a, b, ("boxes", "scores", "classes", "masks", "scale", "inst", "cls", "bgr"))

    low = [_low_contrast(im) for im in ims]
    fresh = Detector(w).im_segment(ims)
    det2 = Detector(w)
    res = list(det2.im_segment_stream([low, ims]))
    assert sum(e.range_violations for e in det2._engines if e is not None) == 1
    for a, b in zip(res[1], fresh):
        _assert_same(a, b)
    det3 = Detector(w)
    det3.im_segment(low)
    v0 = det3.engine.range_violations
    res3 = det3.im_segment(ims)
    assert det3.engine.range_violations == v0 + 1
    for a, b in zip(res3, fresh):
        _assert_same(a, b)


def test_mask_voting_into_record_views_equals_fresh_tensors():
    from mnc_b200 import ops
    from tests.util import random_boxes
    rng = np.random.default_rng(31)
    B, nb, H, W, R = 2, 300, 375, 500, 128
    boxes = torch.from_numpy(np.stack([random_boxes(nb, 31 + b, W, H) for b in range(B)])).cuda()
    masks = torch.from_numpy((1 / (1 + np.exp(-rng.normal(0, 2, (B, nb, 1, 21, 21))))).astype(np.float32)).cuda()
    logits = rng.normal(0, 2.5, (B, nb, 21))
    scores = torch.from_numpy((np.exp(logits) / np.exp(logits).sum(-1, keepdims=True)).astype(np.float32)).cuda()
    valid = torch.ones((B, nb), dtype=torch.uint8).cuda()
    valid[1, 250:] = 0
    hw = torch.tensor([[H, W]] * B, dtype=torch.int32).cuda()
    want = ops.mask_voting(boxes, masks, scores, hw, max_results=R, box_valid=valid)
    rec = torch.full((ops.vote_record_layout(B, R)[-1],), -7, dtype=torch.int32, device="cuda")  # dirty
    views = ops.vote_record_views(rec, B, R)
    got = ops.mask_voting(boxes, masks, scores, hw, max_results=R, box_valid=valid, out=views)
    assert got["n_res"].data_ptr() == views["n_res"].data_ptr()
    n = want["n_res"].cpu()
    assert torch.equal(views["n_res"].cpu(), n) and int(n.min()) > 0
    assert int(views["overflow"][0]) == int(want["overflow"][0]) == 0
    for k in ("res_score", "result_box", "result_mask"):
        assert torch.equal(views[k].cpu(), want[k].cpu()), k
    for b in range(B):
        assert torch.equal(views["res_class"][b, :n[b]].cpu(), want["res_class"][b, :n[b]].cpu())
    # a record too small for the results: the flag is set, as without out=
    small = ops.vote_record_views(torch.empty(ops.vote_record_layout(B, 4)[-1], dtype=torch.int32,
                                              device="cuda"), B, 4)
    ops.mask_voting(boxes, masks, scores, hw, max_results=4, box_valid=valid, out=small)
    assert int(small["overflow"][0]) == 1 and small["n_res"].cpu().tolist() == [4, 4]


def test_small_voting_cap_takes_the_revote_path(monkeypatch):
    from mnc_b200 import ops
    from mnc_b200.api import Detector
    ims = _mix()
    det = Detector(_weights(), max_batch=8)
    want = det.im_segment(ims, render=True, vis_thresh=0.0)
    assert max(len(r["scores"]) for r in want) > 4
    calls = []
    vote = ops.mask_voting

    def spy(*a, **k):
        calls.append(k.get("max_results"))
        return vote(*a, **k)
    monkeypatch.setattr(ops, "mask_voting", spy)
    monkeypatch.setattr(ops, "default_vote_cap", lambda max_per_image: 4)
    got = det.im_segment(ims, render=True, vis_thresh=0.0)
    assert calls[0] == 4 and len(calls) > 1 and calls == sorted(calls)
    for a, b in zip(got, want):
        _assert_same(a, b, ("boxes", "scores", "classes", "masks", "scale", "inst", "cls", "bgr"))
    got = list(det.im_segment_stream([ims, ims]))       # both slots re-vote
    for a, b in zip(got[0] + got[1], want + want):
        _assert_same(a, b)


def test_d2h_bytes_are_the_voted_record():
    from oracle import oracle as O
    from mnc_b200 import ops
    from mnc_b200.api import Detector
    det = Detector(_weights(), max_batch=8)
    ims = np.stack([O.synthetic_image(i, 375, 500) for i in range(8)])
    det.im_segment(ims)
    rec = ops.vote_record_layout(8, 128)[-1] * 4
    assert det.d2h_bytes == rec + 512
    assert det.d2h_bytes < 1.84e6 < 8.9e6 < ops.record_layout(8, 300)[3] * 4
    det.im_segment(ims, render=True)
    assert det.d2h_bytes == rec + 512 + 8 * 375 * 500 * 11
