"""Mixed-size batches on the GPU: every kernel that takes per-image extents, checked bit for bit
against the same kernel on each image's cropped tensor, then the engine and the public API against
each image run alone."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

DEMO = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "demo")
# odd extents, a 1-pixel-high and a 1-pixel-wide image, and one that fills the blob
SIZES = [(37, 53), (1, 53), (50, 1), (50, 53), (23, 17)]


def _ext(sizes, level=0):
    """Input-resolution sizes whose extents at `level` are `sizes` (h -> h * 2^level - (2^level - 1))."""
    m = (1 << level) - 1
    return torch.tensor([[(h << level) - m, (w << level) - m] for h, w in sizes], dtype=torch.int32).cuda()


def _padded(sizes, C, seed, pad=0.0):
    """(B, H, W, C) fp32: random inside each image's extent, `pad` outside."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    H, W = max(s[0] for s in sizes), max(s[1] for s in sizes)
    x = torch.full((len(sizes), H, W, C), pad, device="cuda")
    for b, (h, w) in enumerate(sizes):
        x[b, :h, :w] = torch.rand(h, w, C, generator=g, device="cuda") * 4 - 1
    return x


def _planes(t):
    from mnc_b200 import dense
    if isinstance(t, dense.Tri):
        return [t.h.view(torch.int16), t.l, t.c]
    return [t[0].view(torch.int16), t[1].view(torch.int16)]


def _alloc(tri, shape, exp=0):
    from mnc_b200 import dense
    if tri:
        o = dense.tri_alloc(shape, "cuda", exp)
        for p in (o.h.view(torch.uint8), o.l, o.c):
            p.fill_(0x55)                   # stale bytes: the kernels must write the zeros
        return o
    o = torch.empty((2,) + tuple(shape), dtype=torch.bfloat16, device="cuda")
    o.view(torch.int16).fill_(0x5555)
    return o


def _act(x, tri):
    from mnc_b200 import dense
    return dense.tri_from_f32(x, 0) if tri else dense.split(x)


def _check_crops(got, want_fn, sizes):
    """got: planes of the batched output (B, h, w, C); want_fn(b) the planes of image b alone."""
    for b, (h, w) in enumerate(sizes):
        for pg, pw in zip(got, want_fn(b)):
            assert torch.equal(pg[b, :h, :w], pw[0]), (b, h, w)
            inside = torch.zeros_like(pg[b], dtype=torch.bool)
            inside[:h, :w] = True
            assert not pg[b][~inside].any(), (b, "outside the image must be exact zeros")


def _conv(x, tri, B, H, W, cin, wgt, cout, bias, pool, split, ext=None, level=0, exp=3):
    from mnc_b200 import dense
    Ho, Wo = ((H + 1) // 2, (W + 1) // 2) if pool else (H, W)
    out = _alloc(tri, (B, Ho, Wo, cout), exp)
    if split == 1:
        dense.igemm2(x, B, H, W, cin, wgt, cout, 9, bias=bias, relu=True, out=out, pool=pool,
                     out_exp=exp, img_hw=ext, level=level)
        return out
    M = B * H * W
    part = torch.empty((split, M, cout), dtype=torch.float32, device="cuda")
    dense.igemm2(x, B, H, W, cin, wgt, cout, 9, out_f32=part, split_k=split, split_stride=M * cout)
    if tri:
        dense.splitk_reduce_tri(part, split, M * cout, M, cout, out, exp, bias=bias, relu=True,
                                img_hw=ext, level=level, map_hw=(H, W))
    else:
        dense.splitk_reduce(part, split, M * cout, M, cout, bias=bias, relu=True, out=out,
                            img_hw=ext, level=level, map_hw=(H, W))
    return out


CONV_CASES = [  # (tri, cout, pool, split, halo pair)
    (True, 64, False, 1, True), (True, 64, True, 1, True), (True, 128, True, 1, False),
    (True, 64, False, 1, False), (True, 256, False, 1, True), (True, 256, True, 1, True),
    (False, 128, False, 1, True), (False, 64, True, 1, True), (False, 256, False, 1, True),
    (False, 256, True, 1, True), (True, 256, False, 3, True), (False, 256, False, 2, True),
]


@pytest.mark.parametrize("tri,cout,pool,split,pair", CONV_CASES)
@pytest.mark.parametrize("level", [0, 2])
def test_conv_with_extents_equals_cropped(tri, cout, pool, split, pair, level):
    _conv_case(tri, cout, pool, split, pair, level)


@pytest.mark.parametrize("cout", [64, 256])
def test_conv_direct_store_with_extents_equals_cropped(cout):
    """The epilogue's direct-store branch (split-bf16 out_mode 0 without the TMA store)."""
    from mnc_b200 import dense
    dense.set_tma_store(False)
    try:
        _conv_case(False, cout, False, 1, True, 1)
    finally:
        dense.set_tma_store(True)


def _conv_case(tri, cout, pool, split, pair, level):
    from mnc_b200 import dense
    cin = 64
    g = torch.Generator(device="cuda").manual_seed(cout + 7 * split)
    wf = torch.randn(cout, cin, 3, 3, generator=g, device="cuda") * 0.05
    wgt = dense.conv_weight_to_tri(wf) if tri else dense.conv_weight_to_split(wf)
    bias = torch.randn(cout, generator=g, device="cuda") * 0.3
    xf = _padded(SIZES, cin, seed=cout)
    B, H, W = xf.shape[:3]
    dense.set_halo_pair(pair)
    try:
        ext = _ext(SIZES, level)
        got = _conv(_act(xf, tri), tri, B, H, W, cin, wgt, cout, bias, pool, split, ext, level)

        def alone(b):
            h, w = SIZES[b]
            xb = xf[b:b + 1, :h, :w].contiguous()
            return _planes(_conv(_act(xb, tri), tri, 1, h, w, cin, wgt, cout, bias, pool, split))
        osz = [((h + 1) // 2, (w + 1) // 2) if pool else (h, w) for h, w in SIZES]
        _check_crops(_planes(got), alone, osz)
        # full extents are the whole-blob launch
        full = torch.tensor([[H << level, W << level]] * B, dtype=torch.int32, device="cuda")
        a = _planes(_conv(_act(xf, tri), tri, B, H, W, cin, wgt, cout, bias, pool, split, full, level))
        b_ = _planes(_conv(_act(xf, tri), tri, B, H, W, cin, wgt, cout, bias, pool, split))
        assert all(torch.equal(p, q) for p, q in zip(a, b_))
    finally:
        dense.set_halo_pair(True)


@pytest.mark.parametrize("tri", [True, False])
def test_conv1_1_tc_with_extents_equals_cropped(tri):
    from mnc_b200 import dense
    g = torch.Generator(device="cuda").manual_seed(11)
    wf = torch.randn(64, 3, 3, 3, generator=g, device="cuda") * 0.1
    wst = dense.conv1_1_weight_to_tc(wf)
    bias = torch.randn(64, generator=g, device="cuda")
    x = _padded(SIZES, 3, seed=5).permute(0, 3, 1, 2).contiguous() * 100
    B, _, H, W = x.shape

    def run(data, ext=None):
        out = _alloc(tri, (data.shape[0], data.shape[2], data.shape[3], 64), 2)
        dense.conv1_1_tc(data, wst, bias, out, out_exp=2, img_hw=ext)
        return _planes(out)
    got = run(x, _ext(SIZES))
    _check_crops(got, lambda b: run(x[b:b + 1, :, :SIZES[b][0], :SIZES[b][1]].contiguous()), SIZES)
    full = torch.tensor([[H, W]] * B, dtype=torch.int32, device="cuda")
    assert all(torch.equal(p, q) for p, q in zip(run(x, full), run(x)))


def test_ragged_prep_equals_each_image_alone():
    import cv2
    from mnc_b200 import ops
    ims = [cv2.imread(os.path.join(DEMO, n + ".jpg")) for n in ("2008_000533", "2008_001602")]
    rng = np.random.default_rng(0)
    ims += [rng.integers(0, 256, size=s + (3,), dtype=np.uint8) for s in ((357, 500), (500, 333), (31, 77), (1, 9))]
    scales = [ops.im_scale_for(im.shape) for im in ims]
    dst = [ops.blob_size_for(im.shape, s) for im, s in zip(ims, scales)]
    H, W = max(d[0] for d in dst), max(d[1] for d in dst)
    offsets = np.concatenate([[0], np.cumsum([im.nbytes for im in ims])[:-1]])
    packed = torch.from_numpy(np.concatenate([im.reshape(-1) for im in ims])).cuda()
    blob, dst_hw = ops.prep_images_ragged(packed, offsets, [im.shape[:2] for im in ims], scales, H, W)
    assert dst_hw.tolist() == [list(d) for d in dst]
    for b, im in enumerate(ims):
        alone = ops.prep_images(torch.from_numpy(im[None].copy()).cuda(), scales[b])
        h, w = dst[b]
        assert alone.shape[2:] == (h, w)
        assert torch.equal(blob[b, :, :h, :w], alone[0])
        rest = blob[b].clone()
        rest[:, :h, :w] = 0
        assert not rest.any() and not torch.signbit(blob[b][:, h:, :]).any()


def test_proposals_with_extents_equal_cropped_maps():
    from mnc_b200 import ops
    from mnc_b200.engine import level_extent
    img = [(600, 1000), (600, 800), (450, 1000), (200, 333), (601, 17)]
    ext5 = [(level_extent(h, 4), level_extent(w, 4)) for h, w in img]
    B, H5, W5 = len(img), max(e[0] for e in ext5), max(e[1] for e in ext5)
    g = torch.Generator(device="cuda").manual_seed(3)
    rpn = torch.randn(B, H5, W5, 64, generator=g, device="cuda")
    rpn[..., 18:54] *= 0.2
    for b, (h5, w5) in enumerate(ext5):          # the padding would win every top-k if it counted
        rpn[b, h5:, :, 9:18] = 50.0
        rpn[b, :, w5:, 9:18] = 50.0
    info = torch.tensor([[h, w, 1.0] for h, w in img], dtype=torch.float32, device="cuda")
    ext = torch.tensor(img, dtype=torch.int32, device="cuda")
    kw = dict(pre_nms_top_n=6000, post_nms_top_n=300, nms_thresh=0.7, min_size=16.0, batch_index_mode=True)
    rois, counts = ops.proposals_from_rpn(rpn, None, info, B, H5, W5, "nhwc", True, img_hw=ext, level=4, **kw)
    for b, (h5, w5) in enumerate(ext5):
        r1, c1 = ops.proposals_from_rpn(rpn[b:b + 1, :h5, :w5].contiguous(), None, info[b:b + 1], 1, h5, w5,
                                        "nhwc", True, **kw)
        assert int(counts[b]) == int(c1[0]) > 0
        assert torch.equal(rois[b, :, 1:], r1[0, :, 1:]) and (rois[b, :int(counts[b]), 0] == b).all()


@pytest.mark.parametrize("tri", [True, False])
@pytest.mark.parametrize("sub", [1, 2])
def test_roi_warp_with_extents_equals_cropped_map(tri, sub):
    from mnc_b200 import dense, ops
    ext5 = [(13, 21), (38, 63), (1, 40), (25, 1)]
    img = [(h * 16, w * 16) for h, w in ext5]
    C = 64
    c5f = _padded(ext5, C, seed=9, pad=1e4)       # the padding must never be sampled
    B, H5, W5 = c5f.shape[:3]
    rng = np.random.default_rng(1)
    rois = []
    for b, (h, w) in enumerate(img):
        x1 = rng.uniform(-40, w, 12)
        y1 = rng.uniform(-40, h, 12)
        x2 = x1 + rng.uniform(0, 400, 12)
        y2 = y1 + rng.uniform(0, 400, 12)
        # samples in (H5_b - 0.5, H5_b) and beyond: boxes ending on and just past the image edge
        edge = np.array([[0, 0, w - 1, h - 1], [w - 30, h - 30, w + 7, h + 7], [0, h - 9, 20, h + 60]])
        bx = np.concatenate([np.stack([x1, y1, x2, y2], 1), edge]).astype(np.float32)
        rois.append(np.concatenate([np.full((len(bx), 1), b, np.float32), bx], 1))
    rois_t = torch.from_numpy(np.concatenate(rois)).cuda()
    R = rois_t.shape[0]
    ext = torch.tensor(img, dtype=torch.int32, device="cuda")

    def run(feat, rr, e=None):
        n = rr.shape[0]
        f14, b7 = _alloc(tri, (n, 14, 14, C), 4), _alloc(tri, (n, 7, 7, C), 4)
        if tri:
            ops.roi_warp_tri(feat, C, feat.shape[1], feat.shape[2], rr, sub, f14, b7, 4, img_hw=e)
        else:
            ops.roi_warp_split(feat, C, feat.shape[1], feat.shape[2], rr, sub, f14, b7, img_hw=e)
        return _planes(f14), _planes(b7)
    g14, g7 = run(c5f, rois_t, ext)
    start = 0
    for b, (h5, w5) in enumerate(ext5):
        n = len(rois[b])
        rb = rois_t[start:start + n].clone()
        rb[:, 0] = 0
        a14, a7 = run(c5f[b:b + 1, :h5, :w5].contiguous(), rb)
        for p, q in zip(g14 + g7, a14 + a7):
            assert torch.equal(p[start:start + n], q), b
        start += n
    assert start == R


# ---------------------------------------------------------------------------------- engine / API
def _demo_images():
    import cv2
    return [cv2.imread(os.path.join(DEMO, n + ".jpg")) for n in ("2008_000533", "2008_001602")]


def _mix():
    from oracle import oracle as O
    return [O.synthetic_image(i, h, w) for i, (h, w) in
            enumerate([(600, 800), (600, 840), (901, 600), (600, 1000)])] + _demo_images()


def _prep(ims):
    from mnc_b200 import ops
    scales = [ops.im_scale_for(im.shape) for im in ims]
    dst = [ops.blob_size_for(im.shape, s) for im, s in zip(ims, scales)]
    H, W = max(d[0] for d in dst), max(d[1] for d in dst)
    offsets = np.concatenate([[0], np.cumsum([im.nbytes for im in ims])[:-1]])
    packed = torch.from_numpy(np.concatenate([im.reshape(-1) for im in ims])).cuda()
    blob, dst_hw = ops.prep_images_ragged(packed, offsets, [im.shape[:2] for im in ims], scales, H, W)
    info = torch.tensor([[h, w, s] for (h, w), s in zip(dst, scales)], dtype=torch.float32).cuda()
    hw = torch.tensor([im.shape[:2] for im in ims], dtype=torch.float32).cuda()
    sc = torch.tensor(scales, dtype=torch.float32).cuda()
    return blob, info, hw, sc, torch.from_numpy(dst_hw).cuda()


@pytest.fixture
def pinned_split(monkeypatch):
    from mnc_b200.engine import MNCEngine
    monkeypatch.setattr(MNCEngine, "_pick_split", lambda self, *a, **k: 1)


@pytest.mark.parametrize("arch", ["TINY_ARCH", "FULL_ARCH"])
def test_engine_mixed_batch_is_bit_identical_to_each_image_alone(arch, pinned_split):
    from mnc_b200 import weights as Wt
    from mnc_b200.engine import MNCEngine
    eng = MNCEngine(Wt.make_weights(getattr(Wt, arch)))
    ims = _mix()
    blob, info, hw, sc, ext = _prep(ims)
    got = [t.cpu() for t in eng.detect(blob, info, hw, sc, extents=ext)[:4]]   # calibrates on the mix
    exp = dict(eng.exp)
    for b, im in enumerate(ims):
        ab, ai, ah, asc, _ = _prep([im])
        want = [t.cpu() for t in eng.detect(ab, ai, ah, asc)[:4]]
        for name, g, w in zip(("boxes", "masks", "scores", "valid"), got, want):
            assert torch.equal(g[b], w[0]), (arch, b, name)
        assert int(want[3][0].sum()) > 0
    assert eng.exp == exp
    with pytest.raises(NotImplementedError):
        MNCEngine(Wt.make_weights(Wt.TINY_ARCH), impl="simt").forward(blob, info, extents=ext)


def test_detector_mixed_api(pinned_split):
    from mnc_b200 import weights as Wt
    from mnc_b200.api import Detector
    det = Detector(Wt.make_weights(Wt.TINY_ARCH), max_batch=8)
    ims = _mix()
    out = det.im_detect_mixed(ims)
    boxes, masks, scores, valid, scales = [np.array(o, copy=True) for o in out]
    assert scales.shape == (len(ims),)
    for b, im in enumerate(ims):
        a = det.im_detect_images(im[None])
        for g, w in zip((boxes, masks, scores, valid), a[:4]):
            assert np.array_equal(g[b], w[0]), b
        assert a[4] == scales[b]
    # another size mix that pads to the same blob shape replays the same graph
    n_graphs = len(det.engine._graphs)
    other = list(reversed(ims))
    o2 = det.im_detect_mixed(other)
    assert len(det.engine._graphs) == n_graphs
    for b in range(len(ims)):
        assert np.array_equal(o2[2][b], scores[len(ims) - 1 - b])
    # the stream takes list batches (scales per image) and array batches alternately
    arr = np.stack([ims[0], ims[0]])
    want_arr = [np.array(o, copy=True) for o in det.im_detect_images(arr)[:4]]
    res = [tuple(np.array(o, copy=True) for o in r) for r in det.im_detect_stream([ims, arr, ims[:3], arr])]
    assert len(res) == 4
    for k in (0, 2):
        n = len(res[k][4])
        for g, w in zip(res[k][:3], (boxes, masks, scores)):
            assert np.array_equal(g, w[:n]), k
        assert np.array_equal(res[k][4], scales[:n])
    for k in (1, 3):
        for g, w in zip(res[k][:3], want_arr[:3]):
            assert np.array_equal(g, w), k
        assert np.ndim(res[k][4]) == 0


# ------------------------------------------------------------- unpinned split-K, against the oracle
class _F32(__import__("mnc_b200.dense", fromlist=["Tri"]).Tri):
    """An fp32 tensor where tests.test_gpu_e2e._check_stagewise expects a Tri / split activation."""
    __slots__ = ("x",)

    def __init__(self, x):
        self.x = x

    def float(self):
        return self.x


def _image_view(out, img, h5, w5, n_per=300):
    """Image `img` of a mixed-batch forward (keep_intermediate=True) as a batch-1 output on its own
    unpadded map: maps cropped to the image's level-4 extent, RoI rows of the image, batch index 0."""
    from mnc_b200 import dense
    sl = slice(img * n_per, (img + 1) * n_per)
    B, H5, W5 = out["_rpn_out"].shape[:3]
    p = out["_proposal"]
    v = {"_conv5_3": _F32(dense.merge(out["_conv5_3"])[img:img + 1, :h5, :w5].contiguous()),
         "_rpn_out": out["_rpn_out"][img:img + 1, :h5, :w5].contiguous(),
         "_proposal": dict(
             proposals=p["proposals"].view(B, H5, W5, 9, 4)[img:img + 1, :h5, :w5].reshape(1, -1, 4),
             scores=p["scores"].view(B, H5, W5, 9)[img:img + 1, :h5, :w5].reshape(1, -1),
             valid=p["valid"].view(B, H5, W5, 9)[img:img + 1, :h5, :w5].reshape(1, -1)),
         "roi_counts": out["roi_counts"][img:img + 1],
         "_feat14": _F32(dense.merge(out["_feat14"])[sl]),
         "_feat14_ext": _F32(dense.merge(out["_feat14_ext"])[sl])}
    for k in ("rois", "rois_ext"):
        v[k] = out[k][sl].clone()
        v[k][:, 0] = 0
    for k in ("_mask_logits", "mask_proposal", "seg_cls_prob", "cls_prob", "bbox_pred",
              "mask_proposal_ext", "seg_cls_prob_ext"):
        v[k] = out[k][sl]
    return v


@pytest.mark.parametrize("arch,which", [("TINY_ARCH", "pair"), ("TINY_ARCH", "mix"), ("FULL_ARCH", "pair")])
def test_engine_mixed_batch_unpinned_against_oracle(arch, which, monkeypatch):
    """Split-K as chosen in normal operation (at 2 images of 600x1000 / 600x800 the FULL_ARCH
    conv5_x launches split and go through the extents-aware split-K reduce): every image's conv5_3
    and RPN outputs are within 1e-4 of the image run alone, and the whole cascade of each padded
    image passes the stage-wise oracle check on its UNPADDED blob."""
    from oracle import oracle as O
    from mnc_b200 import dense, weights as Wt
    from mnc_b200.engine import MNCEngine, level_extent
    from tests import util
    from tests.test_gpu_e2e import _check_stagewise
    splits = []
    pick = MNCEngine._pick_split

    def spy(self, *a, **k):
        s_ = pick(self, *a, **k)
        splits.append((k.get("max_split"), s_))
        return s_
    monkeypatch.setattr(MNCEngine, "_pick_split", spy)
    w = Wt.make_weights(getattr(Wt, arch))
    eng = MNCEngine(w)
    ims = ([O.synthetic_image(7, 600, 1000), O.synthetic_image(8, 600, 800)] if which == "pair" else _mix())
    blob, info, hw, sc, ext = _prep(ims)
    out = eng.forward(blob, info, keep_intermediate=True, extents=ext)
    torch.cuda.synchronize()
    if arch == "FULL_ARCH":
        assert any(m == 4 and s_ > 1 for m, s_ in splits), "no conv launch was split"
    data = blob.cpu().numpy()
    info_h = info.cpu().numpy()
    for b, im in enumerate(ims):
        h, wd = int(info_h[b, 0]), int(info_h[b, 1])
        h5, w5 = level_extent(h, 4), level_extent(wd, 4)
        view = _image_view(out, b, h5, w5)
        ab, ai, _, _, _ = _prep([im])
        alone = eng.forward(ab, ai, keep_intermediate=True)
        torch.cuda.synchronize()
        assert util.rel_err(view["_conv5_3"].x.cpu().numpy(),
                            dense.merge(alone["_conv5_3"]).cpu().numpy()) < 1e-4, b
        assert util.rel_err(view["_rpn_out"][..., :54].cpu().numpy(),
                            alone["_rpn_out"][..., :54].cpu().numpy()) < 1e-4, b
        n = _check_stagewise(w, np.ascontiguousarray(data[b:b + 1, :, :h, :wd]), info_h[b:b + 1], eng,
                             view, 0)
        assert n > 50, (b, n)


# ------------------------------------------------------------- range check on a mixed batch
def _low_contrast(im):
    """The image squeezed 16x around the pixel means: activations ~16x smaller."""
    from mnc_b200.ops import PIXEL_MEANS
    x = (im.astype(np.float32) - 128.0) / 16.0 + np.asarray(PIXEL_MEANS, np.float32)
    return np.clip(np.rint(x), 0, 255).astype(np.uint8)


def test_mixed_batch_that_trips_the_range_check_is_recomputed():
    """A Detector calibrated on low-contrast images gets a mixed batch of normal ones: the range
    check fails, the batch is recomputed with exponents measured on it (graphs re-captured with the
    extents as a static input), and the results equal those of a fresh Detector whose first call is
    that batch -- through im_detect_mixed and through the two-slot stream."""
    from mnc_b200 import weights as Wt
    from mnc_b200.api import Detector
    w = Wt.make_weights(Wt.TINY_ARCH)
    ims = _mix()
    low = [_low_contrast(im) for im in ims]
    fresh = [np.array(o, copy=True) for o in Detector(w).im_detect_mixed(ims)]

    det = Detector(w)
    det.im_detect_mixed(low)
    v0 = det.engine.range_violations
    got = [np.array(o, copy=True) for o in det.im_detect_mixed(ims)]
    assert det.engine.range_violations == v0 + 1
    for name, g, f in zip(("boxes", "masks", "scores", "valid", "scales"), got, fresh):
        assert np.array_equal(g, f), name

    det2 = Detector(w)
    res = [tuple(np.array(o, copy=True) for o in r) for r in det2.im_detect_stream([low, ims])]
    assert sum(e.range_violations for e in det2._engines if e is not None) == 1
    for name, g, f in zip(("boxes", "masks", "scores"), res[1][:3], fresh[:3]):
        assert np.array_equal(g, f), ("stream", name)
    assert np.array_equal(res[1][4], fresh[4])
