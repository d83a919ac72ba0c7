"""Precision mode 1 ("f16f8", tri-plane activations) where it can go wrong.

Kernel level: the kernels only the tri-plane path runs -- RoI warp, MaskPooling and the split-K
reduction with tri-plane outputs, tri-plane split-K at the engine's own shapes, the two halves of
the Concat buffer, the epilogue's published maximum -- each against an fp64 reference of the same
operation.  Engine level: the exponents are measured on the first input and then frozen, so inputs
other than the calibration input must still match the oracle, and a batch that outgrows the
exponents must come out as if the engine had been calibrated on it.

"Storage bound": the two precise planes carry a value to 2^-15 of the tensor maximum
(tests/test_gpu_round2.py::test_tri_conversion_device_equals_torch_restatement)."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests.test_gpu_roi import _rois
from tests.test_tri_headroom import SCALES, _monitor_accepts, format_table

pytestmark = pytest.mark.gpu
STORAGE = 2.0 ** -15
DEMO = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "demo")


def relerr(a, b):
    return ((a.double() - b.double()).abs().max() / b.double().abs().max()).item()


def _sentinel_tri(shape, byte=0x5A):
    from mnc_b200 import dense
    t = dense.tri_alloc(shape, "cuda")
    for p in (t.h, t.l, t.c):
        p.view(torch.uint8).fill_(byte)
    return t


def _planes_equal(a, b):
    return all(torch.equal(getattr(a, p).view(torch.uint8), getattr(b, p).view(torch.uint8)) for p in "hlc")


# --------------------------------------------------------------------------- A.1 RoI warp, tri out
@pytest.mark.parametrize("C", [512, 80])
@pytest.mark.parametrize("sub", [2, 1])
def test_roi_warp_tri(sub, C):
    """roi_warp_split_kernel<SUB, true> == oracle ROIWarping (+ 2x2 max) -> 14x14 and 7x7, on both
    images of a batch, with the edge RoIs (whole image, degenerate, partly / entirely outside,
    past the far edge, round-half, malformed)."""
    from oracle import oracle as O
    from mnc_b200 import dense, ops
    rng = np.random.default_rng(11 + C)
    H, W = 38, 63
    feat = np.maximum(rng.normal(size=(2, C, H, W)), 0).astype(np.float32)
    r = _rois(16, 5)
    r1 = r.copy()
    r1[:, 0] = 1
    rois = np.vstack([r, r1])                    # the seven edge RoIs on each image
    R = rois.shape[0]
    c5f = torch.from_numpy(feat).cuda().permute(0, 2, 3, 1).contiguous()
    exp = dense.exp_for(float(c5f.abs().max()))     # as MNCEngine.conv5_f32 sets "roi_feat"
    o14, o7 = _sentinel_tri((R, 14, 14, C)), _sentinel_tri((R, 7, 7, C))
    d_rois = torch.from_numpy(rois).cuda()
    ops.roi_warp_tri(c5f, C, H, W, d_rois, sub, o14, o7, exp)
    want28 = torch.from_numpy(O.roi_warp(feat, rois, 14 * sub, 14 * sub))
    want14 = F.max_pool2d(want28, 2, 2) if sub == 2 else want28
    want7 = F.max_pool2d(want14, 2, 2)
    assert o14.exp == o7.exp == exp
    got14 = o14.float().permute(0, 3, 1, 2).cpu()
    got7 = o7.float().permute(0, 3, 1, 2).cpu()
    assert torch.allclose(got14, want14, rtol=3e-5, atol=1e-6)
    assert torch.allclose(got7, want7, rtol=3e-5, atol=1e-6)
    for row in (3, 3 + 16):                      # entirely outside the map: exact zeros, all planes
        for o in (o14, o7):
            for p in (o.h, o.l, o.c):
                assert int(p[row].view(torch.uint8).abs().max()) == 0
    # an exponent 6 too high: h saturates at +-65504, never inf / NaN
    s14, s7 = _sentinel_tri((R, 14, 14, C)), _sentinel_tri((R, 7, 7, C))
    ops.roi_warp_tri(c5f, C, H, W, d_rois, sub, s14, s7, exp + 6)
    for o in (s14, s7):
        h = o.h.float()
        assert torch.isfinite(h).all() and float(h.abs().max()) == 65504.0
        assert torch.isfinite(o.float()).all()


# --------------------------------------------------------------------------- A.2 MaskPooling, tri
@pytest.mark.parametrize("C", [64, 512])
@pytest.mark.parametrize("R", [1, 37, 600])
def test_mask_pool_tri(R, C):
    from mnc_b200 import dense, ops
    g = torch.Generator(device="cuda").manual_seed(R * 7 + C)
    feat = torch.randn(R, 14, 14, C, device="cuda", generator=g)           # negatives: -FLT_MAX start
    ft = dense.tri_alloc(feat.shape, "cuda")
    dense.f32_to_tri(feat, ft, dense.exp_for(float(feat.abs().max())))
    mask = torch.rand(R, 1, 14, 14, device="cuda", generator=g)
    mask[:, :, 3, :] = 0.0                                                 # rows exactly 0 ...
    mask[:, :, 4, :] = 1.0                                                 # ... and exactly 1
    mask[0, :, 10:, :] = 0.0
    if R > 2:
        mask[1] = 0.0                                                      # a wholly empty mask
        mask[2] = 1.0
    out = _sentinel_tri((R, 7, 7, C))
    ops.mask_pool_tri(ft, mask, R, C, out)
    assert out.exp == ft.exp
    fq = ft.float().double().permute(0, 3, 1, 2)
    want = F.max_pool2d(fq * mask.double(), 2, 2).permute(0, 2, 3, 1)
    got = out.float().double()
    assert (got - want).abs().max() <= STORAGE * want.abs().max()


# --------------------------------------------------------------------------- A.3 split-K reduce, tri
@pytest.mark.parametrize("relu", [False, True])
@pytest.mark.parametrize("bias", [False, True])
@pytest.mark.parametrize("rows,cols", [(300, 256), (2400, 4096)])
@pytest.mark.parametrize("splits", [1, 2, 7, 9, 32])
def test_splitk_reduce_tri(splits, rows, cols, bias, relu):
    """Sum in split order + bias + ReLU, written into one half of a row of 2*cols tri-plane
    channels: planes bit-identical to the torch restatement of the conversion, the other half
    untouched, the published maximum that of the fp32 result.  (2400 x 4096 needs more CTAs than
    the 148 * 16 grid cap: the grid-stride loop runs.)"""
    from mnc_b200 import dense
    g = torch.Generator(device="cuda").manual_seed(splits * 1000 + cols + 2 * bias + relu)
    part = torch.randn(splits, rows, cols, device="cuda", generator=g)
    b = torch.randn(cols, device="cuda", generator=g) if bias else None
    acc = part[0].clone()
    for s in range(1, splits):
        acc = acc + part[s]
    if bias:
        acc = acc + b
    if relu:
        acc = acc.clamp_min(0)
    exp = dense.exp_for(float(acc.abs().max()))
    want = dense.tri_from_f32(acc, exp=exp)
    for off in (0, cols):
        out = _sentinel_tri((rows, 2 * cols))
        amax = torch.zeros(1, dtype=torch.int32, device="cuda")
        dense.splitk_reduce_tri(part, splits, rows * cols, rows, cols, out, exp, bias=b, relu=relu,
                                out_row_stride=2 * cols, out_ch_offset=off, amax=amax)
        torch.cuda.synchronize()
        mine = out[:, off:off + cols]
        assert _planes_equal(_contig(mine), want)
        other = slice(cols - off, 2 * cols - off)
        for p in (out.h, out.l, out.c):
            assert bool((p[:, other].view(torch.uint8) == 0x5A).all())
        assert float(amax.view(torch.float32)) == float(acc.abs().max())
        ref = part.double().sum(0) + (b.double() if bias else 0)
        if relu:
            ref = ref.clamp_min(0)
        assert (mine.float().double() - ref).abs().max() <= STORAGE * ref.abs().max()


def _contig(t):
    from mnc_b200 import dense
    return dense.Tri(t.h.contiguous(), t.l.contiguous(), t.c.contiguous(), t.exp)


# --------------------------------------------------------------------------- A.4 tri split-K, engine shapes
@pytest.mark.parametrize("layer,M", [("fc6_maskest", 300), ("fc6_maskest", 2400), ("fc6", 300)])
def test_tri_split_k_at_engine_shapes(layer, M):
    """Tri-plane operands with split-K partials, the way fc6_maskest and fc6 run: the split the
    engine picks on this device, weights through fc_weight_to_tri's (c,h,w) -> (h,w,c) permutation,
    and Caffe's inner product on the NCHW flattening with the UNPERMUTED weight as the reference."""
    from mnc_b200 import dense
    from mnc_b200.engine import MNCEngine, pick_split_k
    hw, N = {"fc6_maskest": (14, 256), "fc6": (7, 4096)}[layer]
    C = 512
    K = C * hw * hw
    bn = MNCEngine._fc_bn(N)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    split = pick_split_k(-(-M // 128), -(-N // bn), K // 64, sms, dense.cluster_size, 32, M * N)
    assert split > 1, split
    g = torch.Generator(device="cuda").manual_seed(M + N)
    x = torch.relu(torch.randn(M, hw, hw, C, device="cuda", generator=g))   # NHWC RoI features
    w = torch.randn(N, K, device="cuda", generator=g) * (2.0 / K) ** 0.5     # Caffe (N, c*h*w)
    b = torch.randn(N, device="cuda", generator=g) * 0.1
    xt = dense.tri_alloc((M, K), "cuda")
    dense.f32_to_tri(x.reshape(M, K), xt, dense.exp_for(float(x.max())))
    wt = dense.fc_weight_to_tri(w, (C, hw, hw))
    part = torch.empty(split, M, N, device="cuda")
    dense.igemm2(xt.view(1, 1, M, K), 1, 1, M, K, wt, N, 1, out_f32=part, split_k=split,
                 split_stride=M * N, bn=bn)
    x_nchw = x.permute(0, 3, 1, 2).reshape(M, K).double()
    ref = (x_nchw @ w.double().T + b.double()).clamp_min(0)
    del x, x_nchw
    out = dense.tri_alloc((M, N), "cuda")
    dense.splitk_reduce_tri(part, split, M * N, M, N, out, dense.exp_for(float(ref.max())), bias=b, relu=True)
    assert relerr(out.float(), ref) < 1e-4, (split, relerr(out.float(), ref))


# --------------------------------------------------------------------------- A.5 Concat join
def test_concat_join_halves_and_cls_head():
    """fc7 and fc7_mask write the two halves of one tri-plane join buffer with one exponent
    (channel offsets N and 0, row stride 2N); the cls head then reads the whole row (N = 126 fp32
    outputs in rows of 128) through the engine's own inner-product path."""
    from mnc_b200 import dense
    from mnc_b200.engine import MNCEngine
    R, fc = 300, 4096
    g = torch.Generator(device="cuda").manual_seed(5)
    h6, h6m = (torch.relu(torch.randn(R, fc, device="cuda", generator=g)) for _ in range(2))
    w7, w7m = (torch.randn(fc, fc, device="cuda", generator=g) * (2.0 / fc) ** 0.5 for _ in range(2))
    b7, b7m = (torch.randn(fc, device="cuda", generator=g) * 0.1 for _ in range(2))
    wc = torch.randn(126, 2 * fc, device="cuda", generator=g) * (1.0 / fc) ** 0.5
    bc = torch.randn(126, device="cuda", generator=g) * 0.1
    ref = torch.cat([(h6m.double() @ w7m.double().T + b7m.double()).clamp_min(0),
                     (h6.double() @ w7.double().T + b7.double()).clamp_min(0)], 1)
    join = _sentinel_tri((R, 2 * fc))
    e = dense.exp_for(float(ref.max()))
    for src, wgt, bias, off in ((h6, w7, b7, fc), (h6m, w7m, b7m, 0)):
        st = dense.tri_from_f32(src)
        dense.igemm2(st.view(1, 1, R, fc), 1, 1, R, fc, dense.fc_weight_to_tri(wgt), fc, 1, bias=bias,
                     relu=True, out=join, out_pix_stride=2 * fc, out_ch_offset=off,
                     bn=MNCEngine._fc_bn(fc), out_exp=e)
    assert join.exp == e
    assert relerr(join.float(), ref) < 1e-4
    assert relerr(join.float()[:, :fc], ref[:, :fc]) < 1e-4 and relerr(join.float()[:, fc:], ref[:, fc:]) < 1e-4
    eng = MNCEngine.__new__(MNCEngine)
    eng.impl, eng.device, eng._buf = "tc", torch.device("cuda"), {}
    eng.sms = torch.cuda.get_device_properties(0).multi_processor_count
    heads = torch.full((R, 128), 7.0, device="cuda")
    eng._linear(join, R, 2 * fc, dense.fc_weight_to_tri(wc), 126, bc, False, out_f32=heads,
                out_stride=128, key="cls")
    want = ref @ wc.double().T + bc.double()
    assert relerr(heads[:, :126], want) < 1e-4
    assert bool((heads[:, 126:] == 7.0).all())


# --------------------------------------------------------------------------- A.6 epilogue amax
_AMAX_LAYERS = [("fc", 300, 1, 1, 512, 256, False)] + [
    ("conv",) + shape + (pool,) for shape in ((1, 38, 63, 256, 256), (1, 75, 125, 64, 64), (1, 75, 125, 64, 128))
    for pool in (False, True)]


def _layer(kind, B, H, W, Cin, Cout, pool, seed, dist="relu_randn"):
    """(x fp32 (B,H,W,Cin) or (M,K), w fp32 Caffe layout, tri weight, fp64 reference fn)."""
    from mnc_b200 import dense
    g = torch.Generator(device="cuda").manual_seed(seed)
    if kind == "fc":
        shape = (B, Cin)
    else:
        shape = (B, H, W, Cin)
    x = torch.rand(shape, device="cuda", generator=g) if dist == "uniform" else \
        torch.relu(torch.randn(shape, device="cuda", generator=g))
    if kind == "fc":
        w = torch.randn(Cout, Cin, device="cuda", generator=g) * (2.0 / Cin) ** 0.5
        wt = dense.tri_from_f32(w, weight=True)
        ref = lambda xs: (xs.double() @ w.double().T).clamp_min(0)
    else:
        w = torch.randn(Cout, Cin, 3, 3, device="cuda", generator=g) * (2.0 / (9 * Cin)) ** 0.5
        wt = dense.conv_weight_to_tri(w)

        def ref(xs):
            y = F.relu(F.conv2d(xs.permute(0, 3, 1, 2).double(), w.double(), padding=1))
            if pool:
                y = F.max_pool2d(y, 2, 2, ceil_mode=True)
            return y.permute(0, 2, 3, 1)
    return x, wt, ref


def _run_layer(kind, x, wt, B, H, W, Cin, Cout, pool, e_in, e_out):
    """Input converted on the device with exponent e_in, layer run with output exponent e_out.
    -> (output Tri, input amax, output amax)."""
    from mnc_b200 import dense
    a_in = torch.zeros(1, dtype=torch.int32, device="cuda")
    a_out = torch.zeros(1, dtype=torch.int32, device="cuda")
    xt = dense.tri_alloc(x.shape, "cuda")
    dense.f32_to_tri(x.contiguous(), xt, e_in, amax=a_in)
    if kind == "fc":
        out = dense.tri_alloc((B, Cout), "cuda")
        dense.igemm2(xt.view(1, 1, B, Cin), 1, 1, B, Cin, wt, Cout, 1, relu=True, out=out, out_exp=e_out,
                     amax=a_out)
    else:
        Ho, Wo = ((H + 1) // 2, (W + 1) // 2) if pool else (H, W)
        out = dense.tri_alloc((B, Ho, Wo, Cout), "cuda")
        dense.igemm2(xt, B, H, W, Cin, wt, Cout, 9, relu=True, out=out, pool=pool, out_exp=e_out, amax=a_out)
    torch.cuda.synchronize()
    return out, float(a_in.view(torch.float32)), float(a_out.view(torch.float32))


@pytest.mark.parametrize("kind,B,H,W,Cin,Cout,pool", _AMAX_LAYERS)
def test_epilogue_amax(kind, B, H, W, Cin, Cout, pool):
    """The maximum the epilogue publishes (the range monitor's only input) is max |output| --
    also when the output exponent is so high that the stored planes saturate."""
    from mnc_b200 import dense
    x, wt, ref_fn = _layer(kind, B, H, W, Cin, Cout, pool, seed=H * W + Cout)
    ref = ref_fn(x)
    m = float(ref.abs().max())
    e_in = dense.exp_for(float(x.abs().max()))
    for e_out in (dense.exp_for(m), dense.exp_for(m) + 6):
        out, _, a_out = _run_layer(kind, x, wt, B, H, W, Cin, Cout, pool, e_in, e_out)
        assert abs(a_out - m) <= 1e-4 * m, (e_out, a_out, m)
    assert float(out.h.float().abs().max()) == 65504.0       # the last run did saturate


# --------------------------------------------------------------------------- A.7 headroom contract
_HEADROOM_LAYERS = [("fc", 512, 1, 1, 4608, 256, False), ("conv", 1, 38, 63, 256, 256, False),
                    ("conv", 1, 75, 125, 64, 64, False), ("conv", 1, 75, 125, 64, 64, True)]


@pytest.mark.parametrize("dist", ["uniform", "relu_randn"])
@pytest.mark.parametrize("kind,B,H,W,Cin,Cout,pool", _HEADROOM_LAYERS)
def test_headroom_contract(kind, B, H, W, Cin, Cout, pool, dist):
    """Exponents calibrated at s = 1, then inputs s times larger run with those stale exponents:
    whenever the engine's range monitor accepts both the input and the output maximum the kernels
    published, the layer is within 1e-4 of fp64."""
    from mnc_b200 import dense
    x, wt, ref_fn = _layer(kind, B, H, W, Cin, Cout, pool, seed=Cin * Cout + H, dist=dist)
    e_in = dense.exp_for(float(x.abs().max()))
    _, _, a1 = _run_layer(kind, x, wt, B, H, W, Cin, Cout, pool, e_in, 0)
    e_out = dense.exp_for(a1)
    rows = []
    for s in SCALES:
        xs = x * s
        out, a_in, a_out = _run_layer(kind, xs, wt, B, H, W, Cin, Cout, pool, e_in, e_out)
        err = relerr(out.float(), ref_fn(xs))
        rows.append((s, a_in * 2.0 ** e_in, a_out * 2.0 ** e_out, _monitor_accepts(a_in, e_in, a_out, e_out), err))
    table = "%s %dx%dx%d->%d%s, %s:\n%s" % (kind, B, H, W, Cout, " pooled" if pool else "", dist,
                                            format_table(rows))
    print("\n" + table)
    for s, _, _, ok, err in rows:
        if ok:
            assert err <= 1e-4, table
    assert all(ok for s, _, _, ok, _ in rows if s in (2.0 ** -10, 1, 2)), table


# --------------------------------------------------------------------------- C.8 off-calibration inputs
@pytest.fixture(scope="module")
def full_engine():
    from oracle import oracle as O
    from mnc_b200 import weights as Wt
    from mnc_b200.engine import MNCEngine
    w = Wt.make_weights(Wt.FULL_ARCH)
    eng = MNCEngine(w)
    blob0, info0 = O.prep_blob(O.synthetic_image(0, 600, 1000))
    eng.forward_checked(torch.from_numpy(blob0).cuda(), torch.from_numpy(info0).cuda())
    torch.cuda.synchronize()
    assert eng.range_violations == 0
    return dict(w=w, eng=eng, blob0=blob0, info0=info0)


def _natural(name):
    import cv2
    from oracle import oracle as O
    im = cv2.imread(os.path.join(DEMO, name + ".jpg"))
    assert im is not None
    x, scale = O.prep_im_for_blob(im)
    blob = x[None].transpose(0, 3, 1, 2).astype(np.float32).copy()
    info = np.array([[blob.shape[2], blob.shape[3], scale]], dtype=np.float32)
    return blob, info


# (times8 last: it is the one input that moves the exponents)
@pytest.mark.parametrize("which", ["synthetic1", "div16", "2008_000533", "2008_001602", "times8"])
def test_off_calibration_inputs_full_arch(full_engine, which):
    """One FULL_ARCH engine calibrated on synthetic image 0; every other input goes through the
    checked entry point and must pass the stage-wise oracle check.  /16 stays in range (exponents
    unchanged); x8 puts every trunk maximum above 2^14 and recalibrates exactly once."""
    from oracle import oracle as O
    from tests.test_gpu_e2e import _check_stagewise
    eng, w = full_engine["eng"], full_engine["w"]
    if which == "synthetic1":
        blob, info = O.prep_blob(O.synthetic_image(1, 600, 1000))
    elif which == "div16":
        blob, info = full_engine["blob0"] / 16, full_engine["info0"]
    elif which == "times8":
        blob, info = full_engine["blob0"] * 8, full_engine["info0"]
    else:
        blob, info = _natural(which)
    blob = np.ascontiguousarray(blob, dtype=np.float32)
    exp_before, n_before = dict(eng.exp), eng.range_violations
    out = eng.forward_checked(torch.from_numpy(blob).cuda(), torch.from_numpy(info).cuda(), keep_intermediate=True)
    torch.cuda.synchronize()
    print("\n%s: %d recalibration(s)" % (which, eng.range_violations - n_before))
    if which == "times8":
        assert eng.range_violations == n_before + 1
        assert any(eng.exp[k] != exp_before[k] for k in exp_before)
    elif which == "div16":
        assert eng.range_violations == n_before and eng.exp == exp_before
    _check_stagewise(w, blob, info, eng, out, 0)


# --------------------------------------------------------------------------- C.9 blank first frame
BLANK = (103, 116, 123)     # the pixel means: a blob within 0.25 of zero


def _frames():
    from oracle import oracle as O
    blank = np.empty((2, 375, 500, 3), np.uint8)
    blank[...] = BLANK
    real = [np.stack([O.synthetic_image(20 + 10 * k + i, 375, 500) for i in range(2)]) for k in range(2)]
    return blank, real


def _copy(res):
    return [np.array(a, copy=True) for a in res[:4]]


def _assert_same(a, b):
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


@pytest.fixture(scope="module")
def tiny_weights():
    from mnc_b200 import weights as Wt
    return Wt.make_weights(Wt.TINY_ARCH)


@pytest.mark.parametrize("mode", ["images_graphed", "images_eager", "batch"])
def test_blank_first_frame_detector(tiny_weights, mode):
    """A first call on blank frames sets every exponent far too high; the next real batch must be
    detected, re-measured and recomputed so that its results equal, bit for bit, those of a
    Detector whose first call was that batch."""
    from mnc_b200.api import Detector
    from oracle import oracle as O
    blank, real = _frames()
    graph = mode != "images_eager"

    def call(det, frames):
        if mode == "batch":
            blob = np.concatenate([O.prep_blob(im)[0] for im in frames])
            return _copy(det.im_detect_batch(blob))
        return _copy(det.im_detect_images(frames))

    fresh = Detector(tiny_weights, max_batch=2, height=375, width=500, use_graph=graph)
    want = [call(fresh, b) for b in real]
    det = Detector(tiny_weights, max_batch=2, height=375, width=500, use_graph=graph)
    call(det, blank)
    exp_blank = dict(det.engine.exp)
    got = [call(det, b) for b in real]
    assert det.engine.range_violations == 1
    assert det.engine.exp == fresh.engine.exp != exp_blank
    for a, b in zip(got, want):
        _assert_same(a, b)


def test_blank_first_frame_stream(tiny_weights):
    from mnc_b200.api import Detector
    blank, real = _frames()
    fresh = Detector(tiny_weights, max_batch=2, height=375, width=500)
    want = [_copy(r) for r in fresh.im_detect_stream(iter(real))]
    det = Detector(tiny_weights, max_batch=2, height=375, width=500)
    got = [_copy(r) for r in det.im_detect_stream(iter([blank] + real))]
    assert len(got) == 3 and len(want) == 2
    assert det.engine.exp == fresh.engine.exp
    for a, b in zip(got[1:], want):
        _assert_same(a, b)


def test_blank_first_frame_caffe_net(tiny_weights):
    import mnc_b200.lib as L
    L.install()
    import caffe
    from oracle import oracle as O
    caffe.set_mode_gpu()
    caffe.set_device(0)
    blank, real = _frames()

    def fwd(net, im):
        blob, info = O.prep_blob(im)
        net.blobs["data"].reshape(*blob.shape)
        net.blobs["im_info"].reshape(*info.shape)
        return {k: np.array(v, copy=True) for k, v in net.forward(data=blob, im_info=info).items()}

    want = fwd(caffe.Net(None, tiny_weights, caffe.TEST), real[0][0])
    net = caffe.Net(None, tiny_weights, caffe.TEST)
    fwd(net, blank[0])
    got = fwd(net, real[0][0])
    assert net._engine.range_violations == 1
    assert set(got) == set(want)
    for k in want:
        assert np.array_equal(got[k], want[k]), k
