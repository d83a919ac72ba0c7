"""CPU tests of mixed-size batches: the per-level extent arithmetic, the padding argument in fp64,
and the host validation that runs before anything is launched."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F


def _caffe_pooled(n):
    """pooling_layer.cpp:90-93 for kernel 2, stride 2, pad 0 (ceil mode; the pad clip is inert)."""
    return int(np.ceil((n - 2) / 2.0)) + 1


def test_level_extent_is_caffes_chain_of_pooled_sizes():
    from mnc_b200.engine import level_extent
    for n in range(1, 1001):
        m = n
        for level in range(5):
            assert level_extent(n, level) == m, (n, level)
            m = _caffe_pooled(m) if m > 1 else 1
    # (a 1-pixel map pools to 1 pixel in Caffe as well: ceil(-1/2) + 1 = 1)
    assert _caffe_pooled(1) == 1


def _trunk64(w, x, ext=None):
    """fp64 TINY_ARCH trunk + rpn_conv_3x3.  ext: per-image (h, w) of a zero-padded batch -- then
    every layer zeroes pixels outside its image and pad pixels take no part in pool windows."""
    from mnc_b200.weights import TRUNK_NAMES, POOL_AFTER
    from mnc_b200.engine import level_extent

    def mask(y, level, fill=0.0):
        if ext is None:
            return y
        keep = torch.zeros(y.shape[0], 1, y.shape[2], y.shape[3], dtype=torch.bool)
        for b, (h, wd) in enumerate(ext):
            keep[b, :, :level_extent(h, level), :level_extent(wd, level)] = True
        return torch.where(keep, y, torch.full_like(y, fill))

    level = 0
    for name in TRUNK_NAMES + ["rpn_conv_3x3"]:
        wt, b = w[name]
        x = mask(F.relu(F.conv2d(x, wt.double(), b.double(), padding=1)), level)
        if name in POOL_AFTER:
            x = F.max_pool2d(mask(x, level, -np.inf), 2, 2, ceil_mode=True)
            level += 1
            x = mask(x, level)
    return x, level


def test_padding_with_per_layer_masking_reproduces_each_image_alone_fp64():
    from mnc_b200 import weights as Wt
    from mnc_b200.engine import level_extent
    w = Wt.make_weights(Wt.TINY_ARCH)
    sizes = [(37, 53), (50, 29), (1, 7), (50, 53), (33, 1)]
    H, W = max(s[0] for s in sizes), max(s[1] for s in sizes)
    g = torch.Generator().manual_seed(0)
    blob = torch.zeros(len(sizes), 3, H, W, dtype=torch.float64)
    alone = []
    for b, (h, wd) in enumerate(sizes):
        im = torch.randn(1, 3, h, wd, generator=g, dtype=torch.float64) * 50
        blob[b, :, :h, :wd] = im[0]
        alone.append(_trunk64(w, im)[0])
    got, level = _trunk64(w, blob, sizes)
    for b, (h, wd) in enumerate(sizes):
        h5, w5 = level_extent(h, level), level_extent(wd, level)
        ref = alone[b][0]
        assert ref.shape[1:] == (h5, w5)
        err = (got[b, :, :h5, :w5] - ref).abs().max() / ref.abs().max().clamp_min(1e-300)
        assert err < 1e-12, (sizes[b], float(err))
        assert not got[b, :, h5:, :].any() and not got[b, :, :, w5:].any()
    # without the masking, padding changes the result (bias + ReLU makes the pad non-zero)
    plain, _ = _trunk64(w, blob)
    h, wd = sizes[0]
    assert not torch.allclose(plain[0, :, :level_extent(h, 4), :level_extent(wd, 4)], alone[0][0],
                              rtol=1e-6, atol=0)


def test_host_validation_rejects_bad_extents_before_any_launch():
    from mnc_b200.engine import check_extents
    ok = check_extents([[600, 800], [901, 600]], 901, 800)
    assert ok.dtype == torch.int32 and ok.tolist() == [[600, 800], [901, 600]]
    for bad in ([[902, 800]], [[600, 801]], [[0, 800]], [[600, 0]], [[-1, 5]]):
        with pytest.raises(ValueError):
            check_extents(bad, 901, 800)
    with pytest.raises(ValueError):
        check_extents(np.zeros((0, 2), np.int32), 10, 10)
    with pytest.raises(ValueError):
        check_extents([[1, 2, 3]], 10, 10)
    with pytest.raises(ValueError):
        check_extents([[1.5, 2]], 10, 10)
    with pytest.raises(ValueError):
        check_extents([[5, 5]] * 9, 10, 10, max_batch=8)


def test_detector_mixed_batch_host_side():
    """Detector._mixed_batch (the host half of im_detect_mixed): scales by the 600/1000 rule,
    blob = the largest scaled sizes, byte offsets of the packed frames, and rejection of too many
    images or non-image arrays before anything reaches the device."""
    from mnc_b200.api import Detector
    d = Detector.__new__(Detector)       # host-side method only: no engine, no device buffers
    d.max_batch = 8
    ims = [np.zeros((357, 500, 3), np.uint8), np.zeros((375, 500, 3), np.uint8),
           np.zeros((500, 333, 3), np.uint8)]
    mb = d._mixed_batch(ims)
    assert mb["dst_hw"].tolist() == [[600, 840], [600, 800], [901, 600]]
    assert (mb["H"], mb["W"]) == (901, 840)
    assert mb["offsets"].tolist() == [0, 357 * 500 * 3, (357 + 375) * 500 * 3]
    assert mb["ext"].tolist() == mb["dst_hw"].tolist()
    with pytest.raises(ValueError):
        d._mixed_batch(ims * 3)                                   # 9 > max_batch
    with pytest.raises(ValueError):
        d._mixed_batch([])
    with pytest.raises(ValueError):
        d._mixed_batch([np.zeros((10, 10), np.uint8)])
    with pytest.raises(ValueError):
        d._mixed_batch([np.zeros((10, 10, 3), np.float32)])
