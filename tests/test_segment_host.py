"""Host side of Detector.im_segment: the voted-result record (ops.vote_record_layout / views),
`api.unpack_voting` and the input validation that runs before anything reaches the device."""
import numpy as np
import pytest
import torch


def test_vote_record_layout_arithmetic():
    from mnc_b200 import ops
    for B, R, M in [(1, 1, 21), (3, 7, 21), (8, 128, 21), (5, 256, 14)]:
        oo, oc, os_, ob, om, end = ops.vote_record_layout(B, R, M)
        assert oo >= B and oc >= oo + 1 and os_ >= oc + B * R and ob >= os_ + B * R
        assert om == ob + B * R * 4 and end == om + B * R * M * M
        assert all(o % 4 == 0 for o in (oo, oc, os_, ob, om))       # 16-byte aligned sections
        assert ob - B * R * 2 - B - 1 <= 4 * 3                      # padding only for alignment
    # batch 8, 128 result slots: 1.83 MB back instead of the 600-row record's 8.95 MB
    assert ops.vote_record_layout(8, 128)[-1] * 4 == pytest.approx(1.83e6, rel=2e-3)
    assert ops.record_layout(8, 300)[3] * 4 == pytest.approx(8.95e6, rel=2e-3)


def test_vote_record_views_share_one_buffer():
    from mnc_b200 import ops
    B, R, M = 3, 5, 21
    rec = torch.zeros(ops.vote_record_layout(B, R, M)[-1], dtype=torch.int32)
    v = ops.vote_record_views(rec, B, R, M)
    assert v["n_res"].dtype == torch.int32 and v["res_score"].dtype == torch.float32
    assert v["result_box"].shape == (B, R, 4) and v["result_mask"].shape == (B, R, 1, M, M)
    v["n_res"][:] = torch.tensor([5, 0, 2], dtype=torch.int32)
    v["overflow"][0] = 1
    v["res_class"][2, 1] = 7
    v["res_score"][2, 1] = 0.75
    v["result_box"][2, 1] = torch.tensor([1, 2, 3, 4], dtype=torch.int32)
    v["result_mask"][2, 1, 0, 20, 20] = 0.5
    oo, oc, os_, ob, om, end = ops.vote_record_layout(B, R, M)
    assert rec[:B].tolist() == [5, 0, 2] and rec[oo] == 1
    assert rec[oc + 2 * R + 1] == 7
    assert rec[os_ + 2 * R + 1].view(torch.int32) == torch.tensor(0.75).view(torch.int32)
    assert rec[ob + (2 * R + 1) * 4:ob + (2 * R + 2) * 4].tolist() == [1, 2, 3, 4]
    assert rec[end - 1 - (R - 2) * M * M].view(torch.float32) == 0.5
    # a float32 record gives the same views (integers as bit patterns)
    v2 = ops.vote_record_views(rec.view(torch.float32), B, R, M)
    assert torch.equal(v2["res_class"], v["res_class"]) and torch.equal(v2["result_mask"], v["result_mask"])


def _hand_built(seed=3, B=2, R=9, M=21):
    from mnc_b200 import ops
    rng = np.random.default_rng(seed)
    rec = torch.zeros(ops.vote_record_layout(B, R, M)[-1], dtype=torch.int32)
    v = ops.vote_record_views(rec, B, R, M)
    n = [6, 0]
    v["n_res"][:] = torch.tensor(n, dtype=torch.int32)
    v["res_class"][0, :6] = torch.tensor([2, 2, 5, 9, 9, 9], dtype=torch.int32)
    v["res_score"][0, :6] = torch.from_numpy(rng.uniform(0, 1, 6).astype(np.float32))
    v["result_box"][0, :6] = torch.from_numpy(rng.integers(0, 500, (6, 4)).astype(np.int32))
    v["result_mask"][0, :6] = torch.from_numpy(rng.uniform(0, 1, (6, 1, M, M)).astype(np.float32))
    v["res_class"][0, 6:] = 3        # past n_res: not results
    return v, n


def test_unpack_voting_hand_built():
    from mnc_b200.api import unpack_voting
    v, n = _hand_built()
    k = n[0]
    res = dict(boxes=v["result_box"][0, :k].numpy(), scores=v["res_score"][0, :k].numpy(),
               classes=v["res_class"][0, :k].numpy(), masks=v["result_mask"][0, :k, 0].numpy())
    list_mask, list_box = unpack_voting(res)
    assert len(list_mask) == len(list_box) == 20
    for c, rows in [(2, [0, 1]), (5, [2]), (9, [3, 4, 5])]:
        want_box = np.hstack((res["boxes"][rows].astype(np.float32), res["scores"][rows, None]))
        assert list_box[c - 1].dtype == np.float32 and np.array_equal(list_box[c - 1], want_box)
        assert np.array_equal(list_mask[c - 1], res["masks"][rows][:, None])
    for c in set(range(1, 21)) - {2, 5, 9}:
        assert list_box[c - 1].shape == (0, 5) and list_mask[c - 1].shape == (0, 1, 21, 21)
    # the batched dict of ops.mask_voting: one pair per image, the same pairs
    per_image = unpack_voting(v)
    assert len(per_image) == 2
    for a, b in zip(per_image[0][0] + per_image[0][1], list_mask + list_box):
        assert np.array_equal(a, b)
    assert all(x.shape[0] == 0 for x in per_image[1][0] + per_image[1][1])
    # the name TesterWrapper has always exported is this function
    import mnc_b200.lib as L
    L.install()
    from caffeWrapper.TesterWrapper import unpack_voting as tw_unpack
    assert tw_unpack is unpack_voting


def _detector(max_batch=2):
    """A Detector without an engine: im_segment validates its input before it touches the device
    (the engine and buffers are never reached)."""
    from mnc_b200.api import Detector
    det = Detector.__new__(Detector)
    det.max_batch = max_batch
    det.device = torch.device("cpu")
    return det


@pytest.mark.parametrize("images", [
    [],                                                              # empty list
    [np.zeros((20, 30, 3), np.uint8)] * 3,                           # more than max_batch images
    [np.zeros((20, 30, 3), np.float32)],                             # not uint8
    [np.zeros((20, 30, 4), np.uint8)],                               # not BGR
    [np.zeros((20, 30), np.uint8)],                                  # not BGR
    np.zeros((3, 20, 30, 3), np.uint8),                              # array batch over max_batch
    np.zeros((0, 20, 30, 3), np.uint8),                              # empty array batch
    np.zeros((2, 20, 30, 3), np.float32),                            # array batch not uint8
    np.zeros((2, 20, 30, 1), np.uint8),                              # array batch not BGR
    torch.zeros((2, 20, 30, 3), dtype=torch.int16),                  # tensor batch not uint8
])
def test_im_segment_rejects_bad_input(images):
    det = _detector()
    with pytest.raises(ValueError):
        det.im_segment(images)
    with pytest.raises(ValueError):
        next(iter(det.im_segment_stream([images], render=True)))
