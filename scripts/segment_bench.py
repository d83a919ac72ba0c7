"""Throughput from host frames to host instances (voted masks) for images of different sizes
(FULL_ARCH weights; the seeded images, SIZES and batching policies of mixed_sizes_bench.py):

  (a) shape buckets through the step-by-step flow: engine.detect_checked + mask_voting_checked +
      unpack_voting (what scripts/demo.py and TesterWrapper did before Detector.im_segment);
  (b) shape buckets, Detector.im_segment per batch;
  (c) mixed batches grouped by orientation through Detector.im_segment_stream.

Prints the card name and power limit, then one JSON line per flow with images/s and the bytes
copied device -> host per batch.  Usage: python scripts/segment_bench.py [--images N] [--reps R]
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from scripts.mixed_sizes_bench import SIZES, batches, card  # noqa: E402


def step_by_step(det, ims):
    """(a): one bucket batch the way the callers did it before im_segment.  -> D2H bytes."""
    from mnc_b200 import ops
    from mnc_b200.api import unpack_voting
    B, H, W = ims.shape[:3]
    dev = det.device
    scale = ops.im_scale_for((H, W))
    out_h, out_w = int(np.rint(H * scale)), int(np.rint(W * scale))
    data = ops.prep_images(torch.from_numpy(ims).to(dev), scale)
    info = torch.tensor([[out_h, out_w, scale]] * B, dtype=torch.float32, device=dev)
    hw = torch.tensor([[H, W]] * B, dtype=torch.float32, device=dev)
    sc = torch.full((B,), scale, dtype=torch.float32, device=dev)
    boxes, masks, scores, valid, _ = det.engine.detect_checked(data, info, hw, sc)
    vote = det.mask_voting(boxes, masks, scores, valid, [[H, W]] * B, max_per_image=100)
    unpack_voting(vote)
    copied = [vote[k] for k in ("n_res", "res_class", "res_score", "result_mask", "result_box")]
    # + the 512-byte maxima of the range check and the 4-byte overflow flag
    return sum(t.numel() * t.element_size() for t in copied) + det.engine._amax_all.numel() * 4 + 4


def run(det, ims, bs, flow):
    """-> D2H bytes of every batch."""
    if flow == "a":
        return [step_by_step(det, np.stack([ims[i] for i in bt])) for bt in bs]
    if flow == "b":
        out = []
        for bt in bs:
            det.im_segment(np.stack([ims[i] for i in bt]))
            out.append(det.d2h_bytes)
        return out
    from mnc_b200 import ops
    for _ in det.im_segment_stream([[ims[i] for i in bt] for bt in bs]):
        pass
    # what _issue copies back per batch: the voted record and the activation maxima
    return [ops.vote_record_layout(len(bt), ops.default_vote_cap(100))[-1] * 4 + 512 for bt in bs]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=96)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    from mnc_b200 import weights as Wt
    from mnc_b200.api import Detector
    rng = np.random.default_rng(2026)
    shapes = [SIZES[k] for k in rng.integers(0, len(SIZES), args.images)]
    ims = [rng.integers(0, 256, size=s + (3,), dtype=np.uint8) for s in shapes]
    det = Detector(Wt.make_weights(Wt.FULL_ARCH), max_batch=8)
    print("card: %s" % card(), flush=True)
    plan = {"a": batches(ims, "a"), "b": batches(ims, "a"), "c": batches(ims, "c")}
    # warm-up: calibration, buffers and graphs of every blob shape; the largest blob (a mixed
    # batch) first, so that no buffer grows -- which drops the graphs captured before it -- later
    for _ in range(2):
        for f in "cba":
            run(det, ims, plan[f], f)
    torch.cuda.synchronize()
    names = {"a": "shape buckets, detect_checked + mask_voting_checked + unpack_voting",
             "b": "shape buckets, im_segment", "c": "mixed by orientation, im_segment_stream"}
    for f in "abc":
        ts = []
        for _ in range(args.reps):
            t0 = time.perf_counter()
            nbytes = run(det, ims, plan[f], f)
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
        t = float(np.median(ts))
        print(json.dumps(dict(flow=f, name=names[f], images=len(ims), batches=len(plan[f]),
                              images_per_s=round(len(ims) / t, 1), seconds=round(t, 4),
                              d2h_bytes_per_batch=int(round(np.mean(nbytes))))), flush=True)


if __name__ == "__main__":
    main()
