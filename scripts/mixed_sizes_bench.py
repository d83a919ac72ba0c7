"""End-to-end throughput of three batching policies for images of different sizes (FULL_ARCH
weights, seeded synthetic uint8 images):

  (a) shape buckets: images grouped by exact size, batches of up to 8 through im_detect_images
      (the policy of scripts/demo.py and TesterWrapper);
  (b) mixed batches of 8 in arrival order through im_detect_mixed;
  (c) mixed batches of 8 after grouping by orientation (landscape / portrait).

Prints the card name and power limit, then one JSON line per policy with images/s and the fraction
of computed blob pixels that are padding.  Usage: python scripts/mixed_sizes_bench.py [--images N]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

# the reference's demo image sizes, plus two common camera sizes
SIZES = [(357, 500), (375, 500), (500, 333), (480, 640), (333, 500)]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:          # the numbers below still stand; the card line says why it is missing
        q = "unknown (%s)" % e
    return q or torch.cuda.get_device_name(0)


def batches(ims, policy, B=8):
    idx = list(range(len(ims)))
    if policy == "a":
        out = []
        for shape in sorted({ims[i].shape for i in idx}):
            grp = [i for i in idx if ims[i].shape == shape]
            out += [grp[k:k + B] for k in range(0, len(grp), B)]
        return out
    if policy == "c":
        land = [i for i in idx if ims[i].shape[0] <= ims[i].shape[1]]
        port = [i for i in idx if ims[i].shape[0] > ims[i].shape[1]]
        return [g[k:k + B] for g in (land, port) for k in range(0, len(g), B)]
    return [idx[k:k + B] for k in range(0, len(idx), B)]


def pad_fraction(ims, bs):
    from mnc_b200 import ops
    total = real = 0
    for bt in bs:
        dst = [ops.blob_size_for(ims[i].shape, ops.im_scale_for(ims[i].shape)) for i in bt]
        H, W = max(d[0] for d in dst), max(d[1] for d in dst)
        total += len(bt) * H * W
        real += sum(h * w for h, w in dst)
    return 1.0 - real / total


def run(det, ims, bs, policy):
    for bt in bs:
        if policy == "a":
            det.im_detect_images(np.stack([ims[i] for i in bt]))
        else:
            det.im_detect_mixed([ims[i] for i in bt])


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
    plan = {p: batches(ims, p) for p in "abc"}
    # warm-up: calibration, buffers and one graph per blob shape.  The largest blob (a mixed batch)
    # goes first and every policy runs twice, so that no buffer grows -- which drops the graphs
    # captured before it -- once timing starts
    for _ in range(2):
        for p in "bca":
            run(det, ims, plan[p], p)
    torch.cuda.synchronize()
    for p, name in (("a", "shape buckets"), ("b", "mixed, arrival order"), ("c", "mixed, by orientation")):
        ts = []
        for _ in range(args.reps):
            t0 = time.perf_counter()
            run(det, ims, plan[p], p)
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
        t = float(np.median(ts))
        print(json.dumps(dict(policy=p, name=name, images=len(ims), batches=len(plan[p]),
                              images_per_s=round(len(ims) / t, 1), seconds=round(t, 4),
                              pad_fraction=round(pad_fraction(ims, plan[p]), 4))), flush=True)


if __name__ == "__main__":
    main()
