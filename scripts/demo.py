#!/usr/bin/env python
"""End-to-end demo on the batched engine -- the flow of the reference's tools/demo.py:121-170
(`im_detect` -> `gpu_mask_voting` -> `get_vis_dict` -> `_convert_pred_to_image` -> colour overlay),
with everything between the uint8 frames and the rendered label images resident on the GPU:

    python scripts/demo.py --images a.jpg b.jpg [--net model.caffemodel] [--out out_dir]

Images of the same size are batched.  --net takes a binary `.caffemodel` or the `.caffemodel.h5`
that data/scripts/fetch_mnc_model.sh downloads; without it the seeded random initialiser is used.
Outputs per image: `cls_<name>.png` (VOC palette) and `final_<name>.jpg`
(0.2 * image + 0.8 * class colours, as demo.py:165-169 blends them)."""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import cv2
import numpy as np
import torch

from mnc_b200.api import Detector


def main():
    ap = argparse.ArgumentParser(description="MNC demo on mnc_b200")
    ap.add_argument("--images", nargs="+", required=True)
    ap.add_argument("--net", default=None, help=".caffemodel or .caffemodel.h5 of the 5-stage net")
    ap.add_argument("--out", default="demo_out")
    ap.add_argument("--gpu", type=int, default=0)
    ap.add_argument("--vis-thresh", type=float, default=0.5)
    ap.add_argument("--max-batch", type=int, default=8)
    args = ap.parse_args()

    dev = torch.device("cuda", args.gpu)
    torch.cuda.set_device(dev)
    if args.net:
        from mnc_b200.caffemodel import weights_from_caffemodel
        weights = weights_from_caffemodel(args.net)
    else:
        from mnc_b200.weights import make_weights
        weights = make_weights()
    det = Detector(weights, device=dev, max_batch=args.max_batch)
    os.makedirs(args.out, exist_ok=True)

    frames = [(p, cv2.imread(p)) for p in args.images]
    missing = [p for p, im in frames if im is None]
    if missing:
        raise SystemExit("cannot read: %s" % ", ".join(missing))
    by_shape = {}
    for p, im in frames:
        by_shape.setdefault(im.shape, []).append((p, im))
    for group in by_shape.values():
        for s in range(0, len(group), args.max_batch):
            chunk = group[s:s + args.max_batch]
            res = det.im_segment(np.stack([im for _, im in chunk]), render=True, vis_thresh=args.vis_thresh)
            for (path, im), r in zip(chunk, res):
                name = os.path.splitext(os.path.basename(path))[0]
                cv2.imwrite(os.path.join(args.out, "cls_%s.png" % name), r["bgr"])
                blend = cv2.addWeighted(im, 0.2, r["bgr"], 0.8, 0.0)
                cv2.imwrite(os.path.join(args.out, "final_%s.jpg" % name), blend)
                drawn = int((r["scores"] >= args.vis_thresh).sum())
                print("%s: %d instances drawn (%d voted)" % (path, drawn, len(r["scores"])))


if __name__ == "__main__":
    main()
