"""The evaluation.py step on the GPU: mIoU of CAM pseudo-labels (or of label-map predictions) against VOC-style ground truth,
at one background threshold (--t) or at every threshold i/100 (--curve), in one pass over the data (cam.LabelEvaluator).

    python scripts/evaluate_cams.py --list val.txt --predict_dir out_cam --gt_dir SegmentationClass --curve [--json out.json]

--type npy reads the {class: float32 [rows, cols]} dicts that save_cam_dict writes; --type png reads label-map predictions
(palette or greyscale indices).  Ground truth: palette PNGs, 255 = ignore.  Files are read on a small thread pool while the
GPU counts the previous batch.  There is no CPU path: without a CUDA device the script fails.
"""
import argparse
import json
import os
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--list", required=True, help="text file with one image id per line")
    ap.add_argument("--predict_dir", required=True)
    ap.add_argument("--gt_dir", required=True)
    ap.add_argument("--type", choices=("npy", "png"), default="npy")
    ap.add_argument("--t", type=float, default=None, help="one background threshold (npy)")
    ap.add_argument("--curve", action="store_true", help="sweep the thresholds i/100, i = 0..99 (npy)")
    ap.add_argument("--num_classes", type=int, default=21)
    ap.add_argument("--json", default=None, help="write the curve and the per-class IoU at the best threshold here")
    ap.add_argument("--batch", type=int, default=32, help="images per host-to-device copy")
    ap.add_argument("--workers", type=int, default=8)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        sys.exit("evaluate_cams.py: needs a CUDA GPU (the counting runs there; there is no CPU path)")
    from PIL import Image
    from acr_wsss_b200 import cam

    if args.type == "npy":
        thresholds = [i / 100 for i in range(100)] if args.curve or args.t is None else [args.t]
    else:
        thresholds = [0.0]                           # label maps do not depend on the threshold
    names = [ln.strip() for ln in open(args.list) if ln.strip()]
    ev = cam.LabelEvaluator(args.num_classes, thresholds)

    def load(name):
        gt = np.asarray(Image.open(os.path.join(args.gt_dir, name + ".png")), dtype=np.uint8)
        if args.type == "npy":
            return cam.load_cam_dict(os.path.join(args.predict_dir, name + ".npy")), gt
        return np.asarray(Image.open(os.path.join(args.predict_dir, name + ".png")), dtype=np.uint8), gt

    batches = [names[i:i + args.batch] for i in range(0, len(names), args.batch)]
    with ThreadPoolExecutor(args.workers) as pool:
        pending = [pool.submit(lambda b: [load(n) for n in b], b) for b in batches[:2]]
        for k in range(len(batches)):
            items = pending[k].result()
            if k + 2 < len(batches):
                pending.append(pool.submit(lambda b: [load(n) for n in b], batches[k + 2]))
            pending[k] = None
            preds, gts = [p for p, _ in items], [g for _, g in items]
            if args.type == "npy":
                ev.add(preds, gts)
            else:
                ev.add_labels(preds, gts)
    iou, miou, best_t, best_m = ev.result()
    b = thresholds.index(best_t)
    if args.type == "npy":
        for t, m in zip(thresholds, miou):
            print(f"threshold {t:.2f}  mIoU {m * 100:.3f}")
        print(f"best threshold {best_t:.2f}  mIoU {best_m * 100:.3f}")
    else:
        print(f"mIoU {best_m * 100:.3f}")
    if args.json:
        with open(args.json, "w") as f:
            json.dump({"images": len(names), "type": args.type, "thresholds": thresholds, "miou": miou.tolist(),
                       "best_threshold": best_t, "best_miou": best_m, "iou_at_best": iou[b].tolist()}, f)


if __name__ == "__main__":
    main()
