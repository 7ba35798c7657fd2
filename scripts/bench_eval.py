"""Pseudo-label evaluation (csrc/label_eval.cu, cam.LabelEvaluator) on a synthetic VOC-val-like set: 1,449 images of VOC's
common sizes, 1-3 present classes with smooth CAMs, ground truth with ignore bands.  Prints one JSON line with the card and
its power limit, and:
  - kernel: device time of cam_label_counts_kernel for the whole set and the 100-threshold sweep (CUDA events around the
    launch, after warm-up; the 2.5 GB of inputs exceed the L2, so every call reads HBM), median / min / max over the runs,
    and the bytes it must read (4 C' HW + HW per image) over that time;
  - call: the same with the host-side table work of ops.cam_label_counts;
  - label_map_kernel: label_map_counts_kernel over the same ground truth with label-map predictions;
  - evaluator: LabelEvaluator.add (batches of 64 host images) + result(), end to end from host arrays;
  - numpy: pseudo_label + label_iou on the host for a stated subset of images and thresholds, per (image, threshold), and
    that rate scaled to the full sweep (an extrapolation, not a measurement).
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

from acr_wsss_b200 import _lib, cam, ops  # noqa: E402

# (rows, cols) and relative frequency of the most common VOC 2012 image sizes
VOC_SIZES = [((375, 500), 40), ((500, 375), 14), ((333, 500), 12), ((500, 333), 6), ((334, 500), 4), ((281, 500), 4),
             ((366, 500), 4), ((500, 500), 3), ((400, 500), 3), ((332, 500), 3), ((335, 500), 3), ((480, 640), 2), ((300, 400), 2)]


def synth_set(n, seed):
    rng = np.random.default_rng(seed)
    g = torch.Generator().manual_seed(seed)
    w = np.array([f for _, f in VOC_SIZES], np.float64)
    picks = rng.choice(len(VOC_SIZES), n, p=w / w.sum())
    dicts, gts = [], []
    for k in picks:
        h, wd = VOC_SIZES[k][0]
        classes = sorted(rng.choice(20, rng.integers(1, 4), replace=False).tolist())
        low = torch.rand(len(classes), 1, 6, 8, generator=g)
        up = F.interpolate(low, (h, wd), mode="bilinear", align_corners=False)[:, 0]
        mn, mx = up.amin((1, 2), keepdim=True), up.amax((1, 2), keepdim=True)
        planes = ((up - mn) / (mx - mn + 1e-6)).numpy()
        d = {c: planes[i] for i, c in enumerate(classes)}
        noise = F.interpolate(torch.rand(len(classes), 1, 12, 16, generator=g), (h, wd), mode="bilinear", align_corners=False)
        noisy = planes + 0.3 * (noise[:, 0].numpy() - 0.5)      # the ground truth disagrees with the CAMs in places
        best = noisy.max(0)
        gt = np.where(best > 0.4, np.asarray(classes)[noisy.argmax(0)] + 1, 0).astype(np.uint8)
        gt[np.abs(best - 0.4) < 0.03] = 255                    # ignore band along the object borders
        dicts.append(d)
        gts.append(gt)
    return dicts, gts


def card():
    dev = torch.device("cuda:0")
    res = {"gpu": torch.cuda.get_device_name(dev)}
    try:
        res["power_limit"] = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        res["power_limit"] = "unknown"
    return res


def stats(v):
    v = sorted(v)
    return {"median": v[len(v) // 2], "min": v[0], "max": v[-1], "runs": len(v)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=1449)
    ap.add_argument("--runs", type=int, default=20)
    ap.add_argument("--numpy_images", type=int, default=8)
    ap.add_argument("--numpy_thresholds", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_eval.py: needs a CUDA GPU")
    res = card()
    dev = torch.device("cuda:0")
    K, thr = 21, [i / 100 for i in range(100)]
    t0 = time.perf_counter()
    dicts, gts = synth_set(args.images, 0)
    res["synth_s"] = time.perf_counter() - t0
    npix = [g.size for g in gts]
    nplanes = sum(len(d) for d in dicts)
    res["images"], res["planes"], res["pixels"] = len(gts), nplanes, int(sum(npix))
    bytes_read = sum(4 * len(d) * n + n for d, n in zip(dicts, npix))
    res["bytes_read_GB"] = bytes_read / 1e9

    # the whole set resident on the device
    flat = np.concatenate([v.ravel() for d in dicts for v in d.values()])
    cams_d = torch.from_numpy(flat).to(dev)
    gt_d = torch.from_numpy(np.concatenate([g.ravel() for g in gts])).to(dev)
    del flat
    planes, images, fo, go = [], [], 0, 0
    for m, (d, g) in enumerate(zip(dicts, gts)):
        images.append((go, g.shape[0], g.shape[1]))
        go += g.size
        for c in d:
            planes.append((fo, m, c))
            fo += g.size
    counts = torch.zeros(ops.cam_label_counts_len(K, len(thr)), device=dev, dtype=torch.int64)
    L = _lib.lib()
    kern, call = [], []
    for r in range(args.runs + 2):
        L.acr_profile_enable(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        ops.cam_label_counts(cams_d, planes, gt_d, images, thr, K, counts)
        b.record()
        torch.cuda.synchronize()
        ms, n = ctypes.c_double(), ctypes.c_longlong()
        _lib.check(L.acr_profile_read(b"cam_label_counts_kernel", ctypes.byref(ms), ctypes.byref(n)), "acr_profile_read")
        L.acr_profile_enable(0)
        if r >= 2:                                              # warm-up: module load, table staging, attribute
            kern.append(ms.value)
            call.append(a.elapsed_time(b))
    res["kernel_ms"] = stats(kern)
    res["kernel_GBps_at_median"] = bytes_read / (res["kernel_ms"]["median"] * 1e-3) / 1e9
    res["call_ms"] = stats(call)

    # label-map mode on the same ground truth (predictions = the pseudo-labels at 0.3)
    preds_d = torch.empty_like(gt_d)
    off = 0
    for d, g in zip(dicts, gts):
        preds_d[off:off + g.size] = torch.from_numpy(cam.pseudo_label(d, K - 1, 0.3).ravel())
        off += g.size
    mk = []
    maps = None
    for r in range(args.runs + 2):
        L.acr_profile_enable(1)
        maps = ops.label_map_counts(preds_d, gt_d, images, K, maps)
        torch.cuda.synchronize()
        ms, n = ctypes.c_double(), ctypes.c_longlong()
        _lib.check(L.acr_profile_read(b"label_map_counts_kernel", ctypes.byref(ms), ctypes.byref(n)), "acr_profile_read")
        L.acr_profile_enable(0)
        if r >= 2:
            mk.append(ms.value)
    res["label_map_kernel_ms"] = stats(mk)
    del cams_d, gt_d, preds_d

    # end to end from host arrays
    e2e = []
    for r in range(4):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ev = cam.LabelEvaluator(K, thr)
        for i in range(0, len(dicts), 64):
            ev.add(dicts[i:i + 64], gts[i:i + 64])
        iou, miou, best_t, best_m = ev.result()
        e2e.append((time.perf_counter() - t0) * 1e3)
        if r == 0:
            e2e.clear()                                         # first pass: pinned-allocator growth
            res["best_threshold"], res["best_miou"] = best_t, best_m
    res["evaluator_ms"] = stats(e2e)

    # the numpy composition on the host, for a subset
    sub = list(range(args.numpy_images))
    sub_t = thr[::len(thr) // args.numpy_thresholds][:args.numpy_thresholds]
    t0 = time.perf_counter()
    for t in sub_t:
        cam.label_iou([cam.pseudo_label(dicts[i], K - 1, t) for i in sub], [gts[i] for i in sub], K)
    np_s = time.perf_counter() - t0
    per = np_s / (len(sub) * len(sub_t))
    res["numpy"] = {"images": len(sub), "thresholds": len(sub_t), "seconds": np_s, "ms_per_image_threshold": per * 1e3,
                    "full_sweep_s_extrapolated": per * len(dicts) * len(thr)}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
