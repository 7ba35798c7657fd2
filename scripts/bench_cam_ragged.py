"""CAM inference over images of different original sizes: infer_cam_image one image at a time against infer_cam_batch with
per-image output sizes, and the finish kernel (csrc/cam_finish.cu) alone.  Prints one JSON line.

Workload: the cfg1 options (448x448 trunk input, start_layer=10, GETAM 'grad', 3 present classes, bf16, CUDA graphs) on 8
images whose original sizes are VOC-like: long side 500, both orientations.  Timings include the copy of the results to
the host and end in a device synchronise; every shape is warmed up first.
  python scripts/bench_cam_ragged.py
"""
import ctypes
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from bench import peaks  # noqa: E402

S, C, START_LAYER, PRESENT = 448, 20, 10, (3, 7, 14)
SIZES = [(375, 500), (500, 375), (333, 500), (500, 333), (281, 500), (500, 442), (400, 500), (500, 366)]     # (rows, cols)


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "nvidia-smi unavailable"
    return {"name": name, "power_limit_and_max_sm_clock": q}


def main():
    from acr_wsss_b200 import ACR, infer_cam_image, infer_cam_batch, ops, synth, _lib
    from acr_wsss_b200.cam import _finish_planes
    if not torch.cuda.is_available():
        raise SystemExit("bench_cam_ragged.py: no CUDA device")
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    model = ACR(C, "vitb", precision="bf16").to(dev).eval()
    model.set_capture_grad(True)
    M = len(SIZES)
    imgs = torch.cat([synth.images(1, S, seed=300 + i) for i in range(M)]).to(dev)
    labels = synth.labels(1, C, present=PRESENT).to(dev).repeat(M, 1)
    kw = dict(start_layer=START_LAYER, getam_func="grad", cuda_graph=True)

    def per_image():
        for i in range(M):
            infer_cam_image(model, imgs[i:i + 1], labels[i:i + 1], SIZES[i], **kw)

    def batched():
        infer_cam_batch(model, imgs, labels, SIZES, **kw)

    def timed(fn, reps):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / reps

    res = {"gpu": gpu_info(), "workload": f"{M} images, trunk input {S}x{S}, original sizes (rows, cols) {SIZES}, classes {PRESENT}, "
                                          f"start_layer={START_LAYER}, GETAM 'grad', bf16, cuda_graph=True, results copied to host"}
    reps = 5
    s_img, s_bat = timed(per_image, reps), timed(batched, reps)
    res["per_image"] = {"img_per_s": M / s_img, "ms_per_image": s_img * 1e3 / M}
    res["batched_ragged"] = {"img_per_s": M / s_bat, "ms_per_image": s_bat * 1e3 / M}

    # the finish kernel alone, on maps of the shapes the batched pass hands it (one scale, 28x28 grid, n = 3 copies)
    g = torch.Generator().manual_seed(0)
    ph = pw = S // 16
    n = len(PRESENT)
    cams = [torch.rand(2 * M, ph * pw, n, generator=g).to(dev)]
    patch = [torch.rand(2 * M, ph * pw, C, generator=g).to(dev)]
    planes, total = _finish_planes([list(PRESENT)] * M, SIZES)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)       # larger than L2: every launch starts from a cold cache
    iters = 50
    for _ in range(3):
        ops.cam_finish(cams, patch, [(ph, pw)], labels, planes, total)
    torch.cuda.synchronize()
    L = _lib.lib()
    L.acr_profile_enable(1)            # CUDA events recorded around the kernel launch itself, inside the C ABI
    for _ in range(iters):
        flush.zero_()
        ops.cam_finish(cams, patch, [(ph, pw)], labels, planes, total)
    tot, cnt = ctypes.c_double(0.0), ctypes.c_longlong(0)
    _lib.check(L.acr_profile_read(b"cam_finish_kernel", ctypes.byref(tot), ctypes.byref(cnt)), "acr_profile_read")
    L.acr_profile_enable(0)
    assert cnt.value == iters
    ms = tot.value / iters
    written = 4 * total
    lowres = 4 * 2 * ph * pw * len(planes)              # per plane: its channel of both views of the one scale
    pk = peaks()
    res["finish_kernel"] = {"us": ms * 1e3, "planes": len(planes), "bytes_written": written, "bytes_lowres_read": lowres,
                            "GB_per_s": (written + lowres) / ms / 1e6, "hbm_peak_GB_per_s": pk["hbm_gbs"], "peak_source": pk["src"],
                            "frac_of_peak": (written + lowres) / ms / 1e6 / pk["hbm_gbs"],
                            "timing": f"CUDA events around each of {iters} kernel launches, L2 flushed before each"}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
