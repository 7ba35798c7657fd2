"""Dense-CRF mean-field inference (ops.dense_crf): per-image time at VOC sizes with CUDA events, launches per call, lattice
sizes, and one image through the CPU oracle (oracle/densecrf_oracle.c, single thread) for scale.  Prints one JSON line."""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from acr_wsss_b200 import ops, synth  # noqa: E402
from oracle import densecrf_oracle  # noqa: E402

dev = torch.device("cuda:0")
res = {"gpu": torch.cuda.get_device_name(dev)}
try:
    res["power_limit"] = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                                        capture_output=True, text=True, timeout=30).stdout.strip()
except (OSError, subprocess.SubprocessError):
    res["power_limit"] = "unknown"
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > the 126 MB L2: inputs come from HBM in every timed call


def timeit(fn, iters=10):
    fn()
    torch.cuda.synchronize()
    tot = 0.0
    for _ in range(iters):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        tot += a.elapsed_time(b)
    return tot / iters


T = 10
for (N, C, H, W) in [(8, 21, 375, 500), (8, 21, 500, 375), (8, 81, 375, 500)]:
    img = synth.smooth_rgb(N, H, W, seed=1)
    P = synth.probabilities(N, C, H, W, seed=2)
    gi, gp = img.to(dev), P.to(dev)
    ms = timeit(lambda: ops.dense_crf(gi, gp, n_iter=T))
    key = f"crf_N{N}_C{C}_{H}x{W}_t{T}"
    res[f"{key}_ms_per_image"] = round(ms / N, 3)
    res[f"{key}_launches"] = (11 + 8 * T) * ((N + 7) // 8)
    _, (mg, mb) = densecrf_oracle.dense_crf(img[0].numpy(), P[0].numpy(), 0, return_lattice_sizes=True)
    res[f"{key}_lattice_gauss_bilateral"] = [mg, mb]
img = synth.smooth_rgb(1, 375, 500, seed=1)[0].numpy()
P = synth.probabilities(1, 21, 375, 500, seed=2)[0].numpy()
t0 = time.perf_counter()
densecrf_oracle.dense_crf(img, P, T)
res["oracle_cpu_1thread_C21_375x500_t10_ms"] = round((time.perf_counter() - t0) * 1e3, 1)
res["host_cores"] = os.cpu_count()
print(json.dumps(res))
