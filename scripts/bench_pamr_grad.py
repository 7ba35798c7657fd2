"""PAMR forward + backward (ops.pamr_forward under autograd: acr_pamr_fwd_save + acr_pamr_bwd) at cfg3 (one image, 21 classes,
448 x 448, 10 iterations, dilations [1, 2, 4, 8, 12, 24], mask 28 x 28) and at a batch of 8, with the gradient of the mask
alone and of both inputs.  Baseline: torch autograd of the reference's composition (oracle.acr_oracle.pamr) in fp32 on the
same GPU, which is what the reference module costs a user.  CUDA events, a warm-up call, the L2 overwritten before every
timed call.  Reports ms, algorithmic bytes / time against the 7.7 TB/s HBM peak, peak memory, card name and power limit.
Prints one JSON line (and writes it to the file named by the first argument, if any)."""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from acr_wsss_b200 import PAMR, synth  # noqa: E402
from oracle import acr_oracle as orc  # noqa: E402

HBM_PEAK = 7.7e12
dev = torch.device("cuda:0")
res = {"gpu": torch.cuda.get_device_name(dev)}
try:
    res["power_limit"] = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                                        capture_output=True, text=True, timeout=30).stdout.strip()
except (OSError, subprocess.SubprocessError):
    res["power_limit"] = "unknown"
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > the 126 MB L2


def timeit(fn, iters):
    fn()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats(dev)
    base = torch.cuda.memory_allocated(dev)
    tot = 0.0
    for _ in range(iters):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        tot += a.elapsed_time(b)
    return tot / iters, (torch.cuda.max_memory_allocated(dev) - base) / 1e9


def algorithmic_bytes(B, K, C, H, W, D, T, need_x):
    """Compulsory HBM traffic of the CUDA path, from shapes: each kernel reads its inputs and writes its outputs once."""
    hw = B * H * W
    fwd = hw * (4 * C + 4 * K + 32 * D) + T * hw * (32 * D + 8 * C)           # up-sampling, weights, iterations
    adj = T * hw * (32 * D + 8 * C) + hw * 4 * C                     # iteration adjoints, bilinear adjoint
    img = 0
    if need_x:
        img = T * hw * (8 * C + 64 * D)                                        # weight gradient: G_t, M_{t-1}, dW read + write
        img += hw * (4 * K + 96 * D + 16 * K)                                  # softmax / affinity backward
        img += hw * (4 * K + 32 * D + 16 * K + 4 * K)                          # image-gradient gather
    return fwd + adj + img


def run(B, C, iters):
    H = W = 448
    K, T, dil, mh = 3, 10, [1, 2, 4, 8, 12, 24], 28
    x = ((synth.smooth_rgb(B, H, W, seed=1) - 120.0) / 58.0).to(dev)
    mask = synth.probabilities(B, C, mh, mh, seed=2).to(dev)
    g = torch.randn(B, C, H, W, device=dev)
    pamr = PAMR(T, dil)
    for mode in ("mask", "both"):
        need_x = mode == "both"

        def ours():
            xr, mr = x.clone().requires_grad_(need_x), mask.clone().requires_grad_()
            out = pamr(xr, mr)
            return torch.autograd.grad(out, [xr, mr] if need_x else [mr], g)

        def ref():
            xr, mr = x.clone().requires_grad_(need_x), mask.clone().requires_grad_()
            out = orc.pamr(xr, mr, T, dil)
            return torch.autograd.grad(out, [xr, mr] if need_x else [mr], g)

        key = f"B{B}_C{C}_448_t{T}_{mode}"
        ms, mem = timeit(ours, iters)
        nbytes = algorithmic_bytes(B, K, C, H, W, len(dil), T, need_x)
        res[f"{key}_ms"] = round(ms, 3)
        res[f"{key}_peak_gb"] = round(mem, 2)
        res[f"{key}_algorithmic_gb"] = round(nbytes / 1e9, 3)
        res[f"{key}_hbm_share"] = round(nbytes / (ms * 1e-3) / HBM_PEAK, 3)
        ms_ref, mem_ref = timeit(ref, max(2, iters // 4))
        res[f"{key}_torch_fp32_ms"] = round(ms_ref, 3)
        res[f"{key}_torch_fp32_peak_gb"] = round(mem_ref, 2)


run(1, 21, 20)
run(8, 21, 8)
line = json.dumps(res)
print(line)
if len(sys.argv) > 1:
    with open(sys.argv[1], "w") as f:
        f.write(line + "\n")
