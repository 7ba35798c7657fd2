"""Timing of PAMR and the bilateral filter at the BASELINE shapes (CUDA events, L2 flushed), with algorithmic bytes."""
import sys, os, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from acr_wsss_b200 import ops, synth, PAMR

dev = torch.device("cuda:0")
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

def timeit(fn, iters=10):
    fn(); torch.cuda.synchronize()
    tot = 0.0
    for _ in range(iters):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); torch.cuda.synchronize()
        tot += a.elapsed_time(b)
    return tot / iters * 1e3

res = {}
STD = [1, 2, 4, 8, 12, 24]
# 500 x 375 (a VOC-sized image) times a width that is not a multiple of 4: its rows end in unused cells up to the 16-byte pitch
for (B, C, H, W, it, dil) in [(1, 21, 448, 448, 10, STD), (8, 21, 448, 448, 10, STD), (1, 81, 448, 448, 10, STD), (1, 21, 500, 375, 10, STD)]:
    x = ((synth.smooth_rgb(B, H, W, seed=4) - 120.0) / 58.0).to(dev)
    mask = synth.probabilities(B, C, H // 16, W // 16, seed=4).to(dev)
    pamr = PAMR(it, dil)
    t = timeit(lambda: pamr(x, mask))
    D = len(dil); HW = H * W
    alg = B * (HW * (3 * 4 + 8 * D * 4) + it * HW * (8 * D * 4 + 2 * C * 4))
    key = f"pamr_B{B}_C{C}_{H}x{W}"
    res[f"{key}_us"] = round(t, 1); res[f"{key}_GBs"] = round(alg / t / 1e3, 1)
for (N, K, S) in ([] if 'pamr' in sys.argv else [(1, 21, 224), (8, 21, 224), (8, 81, 224)]):
    img = synth.smooth_rgb(N, S, S, seed=0).to(dev); ins = synth.probabilities(N, K, S, S, seed=0).to(dev)
    t = timeit(lambda: ops.bilateral_filter(img, ins, 15.0, 50.0))
    alg = 2 * N * K * S * S * 4 + N * 3 * S * S * 4
    res[f"bilateral_N{N}_K{K}_us"] = round(t, 1); res[f"bilateral_N{N}_K{K}_GBs"] = round(alg / t / 1e3, 1)
    _, m = ops.bilateral_filter(img, ins, 15.0, 50.0, return_lattice_size=True); res[f"bilateral_N{N}_K{K}_M"] = m[0]
if 'pamr' not in sys.argv:      # worst case for the lattice: white-noise images (what the synthetic training batches are), every pixel its own vertices
    img = (torch.randn(8, 3, 224, 224, generator=torch.Generator().manual_seed(0)) * 58.0 + 120.0).clamp(0, 255).to(dev)
    ins = synth.probabilities(8, 81, 224, 224, seed=0).to(dev)
    t = timeit(lambda: ops.bilateral_filter(img, ins, 15.0, 50.0))
    res["bilateral_noise_N8_K81_us"] = round(t, 1)
    _, m = ops.bilateral_filter(img, ins, 15.0, 50.0, return_lattice_size=True); res["bilateral_noise_N8_K81_M"] = m[0]
print(json.dumps(res))
