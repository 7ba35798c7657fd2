#!/usr/bin/env python
"""bench.py -- headline benchmark: ACR training throughput (BASELINE.json configs[1]).

  python bench.py --gpus N --steps K --warmup W            this repo's CUDA path (one rank per GPU under torchrun)
  python bench.py --impl reference --steps K --warmup W    the reference algorithm's CPU path (oracle port) on host cores
  python bench.py ... --dump-outputs DIR                    also write what the last timed step returned (see dump_outputs)

A "step" = one pass of train_acr.py:127-174 over one synthetic batch: two views forward (ViT-B/16, 448x448, 20
classes, B=8 per GPU), BCE + all-pairs consistency loss, backward, gradient all-reduce (N>1), SGD step.
Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for the definition of every field.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

S, C, B_PER_GPU, ALPHA, LR = 448, 20, 8, 100.0, 0.01
N_TOK, HEADS, HD, LAYERS = (S // 16) ** 2 + 1, 12, 64, 12
METRIC, UNIT = "train_imgs_per_sec", "img/s"
WORKLOAD = "train_acr.py VOC-shaped: ViT-B/16 448x448, two-view all-pairs consistency loss, B=8/GPU, bf16 operands"
# BASELINE.json configs: [1] = voc448 (the headline), [3] = coco448crf, [4] = vitl512
CONFIGS = {
    "voc448": dict(backbone="vitb", S=448, C=20, B=8, heads=12, layers=12, dense_crf=None, workload=WORKLOAD),
    "coco448crf": dict(backbone="vitb", S=448, C=80, B=8, heads=12, layers=12,
                       dense_crf={"weight": 1e-7, "sigma_rgb": 15.0, "sigma_xy": 100.0, "scale": 0.5},
                       workload="train_acr_coco.py COCO-shaped: ViT-B/16 448x448, 80 classes, two-view consistency loss + bilateral dense-CRF term "
                                "(K=81 planes at 224x224, sigma_rgb 15, sigma_xy 100, rloss-scale 0.5, weight 1e-7), B=8/GPU, bf16 operands"),
    "vitl512": dict(backbone="vitl", S=512, C=20, B=4, heads=16, layers=24, dense_crf=None,
                    workload="stress: ViT-L/16 512x512 (1025 tokens), all-pairs consistency over all 24 blocks, B=4/GPU, bf16 operands"),
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tflops_burst": d["bf16_tflops"], "tflops_sustained": d["bf16_tflops_sustained"], "src": "measured"}
    return {"hbm_gbs": 6650.0, "tflops_burst": 1590.0, "tflops_sustained": 1400.0, "src": "fallback"}


DUMP_SAMPLE = 1 << 22       # sampled elements per array: 2 x 16 MB of float32


def dump_outputs(out_dir, loss, model):
    """What a caller of the timed training step receives after its last step, as float32 .npy files in `out_dir`: the returned
    loss (loss.npy), and one fixed, seeded sample of the updated parameters (params_sample.npy) and of their gradients `p.grad`
    (grads_sample.npy), both indexed in the concatenation of the trained parameters in model.named_parameters() order, so the
    files of two builds compare element for element."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    params = [p for _, p in model.named_parameters() if p.requires_grad]
    n = sum(p.numel() for p in params)
    idx = torch.randint(0, n, (min(DUMP_SAMPLE, n),), generator=torch.Generator().manual_seed(0)).sort().values.to(params[0].device)

    def sample(ts):
        return torch.cat([t.detach().reshape(-1).float() for t in ts])[idx].cpu().numpy()

    np.save(os.path.join(out_dir, "loss.npy"), loss.detach().float().cpu().numpy())
    np.save(os.path.join(out_dir, "params_sample.npy"), sample(params))
    np.save(os.path.join(out_dir, "grads_sample.npy"), sample([p.grad for p in params]))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 7 for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        mx = [int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------
def cpu_reference_step_time(steps, warmup, batch=1):
    """The reference algorithm on host cores: oracle port (torch-CPU fp32, all threads) of one training step on a
    bounded sample (batch `batch` of the same 448x448 workload).  Returns (img/s, seconds per step, cores)."""
    import torch
    from oracle import acr_oracle as orc
    from acr_wsss_b200 import synth
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sd = orc.synth_state_dict(orc.vit_shapes(768, LAYERS, C))
    params = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    opt = torch.optim.SGD([p for p in params.values()], lr=LR, momentum=5e-4)
    img, label = synth.images(batch, S), synth.labels(batch, C)
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        loss, _, _ = orc.train_step_loss(params, img, label, ALPHA)
        opt.zero_grad()
        loss.backward()
        opt.step()
        if it >= warmup:
            times.append(time.perf_counter() - t0)
    sec = sum(times) / len(times)
    return batch / sec, sec, cores


def cpu_reference_cam_time():
    """The reference's CAM-inference loop body (infer_cam.py:145-215: 2 flips, one full backward per present class, GETAM +
    affinity refinement) on host cores through the oracle port: ONE image of the same cfg1 workload (bounded sample)."""
    import torch
    from oracle import acr_oracle as orc
    from acr_wsss_b200 import synth
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sd = orc.synth_state_dict(orc.vit_shapes(768, LAYERS, C))
    img = synth.images(1, S, seed=100)
    lab = synth.labels(1, C, present=(3, 7, 14))
    t0 = time.perf_counter()
    orc.infer_cam_image(sd, img, lab, (S, S), scales=(1,), start_layer=10, getam_func="grad")
    sec = time.perf_counter() - t0
    return 1.0 / sec, sec, cores


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = max(1, min(args.steps, 3)), max(1, min(args.warmup, 1))
    v, sec, cores = cpu_reference_step_time(steps, warmup)
    sample = f"{steps} timed steps (+{warmup} warm-up) of batch 1 of the same workload; fp32; torch CPU threads={cores}"
    _emit(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
        "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "note": "reference algorithm on host CPU cores (oracle port of train_acr.py:127-174)"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# ---------------------------------------------------------------------------------------------
def build_trainer(cfg, dev, precision, world):
    import torch
    from acr_wsss_b200 import ACR, Trainer
    torch.manual_seed(0)
    model = ACR(cfg["C"], cfg["backbone"], precision=precision).to(dev)
    for n, p in model.named_parameters():   # parameters without gradient on the ACR path (SURVEY Q4)
        if n.startswith(("pretrained.model.norm.", "pretrained.model.head.", "scratch.")) or n.endswith("bkg_token"):
            p.requires_grad_(False)
    # (Trainer broadcasts rank 0's weights to every rank before it builds its flat buffers)
    return model, Trainer(model, lr=LR, max_step=10 ** 6, alpha=ALPHA, dense_crf=cfg["dense_crf"])


def measure_other_config(name, dev, precision, world, rank, timed, steps=5):
    """Device-resident step time of another BASELINE config with the same Trainer (inputs in HBM, N ranks, all-reduce included)."""
    import gc
    import torch
    from acr_wsss_b200 import synth
    cfg = CONFIGS[name]
    model, trainer = build_trainer(cfg, dev, precision, world)
    img = synth.images(cfg["B"], cfg["S"], seed=rank).to(dev)
    lab = synth.labels(cfg["B"], cfg["C"], seed=rank).to(dev)
    losses = [float(trainer.step(img, lab)) for _ in range(4)]
    ms = timed(lambda: trainer.step(img, lab), steps)
    out = {"workload": cfg["workload"], "value": cfg["B"] * world * steps / (ms / 1e3), "unit": UNIT, "ms_per_step": ms / steps, "steps": steps,
           "per_gpu_batch": cfg["B"], "tokens": (cfg["S"] // 16) ** 2 + 1, "first_losses": [round(l, 4) for l in losses],
           "replicas_in_sync_max_rel_diff": trainer.check_replicas_in_sync(), "peak_mem_GB": round(torch.cuda.max_memory_allocated() / 2 ** 30, 1)}
    del trainer, model
    gc.collect()
    torch.cuda.empty_cache()
    return out


def measure_refine(dev, pk):
    """BASELINE north star (4): PAMR and the bilateral filter, each timed alone with CUDA events (L2 flushed between iterations)
    against the measured HBM peak on ALGORITHMIC bytes (DESIGN.md section 4)."""
    import torch
    from acr_wsss_b200 import ops, synth, PAMR
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def timeit(fn, iters=10):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        tot = 0.0
        for _ in range(iters):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record(); torch.cuda.synchronize()
            tot += a.elapsed_time(b)
        return tot / iters      # ms

    res = {}
    it, dil = 10, [1, 2, 4, 8, 12, 24]
    for key, (B, Cm, Sz) in {"pamr_cfg3": (1, 21, 448), "pamr_batch8": (8, 21, 448)}.items():
        x = ((synth.smooth_rgb(B, Sz, Sz, seed=4) - 120.0) / 58.0).to(dev)
        mask = synth.probabilities(B, Cm, Sz // 16, Sz // 16, seed=4).to(dev)
        pamr = PAMR(it, dil)
        ms = timeit(lambda: pamr(x, mask))
        D, HW = len(dil), Sz * Sz
        alg = B * (HW * (3 * 4 + 8 * D * 4) + it * HW * (8 * D * 4 + 2 * Cm * 4))       # image + weight planes written once; per iteration: weights + mask in/out
        res[key] = {"workload": f"PAMR B={B} C={Cm} {Sz}x{Sz}, {it} iterations, dilations {dil}", "ms": ms, "algorithmic_bytes": alg,
                    "roofline": {"bound": "hbm", "achieved": alg / ms / 1e6, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": alg / ms / 1e6 / pk["hbm_gbs"]}}
    for key, (N, K, Sz) in {"bilateral_cfg_k21": (8, 21, 224), "bilateral_cfg4_k81": (8, 81, 224)}.items():
        img = synth.smooth_rgb(N, Sz, Sz, seed=0).to(dev)
        ins = synth.probabilities(N, K, Sz, Sz, seed=0).to(dev)
        ms = timeit(lambda: ops.bilateral_filter(img, ins, 15.0, 50.0))
        alg = 2 * N * K * Sz * Sz * 4 + N * 3 * Sz * Sz * 4                                  # planes in + out, image in
        res[key] = {"workload": f"bilateral filter N={N} K={K} {Sz}x{Sz}, sigma_rgb 15, sigma_xy 50", "ms": ms, "algorithmic_bytes": alg,
                    "roofline": {"bound": "hbm", "achieved": alg / ms / 1e6, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": alg / ms / 1e6 / pk["hbm_gbs"]}}
    # north star (2): the consistency loss in the mode the training step uses (sign codes), cfg2 shape
    g = torch.Generator(device="cuda").manual_seed(0)
    Bc, Lc, Nc = 8, 12, N_TOK
    a1 = torch.softmax(torch.randn(Bc, Lc, Nc, Nc, device=dev, generator=g), -1)
    a2 = torch.softmax(torch.randn(Bc, Lc, Nc, Nc, device=dev, generator=g), -1)
    ms = timeit(lambda: ops.consistency_codes(a1, a2, S // 16))
    alg = 10 * Bc * Lc * Nc * Nc                                                             # both stacks read once (fp32), one code byte per element written for each
    res["consistency_codes_cfg2"] = {"workload": f"all-pairs consistency loss + sign-code gradient, B={Bc} L={Lc} N={Nc}", "ms": ms, "algorithmic_bytes": alg,
                                     "roofline": {"bound": "hbm", "achieved": alg / ms / 1e6, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": alg / ms / 1e6 / pk["hbm_gbs"]}}
    del a2
    # north star (3): the CAM contractions on the tensor cores (csrc/refine_tc.cu).  They are streams of their A operand
    # (0.4 FLOP per byte), so the roofline that bounds them is HBM; the tensor-pipe share is in profiles/ (ncu).
    for key, Bv in {"affinity_refine_tc_cfg1": 2, "affinity_refine_tc_batch8": 16}.items():
        attn = a1[:Bv] if Bv <= Bc else torch.softmax(torch.randn(Bv, Lc, Nc, Nc, device=dev, generator=g), -1)
        cam = torch.rand(Bv, Nc - 1, 3, device=dev, generator=g)
        ms = timeit(lambda: ops.affinity_refine_tc(attn, cam, 1, False))
        alg = 4 * Bv * Lc * (Nc - 1) ** 2 + 2 * 4 * Bv * (Nc - 1) * 3
        res[key] = {"workload": f"sum_l attn[:,l,1:,1:] . cam (3 classes), {Bv} views of 448x448 (tcgen05, bf16 hi/lo split)", "ms": ms, "algorithmic_bytes": alg,
                    "flop": 2 * Bv * (Nc - 1) ** 2 * 3,
                    "roofline": {"bound": "hbm", "achieved": alg / ms / 1e6, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": alg / ms / 1e6 / pk["hbm_gbs"]}}
        del attn
    del flush, a1
    return res


# ---------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from acr_wsss_b200 import ACR, Trainer, synth, ops, _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
        os.environ["NCCL_DEBUG"] = "WARN"          # keep NCCL's version banner off stdout: rank 0 prints exactly one JSON line
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    precision = args.precision
    if precision == "bf16" and not _lib.lib().acr_device_is_sm100():
        raise SystemExit("bench.py: bf16 fused path needs sm_100a")

    cfg = dict(CONFIGS[args.config])
    if args.batch:
        cfg["B"] = args.batch
    S, C = cfg["S"], cfg["C"]
    N_TOK, HEADS, LAYERS = (S // 16) ** 2 + 1, cfg["heads"], cfg["layers"]
    model, trainer = build_trainer(cfg, dev, precision, world)
    B = cfg["B"]
    img_h = synth.images(B, S, seed=rank).pin_memory()
    lab_h = synth.labels(B, C, seed=rank).pin_memory()
    img_d, lab_d = img_h.to(dev), lab_h.to(dev)

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps):
        sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        sync()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms)

    for _ in range(max(args.warmup, 3)):
        trainer.step(img_d, lab_d)
    if args.profile_range:      # one step between cudaProfilerStart/Stop for `ncu --profile-from-start off`
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        trainer.step(img_d, lab_d)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    last_loss = [None]

    def train_step():
        last_loss[0] = trainer.step(img_d, lab_d)

    ms_dev = timed(train_step, args.steps)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last_loss[0], model)      # before the steps below train the model further

    def e2e_step():
        # the public API's pipelined step: consume the batch whose pinned-host -> device copy was started one step earlier and
        # start the copy of the next batch (copy stream, under this step's kernels); then read the loss back.  One batch
        # crosses PCIe inside every timed step.
        loss = trainer.step_prefetched(img_h, lab_h)
        return float(loss)                               # D2H read of the loss

    trainer.prefetch(img_h, lab_h)                       # prime the pipeline (untimed)
    e2e_step()
    ms_e2e = timed(e2e_step, args.steps)
    clocks = sampler.stop() if rank == 0 else None

    # Per-entry-point timing.  The timed steps above are CUDA-graph replays (no host code runs, so no events can be
    # recorded inside them); the same forward+backward is therefore run eagerly K more times with CUDA events around
    # every C-ABI call on the launching stream.  Identical kernels, shapes and launch counts.
    ops.PROFILE.reset(enabled=True)
    L = _lib.lib()
    L.acr_profile_enable(1)            # CUDA event pairs around the tensor-core attention kernels themselves (inside the C ABI)
    side = trainer._side if trainer._side is not None else torch.cuda.current_stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(args.steps):
            trainer._forward_backward(img_d, lab_d)
    torch.cuda.current_stream().wait_stream(side)
    prof = ops.PROFILE.summary()
    ops.PROFILE.reset(enabled=False)
    kern = {}
    for kname in ("attn_fwd_kernel", "attn_mean_kernel", "attn_delta_kernel", "attn_bwd_kernel"):
        tot, cnt = ctypes.c_double(0.0), ctypes.c_longlong(0)
        if L.acr_profile_read(kname.encode(), ctypes.byref(tot), ctypes.byref(cnt)) == 0 and cnt.value:
            kern[kname] = {"ms": tot.value, "launches": cnt.value}
    L.acr_profile_enable(0)
    launches = prof["launches"] // args.steps * args.steps
    in_sync = trainer.check_replicas_in_sync()        # every rank holds bit-identical weights after the all-reduced steps
    if world > 1 and in_sync > 0.0:
        raise SystemExit(f"bench.py: replicas diverged after the timed steps (max relative checksum difference {in_sync:.3e})")

    # secondary metric: CAM inference (BASELINE.json configs[0]): forward_cam + GETAM over 3 present classes + affinity
    # refinement, 2 flips, one 448x448 image at a time, images sharded per rank, no collective
    cam = None
    if not args.no_cam and args.config == "voc448":
        from acr_wsss_b200 import infer_cam_image
        model.eval()
        model.set_capture_grad(True)
        for p in model.parameters():
            p.grad = None
        img1 = synth.images(1, S, seed=100 + rank).to(dev)
        lab1 = synth.labels(1, C, present=(3, 7, 14)).to(dev)
        n_img = 8
        for _ in range(3):        # warm-up: cuBLAS heuristics for the batch-2 / batch-6 shapes, allocator, pinned staging buffer
            infer_cam_image(model, img1, lab1, (S, S), start_layer=10, getam_func="grad", cuda_graph=True)
        ms_cam = timed(lambda: infer_cam_image(model, img1, lab1, (S, S), start_layer=10, getam_func="grad", cuda_graph=True), n_img)
        # algorithmic FLOPs per image: trunk forward on 2 flips (blocks < start_layer) + blocks >= start_layer forward and backward on
        # 2 x 3 class copies; per block and image 2*N*(12 E^2) (Linear layers) + 4*N^2*E (attention), backward = 2x forward
        E_, st_l, n_cls = 768, 10, 3
        blk = 2.0 * N_TOK * 12 * E_ * E_ + 4.0 * N_TOK * N_TOK * E_
        cam_flops = 2 * st_l * blk + 2 * n_cls * (LAYERS - st_l) * blk * 3.0
        cam = {"metric": "cam_infer_imgs_per_sec", "value": n_img * world / (ms_cam / 1e3), "unit": "img/s", "ms_per_image": ms_cam / n_img,
               "roofline": {"bound": "tensor", "achieved": cam_flops / (ms_cam / n_img * 1e-3) / 1e12, "peak": peaks()["tflops_sustained"], "unit": "TFLOP/s",
                            "frac": cam_flops / (ms_cam / n_img * 1e-3) / 1e12 / peaks()["tflops_sustained"], "algorithmic_flop_per_image": cam_flops,
                            "note": "batch-2 / batch-6 GEMMs and ~270 launches per image: latency bound, replayed as a CUDA graph"},
               "workload": "infer_cam.py: ViT-B/16 448x448, 2 flips, 3 present classes, GETAM start_layer=10 + affinity refine, results copied to host"}
        # the same workload through infer_cam_batch: 8 images per trunk pass (one backward, batched GETAM / affinity contraction)
        from acr_wsss_b200 import infer_cam_batch
        MB = 8
        imgb = torch.cat([synth.images(1, S, seed=200 + rank * MB + i) for i in range(MB)]).to(dev)
        labb = synth.labels(1, C, present=(3, 7, 14)).to(dev).repeat(MB, 1)
        for _ in range(3):
            infer_cam_batch(model, imgb, labb, (S, S), start_layer=10, getam_func="grad", cuda_graph=True)
        ms_b = timed(lambda: infer_cam_batch(model, imgb, labb, (S, S), start_layer=10, getam_func="grad", cuda_graph=True), 4)
        cam["batched"] = {"value": 4 * MB * world / (ms_b / 1e3), "unit": "img/s", "ms_per_image": ms_b / (4 * MB), "images_per_pass": MB,
                          "roofline": {"bound": "tensor", "achieved": cam_flops / (ms_b / (4 * MB) * 1e-3) / 1e12, "peak": peaks()["tflops_sustained"],
                                       "unit": "TFLOP/s", "frac": cam_flops / (ms_b / (4 * MB) * 1e-3) / 1e12 / peaks()["tflops_sustained"]},
                          "workload": "infer_cam_batch: 8 images of the cfg1 workload per pass (2 flips x 8 images x 3 class copies), results copied to host"}
        # BASELINE.json configs[2]: multi-scale (0.5/1.0/1.5/2.0 + flip), affinity power t=2 (row-normalised), then PAMR on the CAMs
        from acr_wsss_b200 import PAMR
        pamr = PAMR(10, [1, 2, 4, 8, 12, 24]).to(dev)
        ms_kw = dict(scales=(0.5, 1.0, 1.5, 2.0), start_layer=10, getam_func="grad", t=2, normalize=True, cuda_graph=True)

        def multiscale():
            _, _, norm_cam = infer_cam_image(model, img1, lab1, (S, S), **ms_kw)
            return pamr(img1, norm_cam.unsqueeze(0))

        for _ in range(3):
            multiscale()
        ms_multi = timed(multiscale, 4)
        cam["multiscale"] = {"value": 4 * world / (ms_multi / 1e3), "unit": "img/s", "ms_per_image": ms_multi / 4,
                             "workload": "scales 0.5/1.0/1.5/2.0 x 2 flips, t=2 row-normalised affinity power, PAMR(10 it., 6 dilations) on the 20-class CAM"}

    # the other BASELINE configs with the same Trainer, and the refinement kernels of north star (4): short secondary measurements
    others, refine = None, None
    if not args.no_extra and args.config == "voc448":
        import gc
        del trainer, model
        gc.collect()
        torch.cuda.empty_cache()
        others = {name: measure_other_config(name, dev, precision, world, rank, timed) for name in ("coco448crf", "vitl512")}
        if rank == 0:
            refine = measure_refine(dev, peaks())
        sync()
        trainer = None
    if rank == 0:
        pk = peaks()
        imgs = B * world * args.steps
        value = imgs / (ms_dev / 1e3)
        e2e = imgs / (ms_e2e / 1e3)
        # dominant kernel: attn_bwd_kernel (one launch per block on the 2B images of both views), timed by CUDA events
        # recorded around the launch itself inside the C ABI during the eager replay
        dom = kern.get("attn_bwd_kernel") if precision == "bf16" else None
        # algorithmic FLOPs of one launch: dP, dV, dK, dQ = 4 GEMMs of 2*N^2*D per head and image; the S recompute is not counted
        flops_bwd = 8.0 * (2 * B) * HEADS * N_TOK * N_TOK * HD
        roof = None
        if dom:
            avg_ms = dom["ms"] / dom["launches"]
            ach = flops_bwd / (avg_ms * 1e-3) / 1e12
            traffic, traffic_src = None, None
            tpath = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "roofline_traffic.json")
            if os.path.exists(tpath):
                tj = json.load(open(tpath))
                if tj.get("kernel") == "attn_bwd_kernel":
                    traffic, traffic_src = tj["dram_bytes_per_launch"], tj["source"]
            roof = {"bound": "tensor", "kernel": "attn_bwd_kernel", "achieved": ach, "peak": pk["tflops_sustained"], "unit": "TFLOP/s",
                    "frac": ach / pk["tflops_sustained"], "traffic": traffic, "traffic_unit": "bytes/launch", "traffic_source": traffic_src,
                    "avg_launch_ms": avg_ms, "launches_per_step": dom["launches"] / args.steps,
                    "algorithmic_flop_per_launch": flops_bwd,
                    "peak_source": pk["src"] + " (sustained bf16 cuBLAS; the kernel runs inside a long step)",
                    "share_of_step": dom["ms"] / ms_dev,
                    "timing": "CUDA events around the kernel launch on its stream, eager replay of the same steps (the timed steps are CUDA graphs)",
                    "kernels_ms_per_step": {k: v["ms"] / args.steps for k, v in kern.items()},
                    "entry_points_ms_per_step": {k: v["ms"] / args.steps for k, v in prof["kernels"].items()}}
        elif precision != "bf16":
            d32 = prof["kernels"].get("acr_attn_bwd_f32")
            if d32 and d32["calls"]:
                avg_ms = d32["ms"] / d32["calls"]
                ach = flops_bwd / (avg_ms * 1e-3) / 1e12
                roof = {"bound": "tensor", "kernel": d32["name"], "achieved": ach, "peak": pk["tflops_sustained"], "unit": "TFLOP/s",
                        "frac": ach / pk["tflops_sustained"], "traffic": None, "avg_launch_ms": avg_ms, "peak_source": pk["src"]}
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16" if precision == "bf16" else "f32", "data": "synthetic",
            "config": {"workload": cfg["workload"], "name": args.config, "global_batch": B * world, "per_gpu_batch": B, "tokens": N_TOK, "parallelism": f"dp{world}",
                       "precision": precision, "cuda_graph": True, "l2": "inputs larger than L2: each step streams 2 x 237 MB attention stacks + gradients"},
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": int(img_h.numel() * 4 + lab_h.numel() * 4) * world,
                    "d2h_bytes_per_step": 4 * world, "ms_per_step": ms_e2e / args.steps,
                    "api": "Trainer.step_prefetched(next_img, next_label): every timed step copies one pinned-host batch to the device "
                           "(the one the next step consumes, on a copy stream under this step's kernels) and reads float(loss) back"},
            "gpu_launches": launches, "clocks": clocks, "roofline": roof, "cam_infer": cam,
            "replicas_in_sync_max_rel_diff": in_sync, "other_configs": others, "refine": refine,
        }
        if world == 1 and not args.no_cpu_baseline and args.config == "voc448":
            v, sec, cores = cpu_reference_step_time(2, 1)
            out["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                                   "sample": "2 timed steps (+1 warm-up) of batch 1 of the same workload, fp32 torch CPU (oracle port)"}
            if cam is not None:
                v, sec, cores = cpu_reference_cam_time()
                cam["cpu_baseline"] = {"value": v, "unit": "img/s", "cores": cores, "kind": "port",
                                       "sample": "1 image of the same cfg1 workload (2 flips, 3 classes, full backward per class), fp32 torch CPU (oracle port)"}
        _emit(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: the config's)")
    ap.add_argument("--config", default="voc448", choices=sorted(CONFIGS), help="BASELINE.json configs[1] (default) / [3] / [4]")
    ap.add_argument("--no-extra", action="store_true", help="skip the secondary measurements (other configs, PAMR / bilateral)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cam", action="store_true", help="skip the secondary CAM-inference measurement")
    ap.add_argument("--profile-range", action="store_true", help="wrap one extra step in cudaProfilerStart/Stop (for ncu)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the loss, parameters and gradients of the last timed step (sampled) as .npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what this repo's CUDA path computed; it does not apply to --impl reference")
    # stdout carries exactly ONE JSON line: everything libraries print while the bench runs (e.g. NCCL's version banner goes
    # to stdout) is sent to stderr instead, at file-descriptor level, and the line is written to the real stdout at the end
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    global _emit
    def _emit(line):
        sys.stdout.flush()
        os.write(real_stdout, (line + "\n").encode())
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
