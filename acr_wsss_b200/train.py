"""The ACR training step (train_acr.py:127-174) on this repo's kernels.

PolyOptimizer mirrors tool/torchutils.py:10-31 INCLUDING its argument slip (SURVEY Q2): the reference passes
weight_decay positionally into SGD's momentum slot, so the effective optimiser is SGD(momentum=wt_dec, weight_decay=0)
with lr_t = lr * (1 - t/max_step)^0.9.

Trainer runs the step either eagerly or -- the default on a GPU -- as two CUDA graphs (forward+backward, optimiser
update) around one NCCL all-reduce of the flat gradient buffer: after the kernels were fused the step became CPU-launch
bound (~950 launches), and a graph replay removes that.  The optimiser in graph mode is the same SGD written on flat
buffers with the learning rate in a device scalar (so the poly schedule keeps working across replays).
"""
import torch
import torch.distributed as dist

from . import ops
from .losses import acr_total_loss
from .parallel import GradBuckets


class PolyOptimizer(torch.optim.SGD):
    def __init__(self, params, lr, weight_decay, max_step, momentum=0.9):
        super().__init__(params, lr, weight_decay)          # sic: lands in `momentum` (tool/torchutils.py:13)
        self.global_step = 0
        self.max_step = max_step
        self.momentum = momentum                             # the poly exponent (tool/torchutils.py:24)
        self.__initial_lr = [group['lr'] for group in self.param_groups]

    def step(self, closure=None):
        if self.global_step < self.max_step:
            lr_mult = (1 - self.global_step / self.max_step) ** self.momentum
            for i in range(len(self.param_groups)):
                self.param_groups[i]['lr'] = self.__initial_lr[i] * lr_mult
        super().step(closure)
        self.global_step += 1


class _FlatPolySGD:
    """PolyOptimizer's arithmetic on flat buffers: buf = m*buf + g ; p -= lr_t*buf, m = wt_dec (SURVEY Q2), lr_t on device."""

    def __init__(self, params, flat_grad, offsets, lr, wt_dec, max_step, poly=0.9):
        self.params = params
        self.offsets = offsets                                  # same (128-element aligned) layout as the gradient buffer
        dev = flat_grad.device
        self.flat_grad = flat_grad
        self.flat_param = torch.zeros_like(flat_grad)
        for p in params:
            off, n = offsets[p], p.numel()
            self.flat_param[off:off + n].copy_(p.data.reshape(-1))
            p.data = self.flat_param[off:off + n].view_as(p)
        self.buf = torch.zeros_like(flat_grad)
        # persistent bf16 copy of the master weights for the trunk's Linear layers (refreshed inside update())
        self.flat_param16 = self.flat_param.to(torch.bfloat16)
        self.lr0, self.mom, self.max_step, self.poly = lr, wt_dec, max_step, poly
        self.global_step = 0
        self.neg_lr = torch.zeros((), device=dev, dtype=torch.float32)
        self.param_groups = [{"lr": lr}]

    def set_lr_for_step(self):
        mult = (1 - self.global_step / self.max_step) ** self.poly if self.global_step < self.max_step else 0.0
        if self.global_step >= self.max_step:
            mult = (1 - (self.max_step - 1) / self.max_step) ** self.poly      # the reference stops updating lr there
        self.param_groups[0]["lr"] = self.lr0 * mult
        self.neg_lr.fill_(-self.lr0 * mult)
        self.global_step += 1

    def update(self, s=0, e=None, grad=None):
        """graph-capturable; [s, e): the slice of the flat buffers to update (default: all); grad: the gradients of that slice when
        they do not live in the flat gradient buffer (reduce-scattered slice of a sharded optimiser)."""
        e = self.flat_param.numel() if e is None else e
        g = self.flat_grad[s:e] if grad is None else grad
        if self.flat_param.is_cuda:
            ops.sgd_momentum_step(self.flat_param[s:e], g, self.buf[s:e], self.flat_param16[s:e], self.mom, self.neg_lr)
        else:                   # CPU unit tests of the host logic (gloo)
            self.buf[s:e].mul_(self.mom).add_(g)
            self.flat_param[s:e].addcmul_(self.buf[s:e], self.neg_lr)
            self.flat_param16[s:e].copy_(self.flat_param[s:e])

    def attach_bf16_views(self, model):
        """Give every trunk Linear a bf16 view (`_w16`, `_b16`) of its master parameters."""
        off = self.offsets
        for mod in model.modules():
            if isinstance(mod, torch.nn.Linear) and mod.weight in off and getattr(mod, "weight").requires_grad:
                w = mod.weight
                mod._w16 = self.flat_param16[off[w]:off[w] + w.numel()].view_as(w)
                if mod.bias is not None and mod.bias in off:
                    b = mod.bias
                    mod._b16 = self.flat_param16[off[b]:off[b] + b.numel()].view_as(b)


class Trainer:
    """One object = one rank.  `step(img, label)` takes HOST (pinned) or device tensors and returns the loss tensor
    (device, detached); gradients are averaged across ranks when torch.distributed is initialised.  `prefetch(img, label)`
    followed by `step()` overlaps the host->device copy of the next batch with the current step."""

    def __init__(self, model, lr=0.01, wt_dec=5e-4, max_step=100000, alpha=100.0, bucket_bytes=64 << 20, cuda_graph=None,
                 dense_crf=None):
        """dense_crf: None, or the options of the dense-CRF regulariser of BASELINE.json configs[3] (flags of infer_cam.py:58-65):
        dict(weight=1e-7, sigma_rgb=15.0, sigma_xy=100.0, scale=0.5, mean=120.0, std=58.0).  The term is applied to the softmax over
        [background, classes] of view 1's patch-token logits up-sampled to the image size (K = C + 1 planes), on the image
        de-normalised to 0..255 with (mean, std)."""
        self.model = model
        self.alpha = alpha
        self.dense_crf = None if dense_crf is None else dict({"weight": 1e-7, "sigma_rgb": 15.0, "sigma_xy": 100.0, "scale": 0.5,
                                                              "mean": 120.0, "std": 58.0}, **dense_crf)
        model.train()
        model.set_capture_grad(False)
        self.dev = next(model.parameters()).device
        self.world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
        if self.world > 1:
            # every replica starts from rank 0's weights (what DistributedDataParallel's constructor does for the reference,
            # train_acr.py:99); buffers included.  Done BEFORE the flat fp32 / bf16 / momentum buffers are built from them.
            with torch.no_grad():
                for t in list(model.parameters()) + list(model.buffers()):
                    dist.broadcast(t.data, 0)
        self.graph = (self.dev.type == "cuda") if cuda_graph is None else bool(cuda_graph)
        import os
        # Sharded optimiser (several ranks, bf16 trunk): the training step reads the trunk's Linear weights only through their
        # persistent bf16 copies, so their fp32 masters and momentum need to be current on ONE rank each.  Gradients of that region
        # are reduce-scattered, every rank updates its 1/W slice and the bf16 copies are all-gathered: 3/4 of the all-reduce's
        # bytes, and the HBM-bound optimiser kernel shrinks W-fold.  The small rest (LayerNorm, embeddings, cls_head) stays
        # replicated behind an all-reduce.  ACR_SHARDED_OPT=0 restores the plain all-reduce + full update.
        big = []
        if self.graph and self.world > 1 and getattr(model, "precision", "fp32") == "bf16" and os.environ.get("ACR_SHARDED_OPT", "1") != "0":
            for mod in model.pretrained.model.blocks.modules():
                if isinstance(mod, torch.nn.Linear) and mod.weight.requires_grad:
                    big.append(mod.weight)
                    if mod.bias is not None and mod.bias.requires_grad:
                        big.append(mod.bias)
        self.sharded = len(big) > 0
        self._master_stale = False
        # parameters the ACR path never reaches get no gradient in the reference either (SURVEY Q4)
        self.buckets = GradBuckets(list(model.parameters()), bucket_bytes, hooks=not self.graph, sharded=big or None)
        if self.graph:
            self.opt = _FlatPolySGD(self.buckets.params, self.buckets.flat, self.buckets.offsets, lr, wt_dec, max_step)
            if getattr(model, "precision", "fp32") == "bf16":
                self.opt.attach_bf16_views(model.pretrained.model.blocks)
        else:
            self.opt = PolyOptimizer(model.parameters(), lr=lr, weight_decay=wt_dec, max_step=max_step)
        # weights loaded AFTER construction (model.load / load_state_dict copy into the flat master buffer in place) must
        # reach the persistent bf16 copy the trunk's Linear layers read
        # slices of the gradient all-reduce -> optimiser pipeline.  Measured on 2 x B200: 1 / 2 / 4 / 8 slices = 13.97 / 13.83 / 14.01 /
        # 14.07 ms per step (13.43 on one GPU): the HBM-bound optimiser kernel does not overlap the NCCL kernels in practice.
        self.reduce_chunks = int(os.environ.get("ACR_AR_CHUNKS", "1"))
        self._load_hook = model.register_load_state_dict_post_hook(lambda module, incompatible: self.refresh_bf16())
        # sharded optimiser: the fp32 masters of the trunk weights are current on one rank each -- reading them without a sync would
        # silently save stale weights, so state_dict() refuses until sync_master() has run on every rank (Trainer.state_dict does both)
        self._sd_hook = model.register_state_dict_pre_hook(lambda module, prefix, keep_vars: self._guard_stale())
        self._img = None
        self._label = None
        self._g_fb = None
        self._g_opt = None
        self._loss = None
        self._eager_steps = 0
        self._side = None
        self._copy_stream = None
        self._pf_img = self._pf_label = None
        self._pf_ready = self._pf_taken = None

    def refresh_bf16(self):
        """Re-cast the fp32 master weights into the persistent bf16 copy (normally refreshed inside the optimiser step only).
        Call after writing to the parameters by hand; load_state_dict() does it through a post-hook."""
        if self.graph and hasattr(self.opt, "flat_param16"):
            self.sync_master()
            self.opt.flat_param16.copy_(self.opt.flat_param)

    def _guard_stale(self):
        if self.sharded and self._master_stale:
            raise RuntimeError("Trainer (sharded optimiser): the fp32 master weights are sharded across ranks; call trainer.sync_master() "
                               "-- or trainer.state_dict() -- on EVERY rank before reading model.state_dict()")

    def state_dict(self):
        """model.state_dict() with every rank's fp32 master weights made current first (a collective: call it on all ranks)."""
        self.sync_master()
        return self.model.state_dict()

    def sync_master(self):
        """Sharded optimiser only: make every rank's fp32 master weights current again (each rank updates only its slice of the
        trunk's Linear weights during training).  Call before reading the parameters in fp32: state_dict() / checkpoints,
        evaluation or CAM inference on the trained model, check_replicas_in_sync() (which calls it)."""
        if self.sharded and self._master_stale:
            self.buckets.all_gather_shards(self.opt.flat_param)
            self.buckets.all_gather_shards(self.opt.buf)
            self._master_stale = False

    def check_replicas_in_sync(self):
        """Max |parameter checksum difference| across ranks (0.0 on one rank): every rank must hold bit-identical weights after
        an all-reduced step.  One small all-gather; meant for tests and bench.py, not for the hot loop."""
        self.sync_master()
        flat = self.opt.flat_param if self.graph else torch.cat([p.detach().reshape(-1).float() for p in self.buckets.params])
        cs = torch.stack([flat.double().sum(), flat.double().abs().sum(), (flat.double() * flat.double()).sum()])
        if self.world == 1:
            return 0.0
        allcs = [torch.empty_like(cs) for _ in range(self.world)]
        dist.all_gather(allcs, cs)
        ref = allcs[0]
        return float(max(((c - ref).abs() / (ref.abs() + 1e-300)).max() for c in allcs))

    def _stage(self, img, label):
        if self._img is None or self._img.shape != img.shape:
            if self._g_fb is not None:
                raise RuntimeError("Trainer: input shape changed after CUDA-graph capture")
            self._img = torch.empty(img.shape, device=self.dev, dtype=img.dtype)
            self._label = torch.empty(label.shape, device=self.dev, dtype=label.dtype)
        self._img.copy_(img, non_blocking=True)
        self._label.copy_(label, non_blocking=True)
        return self._img, self._label

    def prefetch(self, img, label):
        """Start the host->device copy of the NEXT batch (pinned host tensors) on a copy stream; it overlaps whatever the
        compute stream is doing (normally the current step).  Consume it with step() called without arguments.  The
        reference loads and copies synchronously inside the step loop (train_acr.py:127-133)."""
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(device=self.dev)
            self._pf_img = torch.empty(img.shape, device=self.dev, dtype=img.dtype)
            self._pf_label = torch.empty(label.shape, device=self.dev, dtype=label.dtype)
        cs = self._copy_stream
        if self._pf_taken is not None:
            cs.wait_event(self._pf_taken)            # the previous prefetched batch has been moved into the step's input buffers
        with torch.cuda.stream(cs):
            self._pf_img.copy_(img, non_blocking=True)
            self._pf_label.copy_(label, non_blocking=True)
            self._pf_ready = torch.cuda.Event()
            self._pf_ready.record(cs)

    def _take_prefetched(self):
        if self._pf_ready is None:
            raise RuntimeError("Trainer.step() without arguments needs a preceding prefetch()")
        cur = torch.cuda.current_stream(self.dev)
        cur.wait_event(self._pf_ready)
        self._pf_ready = None
        img, label = self._stage(self._pf_img, self._pf_label)      # device-to-device into the (graph-captured) input buffers
        self._pf_taken = torch.cuda.Event()
        self._pf_taken.record(cur)
        return img, label

    def step_prefetched(self, next_img, next_label):
        """One step on the batch given to the previous prefetch() / step_prefetched() call, while the copy of
        (next_img, next_label) -- pinned host tensors -- runs underneath it."""
        img, label = self._take_prefetched()
        self.prefetch(next_img, next_label)
        return self.step(img, label)

    def _dense_crf_term(self, img, cls_list):
        """DenseCRF regulariser (losses.dense_crf_loss over this repo's permutohedral filter) for the step's first view."""
        import torch.nn.functional as F
        from .losses import dense_crf_loss, dense_crf_loss_from_patch_logits
        o = self.dense_crf
        B, _, S, _ = img.shape
        p = S // 16
        layer_4 = self.model.pretrained.activations["4"][:B]                  # view 1 (both views ran as one batch of 2B)
        logits = self.model.cls_head(layer_4[:, 1:, :])                         # [B, p*p, C] patch-token logits (DPT/ACR.py:133-134)
        ori = (img * o["std"] + o["mean"]).clamp(0.0, 255.0)
        if o["scale"] == 0.5 and S % 2 == 0 and img.is_cuda:
            # up-sampling, softmax over [background, classes] and the rloss down-scaling as one kernel: the [B,C+1,S,S] tensors
            # of the composition below (0.5 GB each at 448x448, C = 80, six passes forward and backward) never exist
            return dense_crf_loss_from_patch_logits(ori, logits, o["weight"], o["sigma_rgb"], o["sigma_xy"], o["scale"])
        logits = logits.permute(0, 2, 1).reshape(B, -1, p, p)
        logits = F.interpolate(logits, (S, S), mode="bilinear", align_corners=False)
        seg = torch.softmax(torch.cat([torch.zeros_like(logits[:, :1]), logits], dim=1), dim=1)      # K = C + 1, background first
        roi = torch.ones(B, S, S, device=img.device)
        return dense_crf_loss(ori, seg, roi, o["weight"], o["sigma_rgb"], o["sigma_xy"], o["scale"])

    def _forward_backward(self, img, label):
        img2 = img.flip(-1)                                   # transforms.RandomHorizontalFlip(p=1), train_acr.py:135
        with ops.direct_grads():          # gradients land straight in the flat fp32 buffer (see ops.DIRECT_GRADS)
            cls_list, (attn1, attn2) = self.model.forward_mirror(img, img2)
            loss, parts = acr_total_loss(cls_list[0], cls_list[1], label, attn1, attn2, img.shape[2] // 16, self.alpha)
            if self.dense_crf is not None:
                loss = loss + self._dense_crf_term(img, cls_list)
            self.buckets.zero()
            loss.backward()
        return loss.detach()

    def step(self, img=None, label=None):
        if img is None:
            img, label = self._take_prefetched()
        if not self.graph:
            if not img.is_cuda:
                img, label = self._stage(img, label)
            loss = self._forward_backward(img, label)
            self.buckets.finish()
            self.opt.step()
            return loss
        if img is not self._img:
            img, label = self._stage(img, label)
        if self._g_fb is None and self._eager_steps < 2:
            # warm-up eagerly (lazy initialisation inside the kernels' host code, cuBLAS workspaces, autotuning) on the
            # SAME side stream the capture will use, so autograd's gradient-accumulation nodes are bound to it
            self._eager_steps += 1
            if self._side is None:
                self._side = torch.cuda.Stream()
            self._side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(self._side):
                loss = self._forward_backward(img, label)
            torch.cuda.current_stream().wait_stream(self._side)
            self._reduce_and_update()
            return loss
        if self._g_fb is None:
            torch.cuda.synchronize()
            self._g_fb = torch.cuda.CUDAGraph()
            with ops.cuda_graph_capture(self._g_fb, self._side):
                self._loss = self._forward_backward(img, label)
            self._g_opt = torch.cuda.CUDAGraph()
            with ops.cuda_graph_capture(self._g_opt, self._side):
                self.opt.update()
            self._g_fb.replay()              # the capture itself did not execute the step
        else:
            self._g_fb.replay()
        self._reduce_and_update()
        return self._loss

    def _reduce_and_update(self):
        """Gradient all-reduce + optimiser step.  One rank: the captured optimiser kernel.  Several ranks: the flat gradient buffer
        is all-reduced in `reduce_chunks` slices and each slice is updated (one kernel launch) as soon as its collective has
        finished (with more than one slice the optimiser pass can run under the remaining NCCL traffic)."""
        self.opt.set_lr_for_step()
        if self.world == 1:
            if self._g_opt is not None:
                self._g_opt.replay()
            else:
                self.opt.update()
            return
        if self.sharded:
            b = self.buckets
            b.reduce_sharded()
            s, e = b.shard_range()
            self.opt.update(s, e, grad=b.grad_shard)                    # this rank's slice of the trunk weights
            if b.flat.numel() > b.shard_end:
                self.opt.update(b.shard_end, b.flat.numel())            # the replicated rest, identical on every rank
            b.all_gather_shards(self.opt.flat_param16)                  # everyone's refreshed bf16 weights
            self._master_stale = True
            return
        for s, e in self.buckets.reduce_chunks(self.reduce_chunks):
            self.opt.update(s, e)
