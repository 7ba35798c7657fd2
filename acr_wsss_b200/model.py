"""Host-side mirror of the reference's model interface for the hot path.

Mirrors (same class / method names, argument meaning, return structures and state_dict keys):
  * models/vision_transformer.py:167-214  Attention  (forward, get_attn, get_attn_gradients, qkv/proj/num_heads/scale)
  * models/vision_transformer.py:216-233  Block, :148-164 Mlp, :449-504 forward_flex / _resize_pos_embed
  * DPT/ACR.py:40-143  DPT.forward_cls / forward_cam,  :147-215  ACR.forward_mirror / getam / load

Only the attention core, the head mean / stack and GETAM run in this repo's kernels; LayerNorm, the Linear
layers, GELU and the patch convolution are library calls (SURVEY section 2, row 2: "GEMMs stay library").
"""
import math

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import ops

_BACKBONES = {
    # name -> (embed_dim, depth, heads, hooks, scratch in-features)
    "vitb16_384": (768, 12, 12, [2, 5, 8, 11], [96, 192, 384, 768]),
    "deitb16_384": (768, 12, 12, [2, 5, 8, 11], [96, 192, 384, 768]),
    "vitl16_384": (1024, 24, 16, [5, 11, 17, 23], [256, 512, 1024, 1024]),
}
_BACKBONE_ALIASES = {"vitb": "vitb16_384", "deit": "deitb16_384", "vitl": "vitl16_384"}


def _cached(mod, x):
    return getattr(mod, "_w16", None) is not None and x.dtype == torch.bfloat16 and torch.is_grad_enabled()


def _lin(mod, x, skip_bias_grad=False):
    """nn.Linear call; uses the module's cached bf16 weight copy (set by Trainer) when there is one.
    skip_bias_grad: the caller folds this layer's bias gradient into the following add_layer_norm (cached path only)."""
    if _cached(mod, x):
        return ops.linear_cached_bf16(x, mod.weight, mod.bias, mod._w16, getattr(mod, "_b16", None), skip_bias_grad)
    assert not skip_bias_grad
    return mod(x)


def _fold_bias(mod, x):
    """The bias Parameter whose gradient add_layer_norm's backward can take over (cached bf16 path with fp32 .grad), or None."""
    b = mod.bias
    if ops.DIRECT_GRADS and b is not None and _cached(mod, x) and b.requires_grad and b.grad is not None and b.grad.dtype == torch.float32:
        return b
    return None


class Attention(nn.Module):
    """Drop-in for models/vision_transformer.py:167-214.

    precision 'fp32': exact path, P and dP are materialised, so get_attn()/get_attn_gradients() return the
    same [B,H,N,N] tensors as the reference.  precision 'bf16': fused tcgen05 kernel; P never reaches HBM,
    get_attn() recomputes it on demand from the saved qkv, and only row 0 of dP is kept (all GETAM needs).
    """

    def __init__(self, dim, num_heads=8, qkv_bias=False, qk_scale=None, attn_drop=0., proj_drop=0., precision="fp32"):
        super().__init__()
        if attn_drop != 0. or proj_drop != 0.:
            raise NotImplementedError("the ACR path runs with attn_drop = proj_drop = 0 (vision_transformer.py:205)")
        self.num_heads = num_heads
        head_dim = dim // num_heads
        self.scale = qk_scale or head_dim ** -0.5
        self.qkv = nn.Linear(dim, dim * 3, bias=qkv_bias)
        self.proj = nn.Linear(dim, dim)
        self.precision = precision
        self.capture_grad = True       # keep dP (fp32) / its row 0 (bf16) in backward, like the reference hook
        self._state = {}
        self._slot = None              # [B,N,N] view of this block's slot in the [B,L,N,N] stack
        self.attn_mean = None          # head-mean map of the last recorded forward

    # -- accessor protocol (vision_transformer.py:186-196) --
    def get_attn(self):
        st = self._state
        if st.get("attn") is not None:
            return st["attn"]
        if st.get("qkv") is not None:          # fused path: recompute on demand through the exact kernels
            qkv = st["qkv"].float()
            with torch.no_grad():
                tmp = {}
                ops.attention_core(qkv, self.num_heads, self.scale, None, tmp, "fp32")
            return tmp["attn"]
        return None

    def get_attn_gradients(self):
        """dP [B,H,N,N] of the last backward (what the reference's hook keeps, vision_transformer.py:192-193,209).  The exact path
        stores it; the fused path never forms it (the backward kernel keeps row 0 only, which is all getam uses), so it is
        recomputed here on demand from what that backward saw: dP_h = dO_h V_h^T (+ G/H when an affinity gradient came with it)."""
        st = self._state
        if st.get("attn_grad") is not None:
            return st["attn_grad"]
        if st.get("d_out") is not None and st.get("qkv") is not None:
            qkv, d_out = st["qkv"], st["d_out"]
            B, N, _ = qkv.shape
            H = self.num_heads
            v = qkv.view(B, N, 3, H, -1)[:, :, 2].float()                      # [B,N,H,D]
            dP = torch.einsum("bnhd,bmhd->bhnm", d_out.view(B, N, H, -1).float(), v)
            if st.get("g_dense") is not None:
                dP = dP + st["g_dense"].unsqueeze(1) / H
            return dP
        return None

    def get_attn_row0(self):
        """Per-head cls-token row of P, [B,H,N]."""
        st = self._state
        if st.get("row0") is not None:
            return st["row0"]
        return st["attn"][:, :, 0, :] if st.get("attn") is not None else None

    def get_attn_gradients_row0(self):
        st = self._state
        if st.get("grad_row0") is not None:
            return st["grad_row0"]
        return st["attn_grad"][:, :, 0, :] if st.get("attn_grad") is not None else None

    def forward(self, x, skip_bias_grad=False):
        B, N, C = x.shape
        qkv = _lin(self.qkv, x)
        # The reference refreshes its saved map only when x.requires_grad (vision_transformer.py:207-209).
        record = x.requires_grad
        state = None
        if record:
            state = {"capture_grad": self.capture_grad}
        out, mean = ops.attention_core(qkv, self.num_heads, self.scale, self._slot if record else None, state,
                                       self.precision)
        if record:
            self._state = state
            self.attn_mean = mean
        out = out.to(x.dtype) if out.dtype != x.dtype and not torch.is_autocast_enabled() else out
        return _lin(self.proj, out, skip_bias_grad)


class Mlp(nn.Module):
    def __init__(self, in_features, hidden_features=None, out_features=None):
        super().__init__()
        out_features = out_features or in_features
        hidden_features = hidden_features or in_features
        self.fc1 = nn.Linear(in_features, hidden_features)
        self.act = nn.GELU()
        self.fc2 = nn.Linear(hidden_features, out_features)

    def forward(self, x, skip_bias_grad=False):
        w16 = getattr(self.fc1, "_w16", None)
        if w16 is not None and x.dtype == torch.bfloat16 and x.is_cuda and torch.is_grad_enabled():
            h = ops.linear_gelu_cached_bf16(x, self.fc1.weight, self.fc1.bias, w16, getattr(self.fc1, "_b16", None))
        else:
            h = self.act(_lin(self.fc1, x))
        return _lin(self.fc2, h, skip_bias_grad)


class Block(nn.Module):
    def __init__(self, dim, num_heads, mlp_ratio=4., qkv_bias=True, precision="fp32"):
        super().__init__()
        self.norm1 = nn.LayerNorm(dim, eps=1e-6)
        self.attn = Attention(dim, num_heads=num_heads, qkv_bias=qkv_bias, precision=precision)
        self.norm2 = nn.LayerNorm(dim, eps=1e-6)
        self.mlp = Mlp(dim, int(dim * mlp_ratio))

    def _norm(self, ln, x):
        # bf16 path: this repo's LayerNorm kernel writes the Linear's bf16 operand directly (no cast kernel, and a
        # single-pass backward); fp32 path: stock nn.LayerNorm, exactly the reference's call
        if self.attn.precision == "bf16" and x.is_cuda and x.shape[-1] % 128 == 0:
            return ops.layer_norm(x, ln.weight, ln.bias, ln.eps, out_bf16=True)
        return ln(x)

    def forward(self, x):
        x = x + self.attn(self._norm(self.norm1, x))
        x = x + self.mlp(self._norm(self.norm2, x))
        return x

    def fused_ok(self, x):
        return self.attn.precision == "bf16" and x.is_cuda and x.dtype == torch.bfloat16 and x.shape[-1] % 128 == 0

    def forward_stream(self, x, pending, pending_bias=None, fold_out=True):
        """Same arithmetic as forward() with the residual adds folded into the LayerNorm kernels.  The residual stream
        travels as (x, pending) with the true value x + pending.  Returns (stream, pending branch, bias Parameter whose
        gradient the NEXT add_layer_norm must produce (or None), this block's input)."""
        if pending is None:
            s, h = x, self._norm(self.norm1, x)
        else:
            s, h = ops.add_layer_norm(x, pending, self.norm1.weight, self.norm1.bias, self.norm1.eps, out_bf16=True,
                                      branch_bias=pending_bias)
        pb = _fold_bias(self.attn.proj, h)
        s2, h2 = ops.add_layer_norm(s, self.attn(h, pb is not None), self.norm2.weight, self.norm2.bias, self.norm2.eps,
                                    out_bf16=True, branch_bias=pb)
        fb = _fold_bias(self.mlp.fc2, h2) if fold_out else None
        return s2, self.mlp(h2, fb is not None), fb, s


class PatchEmbed(nn.Module):
    def __init__(self, img_size=384, patch_size=16, in_chans=3, embed_dim=768):
        super().__init__()
        self.proj = nn.Conv2d(in_chans, embed_dim, kernel_size=patch_size, stride=patch_size)


_BILINEAR = {}


def _bilinear_matrix(n_in, n_out, device):
    """[n_out, n_in] weights of F.interpolate(mode="bilinear", align_corners=False) along one axis: output d reads
    src = (d + 0.5) * n_in / n_out - 0.5 (clamped at 0) from its two neighbours.  Built with device ops, so a first call inside a
    CUDA-graph capture is captured too; kept for reuse only outside one (a captured tensor holds nothing until the replay)."""
    key = (n_in, n_out, str(device))
    m = _BILINEAR.get(key)
    if m is None:
        src = ((torch.arange(n_out, dtype=torch.float32, device=device) + 0.5) * (n_in / n_out) - 0.5).clamp(min=0.0)
        i0 = src.floor()
        l1 = src - i0
        i1 = torch.clamp(i0 + 1, max=n_in - 1)
        cols = torch.arange(n_in, dtype=torch.float32, device=device)
        m = (cols == i0[:, None]) * (1.0 - l1)[:, None] + (cols == i1[:, None]) * l1[:, None]
        if not (m.is_cuda and torch.cuda.is_current_stream_capturing()):
            _BILINEAR[key] = m
    return m


class _ResizeGrid(torch.autograd.Function):
    """F.interpolate(grid [1,E,g,g], (gs_h, gs_w), mode="bilinear").  The backward is mh^T . grad . mw with the interpolation
    matrices instead of the library's atomic scatter, whose summation order (and so the gradient's rounding) changes from run
    to run."""

    @staticmethod
    def forward(ctx, grid, gs_h, gs_w):
        ctx.sizes = (grid.shape[-1], gs_h, gs_w)
        return F.interpolate(grid, size=(gs_h, gs_w), mode="bilinear")

    @staticmethod
    def backward(ctx, grad):
        gs_old, gs_h, gs_w = ctx.sizes
        mh, mw = (_bilinear_matrix(gs_old, n, grad.device).to(grad.dtype) for n in (gs_h, gs_w))
        return mh.t() @ grad @ mw, None, None


def _trunc_normal_(t, std=.02):
    return nn.init.trunc_normal_(t, std=std, a=-2., b=2.)


class VisionTransformer(nn.Module):
    """The parts of models/vision_transformer.py:VisionTransformer the ACR path touches (forward_flex)."""

    def __init__(self, img_size=384, patch_size=16, embed_dim=768, depth=12, num_heads=12, num_classes=1000,
                 precision="fp32"):
        super().__init__()
        self.patch_size = [patch_size, patch_size]
        self.residual = "auto"         # bf16 path: "auto" (bf16 stream in train mode, fp32 in eval mode), "bf16" or "fp32"
        self.start_index = 1
        self.embed_dim = embed_dim
        self.patch_embed = PatchEmbed(img_size, patch_size, 3, embed_dim)
        num_patches = (img_size // patch_size) ** 2
        self.cls_token = nn.Parameter(torch.zeros(1, 1, embed_dim))
        self.bkg_token = nn.Parameter(torch.zeros(1, 1, embed_dim))
        self.pos_embed = nn.Parameter(torch.zeros(1, num_patches + 1, embed_dim))
        self.blocks = nn.ModuleList([Block(embed_dim, num_heads, 4., True, precision) for _ in range(depth)])
        self.norm = nn.LayerNorm(embed_dim, eps=1e-6)
        self.head = nn.Linear(embed_dim, num_classes)
        # init as vision_transformer.py:339-349,548
        _trunc_normal_(self.pos_embed)
        _trunc_normal_(self.cls_token)
        _trunc_normal_(self.bkg_token)
        self.apply(self._init_weights)

    @staticmethod
    def _init_weights(m):
        if isinstance(m, nn.Linear):
            _trunc_normal_(m.weight)
            if m.bias is not None:
                nn.init.zeros_(m.bias)
        elif isinstance(m, nn.LayerNorm):
            nn.init.zeros_(m.bias)
            nn.init.ones_(m.weight)

    def _resize_pos_embed(self, posemb, gs_h, gs_w):
        # vision_transformer.py:490-504
        posemb_tok, posemb_grid = posemb[:, :self.start_index], posemb[0, self.start_index:]
        gs_old = int(math.sqrt(len(posemb_grid)))
        posemb_grid = posemb_grid.reshape(1, gs_old, gs_old, -1).permute(0, 3, 1, 2)
        posemb_grid = _ResizeGrid.apply(posemb_grid, gs_h, gs_w)
        posemb_grid = posemb_grid.permute(0, 2, 3, 1).reshape(1, gs_h * gs_w, -1)
        return torch.cat([posemb_tok, posemb_grid], dim=1)

    def forward_flex(self, x, last_block_out=None, replicate_at=None, replicas=1, need_norm=True):
        """vision_transformer.py:449-486.  Returns (norm(x), None); `last_block_out`, if a list, receives the
        un-normalised output of the last block (what the reference reads through its forward hook, Q4).
        replicate_at / replicas: batched GETAM (SURVEY 8f rank 1) -- the input of block `replicate_at` is detached and
        repeated `replicas` times along the batch, so ONE backward with one one-hot cotangent per replica yields the
        per-class attention gradients of blocks >= replicate_at; the replicated leaf is kept in self._rep_in.
        need_norm=False skips the final LayerNorm (returns (None, None)): the ACR heads read the un-normalised output of
        the last block (DPT/ACR.py:95-96 discards the return value and reads activations["4"]), so on that path the reference computes norm(x) and drops it."""
        b, c, h, w = x.shape
        pos_embed = self._resize_pos_embed(self.pos_embed, h // self.patch_size[1], w // self.patch_size[0])
        # patch_embed.proj is a stride-16 16x16 convolution (vision_transformer.py:463-464) == one GEMM over
        # unfolded patches; done as a Linear so fp32 stays true fp32 (cuDNN convolutions default to TF32).
        ph, pw = h // self.patch_size[1], w // self.patch_size[0]
        P = self.patch_size[0]
        proj = self.patch_embed.proj
        x = x.reshape(b, c, ph, P, pw, P).permute(0, 2, 4, 1, 3, 5).reshape(b, ph * pw, c * P * P)
        x = F.linear(x, proj.weight.reshape(proj.weight.shape[0], -1), proj.bias)
        cls_tokens = self.cls_token.expand(b, -1, -1)
        x = torch.cat((cls_tokens.to(x.dtype), x), dim=1)
        x = x + pos_embed.to(x.dtype)
        self._block_in = []            # input of every block (references): lets GETAM stop its backward at start_layer
        self._rep_in = None

        def replicate(t):       # sample b -> copies b*replicas .. b*replicas + replicas - 1
            t = t.detach().repeat_interleave(replicas, dim=0).requires_grad_(True)
            self._rep_in = t
            return t

        # Residual stream of the bf16 path.  Training keeps it in bf16 (the add is folded into the LayerNorm kernels and the
        # stream is read / written once per LayerNorm in 2-byte elements); inference (eval mode) keeps it in fp32 like stock
        # bf16 autocast does: 24 roundings of the stream to bf16 are what separates the CAMs from the fp32 reference
        # (patch CAM 1.6e-2 -> 0.85e-2 of the reference at 448x448, scripts/diag_bf16_448.py), and speed is not at stake there.
        if self.residual == "fp32" or (self.residual == "auto" and not self.training):
            x = x.float()
        if len(self.blocks) and self.blocks[0].fused_ok(x):
            pending = pbias = None
            for i, blk in enumerate(self.blocks):        # the last block's branch meets a plain add: it keeps its own bias gradient
                if i == replicate_at:
                    assert pbias is None, "batched GETAM runs outside the training path"
                    x, pending = replicate(x if pending is None else x + pending), None
                x, pending, pbias, blk_in = blk.forward_stream(x, pending, pbias, fold_out=i + 1 < len(self.blocks))
                self._block_in.append(blk_in)
            x = x + pending
        else:
            for i, blk in enumerate(self.blocks):
                if i == replicate_at:
                    x = replicate(x)
                self._block_in.append(x)
                x = blk(x)
        if last_block_out is not None:
            last_block_out.append(x)
        return (self.norm(x) if need_norm else None), None


class _Pretrained(nn.Module):
    def __init__(self, model):
        super().__init__()
        self.model = model
        self.activations = {}


class _Scratch(nn.Module):
    def __init__(self, in_shape, features=256):
        super().__init__()
        # DPT/blocks.py _make_scratch: present in the state_dict, dead on the ACR path
        for i, c in enumerate(in_shape):
            setattr(self, f"layer{i + 1}_rn", nn.Conv2d(c, features, kernel_size=3, stride=1, padding=1, bias=False))


class ACR(nn.Module):
    """Drop-in for DPT/ACR.py:147-215 (class ACR) and :40-143 (class DPT) on the plain-ViT backbones.

    ACR(num_classes, backbone_name, path=None, precision='fp32'|'bf16').  `use_pretrain` is accepted and
    ignored (weights are random-init or come from `path` / load_state_dict; there is no network here).
    """

    def __init__(self, num_classes, backbone_name, path=None, precision="fp32", features=256, **kwargs):
        super().__init__()
        self.num_class = num_classes
        cur = _BACKBONE_ALIASES.get(backbone_name, backbone_name)
        if cur not in _BACKBONES:
            raise NotImplementedError(f"backbone {backbone_name!r}: only the plain ViT backbones are on the hot path "
                                      "(SURVEY section 2 rows 13-14)")
        self.cur_backbone = cur
        self.precision = precision
        dim, depth, heads, hooks, scratch_in = _BACKBONES[cur]
        self.hooks = hooks
        self.pretrained = _Pretrained(VisionTransformer(384, 16, dim, depth, heads, 1000, precision))
        self.scratch = _Scratch(scratch_in, features)
        # The reference hard-codes 768 (DPT/ACR.py:88), which breaks ViT-L (SURVEY Q6); use the trunk width.
        self.cls_head = nn.Linear(dim, num_classes)
        self.use_gap = True
        self.fuse_views = True
        if path is not None:
            self.load(path)

    def load(self, path):
        parameters = torch.load(path, map_location=torch.device("cpu"))
        if "optimizer" in parameters:
            parameters = parameters["model"]
        self.load_state_dict(parameters)

    def set_capture_grad(self, flag):
        for blk in self.pretrained.model.blocks:
            blk.attn.capture_grad = flag

    # ------------------------------------------------------------------ trunk
    def _trunk(self, x, split_views=False):
        vit = self.pretrained.model
        B = x.shape[0]
        p_h, p_w = x.shape[2] // 16, x.shape[3] // 16
        N = p_h * p_w + 1
        L = len(vit.blocks)
        stack = None
        record = torch.is_grad_enabled()
        if record:
            stack = torch.empty(B, L, N, N, device=x.device, dtype=torch.float32)
        for l, blk in enumerate(vit.blocks):
            blk.attn._slot = stack[:, l] if record else None
        last = []
        if self.precision == "bf16":
            with torch.autocast("cuda", dtype=torch.bfloat16):
                vit.forward_flex(x, last, need_norm=False)
        else:
            vit.forward_flex(x, last, need_norm=False)
        layer_4 = last[0].float()
        self.pretrained.activations["4"] = layer_4
        for blk in vit.blocks:
            blk.attn._slot = None
        if record and split_views:
            attn = ops.stack_views_split(stack, [blk.attn.attn_mean for blk in vit.blocks], [blk.attn._state for blk in vit.blocks])
        elif record:
            attn = ops.stack_views(stack, [blk.attn.attn_mean for blk in vit.blocks], [blk.attn._state for blk in vit.blocks])
        else:
            # no_grad: the reference returns the stale maps of the last recorded forward (SURVEY Q3)
            maps = [blk.attn.attn_mean for blk in vit.blocks]
            attn = torch.stack(maps, dim=1) if all(m is not None for m in maps) else None
        return layer_4, attn

    def forward_cls(self, x):
        """DPT/ACR.py:92-116 -> (x_cls [B,C], x_patch_cls [B,C], attn [B,L,N,N], None)."""
        layer_4, attn = self._trunk(x)
        x_cls = layer_4[:, 0, :]
        x_patch = layer_4[:, 1:, :]
        x_patch_cls = self.cls_head(x_patch.mean(dim=1))
        x_cls = self.cls_head(x_cls)
        return x_cls, x_patch_cls, attn, None

    def forward_cam(self, x):
        """DPT/ACR.py:118-143 -> (x_cls, x_patch_cls, attn [B,L,N,N], x_patch_cam [B,N-1,C])."""
        layer_4, attn = self._trunk(x)
        x_cls = layer_4[:, 0, :]
        x_patch = layer_4[:, 1:, :]
        x_cls = self.cls_head(x_cls)
        x_patch_cls = self.cls_head(x_patch.mean(dim=1))
        x_patch_cam = self._patch_cam(x_patch)
        return x_cls, x_patch_cls, attn, x_patch_cam

    def _patch_cam(self, x_patch):
        """relu(cls_head(x_patch)), DPT/ACR.py:133-134, on the tensor cores (csrc/refine_tc.cu) when the tokens live on a GPU."""
        if x_patch.is_cuda and x_patch.dtype == torch.float32 and x_patch.stride(2) == 1 and self.cls_head.out_features <= 128:
            return ops.patch_cam(x_patch, self.cls_head.weight, self.cls_head.bias)
        return F.relu(self.cls_head(x_patch))

    def forward_cam_batched(self, x, replicas, start_layer):
        """forward_cam with the blocks >= start_layer run on `replicas` identical copies of every sample (batched GETAM,
        SURVEY 8f rank 1); copy k of sample b sits at batch index b*replicas + k.  Returns (x_cls [B*replicas,C],
        x_patch_cls [B,C], attn [B,L,N,N], x_patch_cam [B,N-1,C]); follow with backward_for_getam_batched(x_cls, classes)."""
        assert replicas >= 1
        vit = self.pretrained.model
        B = x.shape[0]
        p_h, p_w = x.shape[2] // 16, x.shape[3] // 16
        N = p_h * p_w + 1
        L = len(vit.blocks)
        stack = torch.empty(B, L, N, N, device=x.device, dtype=torch.float32)
        rep = torch.empty(B * replicas, L - start_layer, N, N, device=x.device, dtype=torch.float32)
        for l, blk in enumerate(vit.blocks):
            blk.attn._slot = stack[:, l] if l < start_layer else rep[:, l - start_layer]
        last = []
        with torch.enable_grad():
            if self.precision == "bf16":
                with torch.autocast("cuda", dtype=torch.bfloat16):
                    vit.forward_flex(x, last, replicate_at=start_layer, replicas=replicas, need_norm=False)
            else:
                vit.forward_flex(x, last, replicate_at=start_layer, replicas=replicas, need_norm=False)
            layer_4 = last[0].float()
            x_cls = self.cls_head(layer_4[:, 0, :])
        for blk in vit.blocks:
            blk.attn._slot = None
        stack[:, start_layer:] = rep[::replicas]
        self.pretrained.activations["4"] = layer_4
        with torch.no_grad():
            x_patch = layer_4[::replicas, 1:, :]
            x_patch_cls = self.cls_head(x_patch.mean(dim=1))
            x_patch_cam = self._patch_cam(x_patch)
        return x_cls, x_patch_cls, stack, x_patch_cam

    def backward_for_getam_batched(self, x_cls, classes):
        """One backward for all copies: batch index i receives the one-hot cotangent of classes[i] (infer_cam.py:173-179
        runs one full backward per class).  Afterwards getam(i, start_layer, ...) is the GETAM of classes[i] for that copy."""
        idx = classes if torch.is_tensor(classes) else torch.as_tensor(list(classes), device=x_cls.device)
        sel = x_cls.gather(1, idx.view(-1, 1)).sum()
        torch.autograd.grad(sel, self.pretrained.model._rep_in)

    def forward_mirror(self, x1, x2):
        """DPT/ACR.py:170-174.  The reference runs the two views one after the other; nothing on the path couples
        samples of a batch (LayerNorm is per token, there is no BatchNorm), so with `fuse_views` both views go through
        the trunk as ONE batch of 2B -- same results, half the launches, larger GEMMs."""
        if self.fuse_views and torch.is_grad_enabled() and x1.shape == x2.shape:
            B = x1.shape[0]
            layer_4, (attn1, attn2) = self._trunk(torch.cat([x1, x2], dim=0), split_views=True)
            x_cls = self.cls_head(layer_4[:, 0, :])
            x_p_cls = self.cls_head(layer_4[:, 1:, :].mean(dim=1))
            return [x_cls[:B], x_cls[B:], x_p_cls[:B], x_p_cls[B:], None, None], [attn1, attn2]
        x_cls_1, x_p_cls_1, attn1, b1 = self.forward_cls(x1)
        x_cls_2, x_p_cls_2, attn2, b2 = self.forward_cls(x2)
        return [x_cls_1, x_cls_2, x_p_cls_1, x_p_cls_2, b1, b2], [attn1, attn2]

    def getam(self, batch, start_layer=0, func="grad", full=False):
        """DPT/ACR.py:177-215.  Returns (cls_cam [1,N-1], attn_list, cam_list).

        attn_list[l] is the head-mean map [B,N,N] as in the reference.  cam_list[l] is c_l restricted to
        row 0, shape [1,1,N] (the only row the reference's result and its caller use, DPT/ACR.py:213 /
        infer_cam.py:180-184); pass full=True to get the reference's full [1,N,N] maps (on the fused path P and dP are
        recomputed on demand for that, see Attention.get_attn / get_attn_gradients).
        """
        blocks = self.pretrained.model.blocks
        skip = 1      # (2 for the distilled DeiT variant, DPT/ACR.py:210-211: a hybrid/distilled backbone is outside the hot path --
        #               the constructor rejects it; the kernels keep the `skip` argument)
        attn_list = [blk.attn.attn_mean for blk in blocks]
        used = blocks[start_layer:]          # only these reach the result (DPT/ACR.py:208-209), so only they need a gradient
        p0 = torch.stack([blk.attn.get_attn_row0()[batch] for blk in used])              # [L',H,N]
        g0 = torch.stack([blk.attn.get_attn_gradients_row0()[batch] for blk in used])    # [L',H,N]
        cls_cam, rows = ops.getam_row0(p0, g0, 0, func, skip, want_rows=True)
        if full:
            cam_list = [_getam_full(blk.attn.get_attn()[batch], blk.attn.get_attn_gradients()[batch], func).unsqueeze(0)
                        for blk in used]
        else:
            cam_list = [rows[l].view(1, 1, -1) for l in range(len(used))]
        return cls_cam, attn_list, cam_list

    def getam_batch(self, start_layer=0, func="grad"):
        """getam() for EVERY sample of the last (batched) forward / backward at once: [S, N-skip] (row s = getam(s, ...)[0][0]);
        one kernel launch instead of S (batched CAM inference)."""
        blocks = self.pretrained.model.blocks
        skip = 1
        used = blocks[start_layer:]
        p0 = torch.stack([blk.attn.get_attn_row0() for blk in used])               # [L',S,H,N]
        g0 = torch.stack([blk.attn.get_attn_gradients_row0() for blk in used])
        return ops.getam_row0_batch(p0, g0, 0, func, skip)

    def backward_for_getam(self, logit, start_layer=0):
        """Gradient pass that feeds getam().  The reference calls logit.backward(retain_graph=True) through the whole
        model and all parameters (infer_cam.py:173-179); only dP of blocks >= start_layer is ever read, so this stops
        at the input of block `start_layer` and accumulates no parameter gradients (same GETAM result)."""
        torch.autograd.grad(logit, self.pretrained.model._block_in[start_layer], retain_graph=True)


def _getam_full(cam, grad, func):
    # DPT/ACR.py:187-206 on full [H,N,N] maps (fp32 path only; not on the hot path)
    pos = grad.clamp(min=0).mean(dim=0)
    if func == "grad":
        return pos
    if func == "grad_s":
        return pos * pos
    gp = (grad * cam).clamp(min=0).mean(dim=0)
    return gp if func == "cam_grad" else gp * pos
