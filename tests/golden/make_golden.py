"""Generates tests/golden/*.npz by EXECUTING the unmodified reference (Python imported from
/root/reference, C++ compiled by oracle/Makefile into oracle/_ref) on seeded synthetic inputs.

Run in the build container only:   python tests/golden/make_golden.py
The inline blocks of train_acr.py:140-168 and infer_cam.py:145-215 cannot be imported (the scripts need
matplotlib / pydensecrf and run argparse at import), so their lines are restated here around the
reference model's own outputs; everything else below is the reference's code running.
"""
import os
import sys

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle.refimport import loader          # noqa: E402
from oracle import acr_oracle as orc         # noqa: E402
from oracle import bilateral_oracle as bo    # noqa: E402
from acr_wsss_b200 import synth              # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
torch.set_num_threads(os.cpu_count())


def save(name, **arrs):
    arrs = {k: (v.detach().cpu().numpy() if torch.is_tensor(v) else np.asarray(v)) for k, v in arrs.items()}
    np.savez_compressed(os.path.join(OUT, name), **arrs)
    print(name, {k: v.shape for k, v in arrs.items()})


def ref_loss_block(attn1, attn2, x1, x2, label, h, alpha):
    """train_acr.py:143-168, restated line for line (mutates attn2 in place exactly like the reference)."""
    attn1_cls = attn1[:, :, 0, 1:].unsqueeze(2)
    attn2_cls = attn2[:, :, 0, 1:].unsqueeze(2)
    attn1_aff = attn1[:, :, 1:, 1:]
    attn2_aff = attn2[:, :, 1:, 1:]
    p = h // 16
    for i in range(p):
        attn2_cls[:, :, :, i * p:i * p + p] = attn2_cls[:, :, :, i * p:i * p + p].flip(3)
    for i in range(p):
        attn2_aff[:, :, i * p:i * p + p, :] = attn2_aff[:, :, i * p:i * p + p, :].flip(2)
    for i in range(p):
        attn2_aff[:, :, :, i * p:i * p + p] = attn2_aff[:, :, :, i * p:i * p + p].flip(3)
    cls_align_loss = F.l1_loss(attn1_cls, attn2_cls, reduction='mean')
    aff_align_loss = F.l1_loss(attn1_aff, attn2_aff, reduction='mean')
    cls_loss_1 = F.multilabel_soft_margin_loss(x1, label)
    cls_loss_2 = F.multilabel_soft_margin_loss(x2, label)
    loss = cls_loss_1 + cls_loss_2 + cls_align_loss * alpha + aff_align_loss * alpha
    return loss, cls_loss_1, cls_loss_2, cls_align_loss, aff_align_loss


GRAD_KEYS = ["pretrained.model.blocks.0.attn.qkv.weight", "pretrained.model.blocks.11.attn.qkv.weight",
             "pretrained.model.blocks.5.mlp.fc1.weight", "cls_head.weight", "pretrained.model.pos_embed"]


def train_golden(name, backbone, S, B, C, alpha, depth_key=11, qkv_gain=4.0):
    model = loader.build_acr(C, backbone)
    dim = model.pretrained.model.embed_dim
    if backbone == "vitl":   # SURVEY Q6: the reference hard-codes 768 and cannot run ViT-L unpatched
        model.cls_head = torch.nn.Linear(dim, C)
    shapes = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    model.load_state_dict(orc.synth_state_dict(shapes, qkv_gain=qkv_gain))
    model.train()
    img = synth.images(B, S)
    label = synth.labels(B, C)
    img2 = img.flip(-1)
    cls_list, attn_list = model.forward_mirror(img, img2)
    attn1, attn2 = attn_list
    a1_keep, a2_keep = attn1.detach().clone(), attn2.detach().clone()
    x1, x2 = cls_list[0], cls_list[1]
    loss, l1, l2, lc, la = ref_loss_block(attn1, attn2, x1, x2, label, S, alpha)
    model.zero_grad()
    loss.backward()
    params = dict(model.named_parameters())
    keys = [k.replace(".11.", f".{depth_key}.") for k in GRAD_KEYS]
    out = dict(loss=loss, cls_loss_1=l1, cls_loss_2=l2, cls_align_loss=lc, aff_align_loss=la,
               x_cls_1=x1, x_cls_2=x2, x_patch_cls_1=cls_list[2], alpha=alpha, S=S, B=B, C=C, qkv_gain=qkv_gain)
    if attn1.numel() <= 200000:
        out.update(attn1=a1_keep, attn2=a2_keep)
    else:   # sub-sample: a few layers, rows and a column stride
        out.update(attn1_sub=a1_keep[:, ::5, ::97, ::7], attn2_sub=a2_keep[:, ::5, ::97, ::7],
                   attn1_rowsum=a1_keep.sum(-1)[:, :, ::97])
    for k in keys:
        g = params[k].grad
        out["grad_norm/" + k] = g.norm()
        out["grad_slice/" + k] = g.reshape(g.shape[0] if g.dim() > 1 else 1, -1)[:8, :16] if g.dim() <= 2 else g.reshape(-1, g.shape[-1])[:8, :16]
    save(name, **out)


def infer_golden(name, S, C, present, out_size, start_layer, func, scales=(1,), qkv_gain=4.0):
    """infer_cam.py:145-215 around the reference model (lines restated; model/getam are the reference's)."""
    model = loader.build_acr(C, "vitb")
    shapes = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    model.load_state_dict(orc.synth_state_dict(shapes, qkv_gain=qkv_gain))
    model.eval()
    img = synth.images(1, S, seed=3)
    label = synth.labels(1, C, present=present)
    W, H = out_size          # the reference's naming (rows, cols)
    b, c, h, w = img.shape
    cam_list, patch_cam_list, raw = [], [], {}
    for scale in scales:
        for hflip in [1, 2]:
            cam_matrix = torch.zeros((b, C, W, H))
            model.zero_grad()
            inp = F.interpolate(img, size=(int(h * scale), int(w * scale)), mode='bilinear', align_corners=False)
            if hflip % 2 == 1:
                inp = inp.flip(-1)
            cls_pred, _, attn, patch_cam = model.forward_cam(inp)
            if scale == 1 and hflip == 2:
                raw.update(cls_pred=cls_pred.detach().clone(), patch_cam_tokens=patch_cam.detach().clone(),
                           attn_sub=attn.detach()[:, ::11, ::97, ::7].clone(),
                           attn_rowsum=attn.detach().sum(-1)[:, :, ::97].clone())
            patch_cam = patch_cam.permute(0, 2, 1).reshape(1, C, int((h * scale) // 16), int((w * scale) // 16))
            patch_cam = F.interpolate(patch_cam, [W, H], mode='bilinear', align_corners=False)[0]
            patch_cam = patch_cam.detach().cpu().numpy() * label[0, :].cpu().clone().view(C, 1, 1).numpy()
            if hflip % 2 == 1:
                patch_cam = np.flip(patch_cam, axis=-1)
            patch_cam_list.append(patch_cam)
            patch_aff = attn[:, :, 1:, 1:]
            patch_aff = torch.sum(patch_aff, dim=1)
            cur_label = label[0, :]
            output = cls_pred[0, :]
            for class_index in range(C):
                if cur_label[class_index] > 1e-5:
                    one_hot = np.zeros((1, output.size()[-1]), dtype=np.float32)
                    one_hot[0, class_index] = 1
                    one_hot = torch.from_numpy(one_hot).requires_grad_(True)
                    one_hot = torch.sum(one_hot * output)
                    model.zero_grad()
                    one_hot.backward(retain_graph=True)
                    cam, _, _ = model.getam(0, start_layer=start_layer, func=func)
                    if scale == 1 and hflip == 2:
                        raw[f"getam_{class_index}"] = cam.detach().clone()
                    cam = torch.matmul(patch_aff, cam.unsqueeze(2))
                    if scale == 1 and hflip == 2:
                        raw[f"refined_{class_index}"] = cam.detach().clone().reshape(-1)
                    cam = cam.reshape(int((h * scale) // 16), int((w * scale) // 16))
                    cam = F.interpolate(cam.unsqueeze(0).unsqueeze(0), (W, H), mode='bilinear', align_corners=True)
                    cam_matrix[0, class_index, :, :] = cam
            cam_up_single = cam_matrix[0, :, :, :].cpu().data.numpy()
            if hflip % 2 == 1:
                cam_up_single = np.flip(cam_up_single, axis=2)
            cam_list.append(cam_up_single)
    patch_sum_cam = np.sum(patch_cam_list, axis=0)
    patch_norm_cam = (patch_sum_cam - np.min(patch_sum_cam, (1, 2), keepdims=True)) / (np.max(patch_sum_cam, (1, 2), keepdims=True) - np.min(patch_sum_cam, (1, 2), keepdims=True) + 1e-5)
    sum_cam = np.sum(cam_list, axis=0)
    norm_cam = (sum_cam - np.min(sum_cam, (1, 2), keepdims=True)) / (np.max(sum_cam, (1, 2), keepdims=True) - np.min(sum_cam, (1, 2), keepdims=True) + 1e-6)
    cam_dict = {ci: norm_cam[ci] for ci in present}
    labels = {f"label_t{int(t * 100)}": orc.pseudo_label(cam_dict, C, t) for t in (0.25, 0.4)}
    save(name, norm_cam=norm_cam[list(present)], patch_norm_cam=patch_norm_cam[list(present)], present=list(present),
         S=S, C=C, out_size=list(out_size), start_layer=start_layer, func=func, scales=list(scales), qkv_gain=qkv_gain, **labels, **raw)


def attention_golden():
    """Op-level: the reference Attention module (models/vision_transformer.py:167-214) at a small width."""
    _, _, ref_vit = loader.import_reference()
    torch.manual_seed(0)
    att = ref_vit.Attention(dim=128, num_heads=2, qkv_bias=True)
    with torch.no_grad():
        att.qkv.weight.mul_(6.0)
    x = torch.randn(2, 37, 128, requires_grad=True)
    y = att(x)
    P = att.get_attn()
    wy = torch.randn(y.shape)
    G = torch.randn(2, 37, 37) * 0.1
    loss = (y * wy).sum() + (P.mean(dim=1) * G).sum()
    loss.backward()
    save("attention_small.npz", x=x, qkv_w=att.qkv.weight, qkv_b=att.qkv.bias, proj_w=att.proj.weight, proj_b=att.proj.bias,
         y=y, P=P, wy=wy, G=G, dP=att.get_attn_gradients(), dx=x.grad, d_qkv_w=att.qkv.weight.grad)


def pamr_golden():
    _, ref_pamr, _ = loader.import_reference()
    x = synth.smooth_rgb(2, 40, 48, seed=1) / 255.0
    mask = synth.probabilities(2, 5, 10, 12, seed=1)
    out_a = ref_pamr.PAMR(3, [1, 2, 4])(x, mask)
    out_b = ref_pamr.PAMR()(x, mask)
    xn = (synth.smooth_rgb(1, 112, 96, seed=2) - 120.0) / 58.0
    mask2 = synth.probabilities(1, 21, 7, 6, seed=2)
    out_c = ref_pamr.PAMR(10, [1, 2, 4, 8, 12, 24])(xn, mask2)
    save("pamr.npz", out_a=out_a, out_b=out_b, out_c=out_c)


def pamr_448_golden():
    """configs[2]'s PAMR call at full size: 448x448, 21 classes, 10 iterations, 6 dilations -- the reference module itself
    (pamr.py:125-144); output sub-sampled ::7 in both image axes."""
    _, ref_pamr, _ = loader.import_reference()
    x = (synth.smooth_rgb(1, 448, 448, seed=4) - 120.0) / 58.0
    mask = synth.probabilities(1, 21, 28, 28, seed=4)
    out = ref_pamr.PAMR(10, [1, 2, 4, 8, 12, 24])(x, mask)
    save("pamr_448.npz", out_sub=out[:, :, ::7, ::7], out_sum=out.sum(dim=(2, 3)))


def densecrf_golden():
    """configs[3]: the dense-CRF term at COCO shape, K = 81 planes, 448x448 inputs down-scaled by rloss-scale 0.5 to 224x224
    (flags of infer_cam.py:58-65: sigma-rgb 15, sigma-xy 100, densecrfloss 1e-7).  The FILTER is the reference C++ compiled in
    place (oracle/_ref); the loss on top of it follows the upstream rloss convention (SURVEY section 9) -- the only part the
    reference repository does not contain."""
    assert bo.have_ref(), "run `make -C oracle` first"
    N, K, S, scale, srgb, sxy, weight = 2, 81, 448, 0.5, 15.0, 100.0, 1e-7
    img = synth.smooth_rgb(N, S, S, seed=11)
    seg = synth.probabilities(N, K, S, S, seed=11)
    roi = (synth.smooth_rgb(N, S, S, seed=12)[:, 0] > 100.0).float()
    img_s = F.interpolate(img, scale_factor=scale, recompute_scale_factor=True)
    seg_s = F.interpolate(seg, scale_factor=scale, mode="bilinear", align_corners=False, recompute_scale_factor=True)
    roi_s = F.interpolate(roi.unsqueeze(1), scale_factor=scale, recompute_scale_factor=True)
    sp = (seg_s * roi_s).contiguous()
    AS = torch.from_numpy(bo.ref_bilateral(img_s.numpy(), sp.numpy(), srgb, sxy * scale))
    loss = -weight * (sp * AS).sum() / N
    grad_sp = -2.0 * weight * AS * roi_s / N            # d loss / d seg_s
    save("densecrf_81.npz", cfg=np.array([N, K, S, scale, srgb, sxy, weight], dtype=np.float64), loss=loss,
         AS_sub=AS[:, ::4, ::5, ::5], AS_sum=AS.sum(dim=(2, 3)), grad_sub=grad_sp[:, ::4, ::5, ::5])


def bilateral_golden():
    assert bo.have_ref(), "run `make -C oracle` first"
    cases = {"a": (2, 4, 24, 28, 15.0, 10.0, 4), "b": (1, 3, 33, 31, 8.0, 4.0, 5), "c": (1, 21, 112, 112, 15.0, 50.0, 6)}
    out, inputs = {}, {}
    for k, (N, K, H, W, srgb, sxy, seed) in cases.items():
        img = synth.smooth_rgb(N, H, W, seed=seed).numpy()
        ins = synth.probabilities(N, K, H, W, seed=seed).numpy()
        r = bo.ref_bilateral(img, ins, srgb, sxy)
        out[f"{k}_cfg"] = np.array([N, K, H, W, srgb, sxy, seed], dtype=np.float64)
        out[f"{k}_out"] = r if r.size < 60000 else r[:, :, ::3, ::3]
        if r.size < 60000:
            # torch's CPU kernels behind synth differ in the last bit between x86 vector extensions; the bit-exact
            # comparison needs the very inputs the reference filtered
            inputs[f"{k}_img"], inputs[f"{k}_ins"] = img, ins
    save("bilateral.npz", **out)
    save("bilateral_inputs.npz", **inputs)


if __name__ == "__main__":
    assert loader.available(), "reference tree not found"
    which = sys.argv[1:] or ["attention", "pamr", "pamr448", "bilateral", "densecrf", "train64", "train64g2", "train448", "train448g2", "vitl64",
                             "infer448", "infer448g2", "infer_ms"]
    if "attention" in which: attention_golden()
    if "pamr" in which: pamr_golden()
    if "pamr448" in which: pamr_448_golden()
    if "bilateral" in which: bilateral_golden()
    if "densecrf" in which: densecrf_golden()
    if "train64" in which: train_golden("train_vitb_64.npz", "vitb", 64, 2, 20, 100.0)
    if "train64g2" in which: train_golden("train_vitb_64_g2.npz", "vitb", 64, 2, 20, 100.0, qkv_gain=2.0)
    if "train448" in which: train_golden("train_vitb_448.npz", "vitb", 448, 1, 20, 100.0)
    if "train448g2" in which: train_golden("train_vitb_448_g2.npz", "vitb", 448, 2, 20, 100.0, qkv_gain=2.0)
    if "vitl64" in which: train_golden("train_vitl_96.npz", "vitl", 96, 1, 20, 100.0, depth_key=23, qkv_gain=2.5)
    if "infer448" in which: infer_golden("infer_vitb_448.npz", 448, 20, (3, 7, 14), (60, 80), 10, "grad")
    if "infer448g2" in which: infer_golden("infer_vitb_448_g2.npz", 448, 20, (3, 7, 14), (60, 80), 10, "grad", qkv_gain=2.0)
    if "infer_ms" in which: infer_golden("infer_vitb_128_ms.npz", 128, 20, (2, 9), (40, 36), 9, "cam_grad_s", scales=(0.5, 1, 1.5))
