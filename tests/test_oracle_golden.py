"""CPU tier: pins the oracle (oracle/) against vectors produced by EXECUTING the unmodified reference
(tests/golden/make_golden.py).  fp32 vs fp32 on the same CPU: tolerances are tight (1e-5 relative)."""
import numpy as np
import pytest
import torch

from oracle import acr_oracle as orc
from oracle import bilateral_oracle as bo
from acr_wsss_b200 import synth
from helpers import load_golden, rel_err, t2n

TOL = 2e-5


def test_attention_core_forward_backward_matches_reference_module():
    g = load_golden("attention_small.npz")
    x = torch.tensor(g["x"], requires_grad=True)
    qkv_w, qkv_b = torch.tensor(g["qkv_w"], requires_grad=True), torch.tensor(g["qkv_b"])
    qkv = torch.nn.functional.linear(x, qkv_w, qkv_b)
    out, P = orc.attention_core(qkv, 2, 64 ** -0.5)
    y = torch.nn.functional.linear(out, torch.tensor(g["proj_w"]), torch.tensor(g["proj_b"]))
    assert rel_err(t2n(y), g["y"]) < TOL
    assert rel_err(t2n(P), g["P"]) < TOL
    # closed-form backward with the dense affinity-gradient term
    d_out = torch.tensor(g["wy"]) @ torch.tensor(g["proj_w"])
    d_qkv, dP = orc.attention_core_backward(qkv.detach(), 2, 64 ** -0.5, d_out, torch.tensor(g["G"]))
    assert rel_err(t2n(dP), g["dP"]) < TOL
    dx = d_qkv @ qkv_w.detach()
    assert rel_err(t2n(dx), g["dx"]) < 1e-4
    d_w = d_qkv.reshape(-1, d_qkv.shape[-1]).t() @ x.detach().reshape(-1, x.shape[-1])
    assert rel_err(t2n(d_w), g["d_qkv_w"]) < 1e-4


def test_consistency_loss_forms_agree_and_match_reference():
    g = load_golden("train_vitb_64.npz")
    a1, a2 = torch.tensor(g["attn1"]), torch.tensor(g["attn2"])
    p = int(g["S"]) // 16
    c1, f1 = orc.consistency_loss_inplace(a1, a2, p)
    assert abs(float(c1) - float(g["cls_align_loss"])) <= TOL * float(g["cls_align_loss"])
    assert abs(float(f1) - float(g["aff_align_loss"])) <= TOL * float(g["aff_align_loss"])
    c2, f2, g1, g2 = orc.consistency_loss_closed_form(a1, a2, p, 100.0, 100.0)
    assert abs(float(c2) - float(c1)) <= TOL * float(c1) and abs(float(f2) - float(f1)) <= TOL * float(f1)
    # analytic gradient == autograd through the literal in-place-flip code
    a1g, a2g = a1.clone().requires_grad_(True), a2.clone().requires_grad_(True)
    c, f = orc.consistency_loss_inplace(a1g, a2g, p)
    (100.0 * (c + f)).backward()
    assert torch.allclose(g1, a1g.grad, atol=1e-9) and torch.allclose(g2, a2g.grad, atol=1e-9)


@pytest.mark.parametrize("name,heads", [("train_vitb_64.npz", 12), ("train_vitb_64_g2.npz", 12), ("train_vitl_96.npz", 16)])
def test_train_step_matches_reference(name, heads):
    g = load_golden(name)
    S, B, C = int(g["S"]), int(g["B"]), int(g["C"])
    dim, depth = (768, 12) if heads == 12 else (1024, 24)
    scratch = (96, 192, 384, 768) if heads == 12 else (256, 512, 1024, 1024)
    sd = orc.synth_state_dict(orc.vit_shapes(dim, depth, C, scratch_in=scratch), qkv_gain=float(g["qkv_gain"]))
    sd = {k: v.requires_grad_(True) for k, v in sd.items()}
    img, label = synth.images(B, S), synth.labels(B, C)
    loss, parts, (attn1, attn2, x1, x2) = orc.train_step_loss(sd, img, label, float(g["alpha"]), heads)
    assert rel_err(t2n(x1), g["x_cls_1"]) < 1e-4 and rel_err(t2n(x2), g["x_cls_2"]) < 1e-4
    if "attn1" in g:
        assert rel_err(t2n(attn1), g["attn1"]) < 1e-4
    for got, key in zip((loss,) + tuple(parts), ("loss", "cls_loss_1", "cls_loss_2", "cls_align_loss", "aff_align_loss")):
        assert abs(float(got) - float(g[key])) <= 1e-4 * abs(float(g[key])), key
    loss.backward()
    for k in [k[len("grad_norm/"):] for k in g if k.startswith("grad_norm/")]:
        gr = sd[k].grad
        assert abs(float(gr.norm()) - float(g["grad_norm/" + k])) <= 2e-3 * float(g["grad_norm/" + k]), k
        sl = gr.reshape(gr.shape[0] if gr.dim() > 1 else 1, -1)[:8, :16] if gr.dim() <= 2 else gr.reshape(-1, gr.shape[-1])[:8, :16]
        assert rel_err(t2n(sl), g["grad_slice/" + k]) < 5e-3, k


def test_infer_cam_multiscale_matches_reference():
    g = load_golden("infer_vitb_128_ms.npz")
    C, S = int(g["C"]), int(g["S"])
    sd = orc.synth_state_dict(orc.vit_shapes(768, 12, C))
    img = synth.images(1, S, seed=3)
    present = [int(c) for c in g["present"]]
    label = synth.labels(1, C, present=present)
    cam_dict, patch_dict, norm_cam = orc.infer_cam_image(sd, img, label, tuple(int(v) for v in g["out_size"]),
                                                         scales=tuple(float(s) for s in g["scales"]),
                                                         start_layer=int(g["start_layer"]), getam_func=str(g["func"]))
    assert rel_err(norm_cam[present], g["norm_cam"]) < 1e-3
    assert rel_err(np.stack([patch_dict[c] for c in present]), g["patch_norm_cam"]) < 1e-3
    for t in (25, 40):
        lab = orc.pseudo_label(cam_dict, C, t / 100.0)
        assert (lab == g[f"label_t{t}"]).mean() >= 0.999


def test_pamr_gather_restatement_matches_reference():
    g = load_golden("pamr.npz")
    x = synth.smooth_rgb(2, 40, 48, seed=1) / 255.0
    mask = synth.probabilities(2, 5, 10, 12, seed=1)
    assert rel_err(t2n(orc.pamr(x, mask, 3, [1, 2, 4])), g["out_a"]) < TOL
    assert rel_err(t2n(orc.pamr(x, mask, 1, [1])), g["out_b"]) < TOL
    xn = (synth.smooth_rgb(1, 112, 96, seed=2) - 120.0) / 58.0
    mask2 = synth.probabilities(1, 21, 7, 6, seed=2)
    assert rel_err(t2n(orc.pamr(xn, mask2, 10, [1, 2, 4, 8, 12, 24])), g["out_c"]) < TOL


def test_bilateral_c_oracle_is_bit_exact_with_reference_outputs():
    g = load_golden("bilateral.npz")
    # a, b: the inputs the reference filtered, as stored (synth's torch CPU kernels differ in the last bit between x86 vector
    # extensions); c's are too large to store and are regenerated, identically under AVX2 and AVX-512
    stored = load_golden("bilateral_inputs.npz")
    for k in "abc":
        N, K, H, W, srgb, sxy, seed = g[f"{k}_cfg"]
        N, K, H, W, seed = int(N), int(K), int(H), int(W), int(seed)
        if f"{k}_img" in stored:
            img, ins = stored[f"{k}_img"], stored[f"{k}_ins"]
        else:
            img = synth.smooth_rgb(N, H, W, seed=seed).numpy()
            ins = synth.probabilities(N, K, H, W, seed=seed).numpy()
        o = bo.oracle_bilateral(img, ins, srgb, sxy)
        if o.size >= 60000:
            o = o[:, :, ::3, ::3]
        assert np.array_equal(o, g[f"{k}_out"]), k


def test_bilateral_c_oracle_vs_compiled_reference_when_present():
    if not bo.have_ref():
        pytest.skip("oracle/_ref not built (needs the reference's bilateral-filter C++ sources, see oracle/Makefile)")
    for (N, K, H, W, srgb, sxy) in [(1, 2, 17, 23, 5.0, 3.0), (2, 3, 40, 40, 15.0, 50.0)]:
        img = synth.smooth_rgb(N, H, W, seed=9).numpy()
        ins = synth.probabilities(N, K, H, W, seed=9).numpy()
        assert np.array_equal(bo.oracle_bilateral(img, ins, srgb, sxy), bo.ref_bilateral(img, ins, srgb, sxy))


def test_bilateral_c_oracle_is_linear():
    # linearity (size-independent property): filter(a*x + y) == a*filter(x) + filter(y) up to rounding
    img = synth.smooth_rgb(1, 30, 30, seed=1).numpy()
    x = synth.probabilities(1, 2, 30, 30, seed=1).numpy()
    y = synth.probabilities(1, 2, 30, 30, seed=2).numpy()
    lhs = bo.oracle_bilateral(img, 2 * x + y, 15.0, 10.0)
    rhs = 2 * bo.oracle_bilateral(img, x, 15.0, 10.0) + bo.oracle_bilateral(img, y, 15.0, 10.0)
    assert rel_err(lhs, rhs) < 1e-5


def test_densecrf_k81_oracle_matches_reference_filter_and_closed_form():
    """configs[3] shape (K = 81 planes, 224x224 after rloss-scale 0.5): the C oracle is bit-exact with the compiled reference filter
    on the golden's sub-sample, and the loss / gradient restatement reproduces the golden's numbers."""
    import torch.nn.functional as F
    g = load_golden("densecrf_81.npz")
    N, K, S, scale, srgb, sxy, weight = g["cfg"]
    N, K, S = int(N), int(K), int(S)
    img = synth.smooth_rgb(N, S, S, seed=11)
    seg = synth.probabilities(N, K, S, S, seed=11)
    roi = (synth.smooth_rgb(N, S, S, seed=12)[:, 0] > 100.0).float()
    img_s = F.interpolate(img, scale_factor=float(scale), recompute_scale_factor=True)
    seg_s = F.interpolate(seg, scale_factor=float(scale), mode="bilinear", align_corners=False, recompute_scale_factor=True)
    roi_s = F.interpolate(roi.unsqueeze(1), scale_factor=float(scale), recompute_scale_factor=True)
    sp = (seg_s * roi_s).contiguous()
    # 21 of the 81 planes (every 4th, the golden's sub-sample): the planes are filtered independently
    AS = bo.oracle_bilateral(img_s.numpy(), sp[:, ::4].contiguous().numpy(), float(srgb), float(sxy) * float(scale))
    assert np.array_equal(AS[:, :, ::5, ::5], g["AS_sub"])
    loss, grad = orc.dense_crf_loss_from_filter(seg_s[:, ::4], roi_s, torch.from_numpy(AS), float(weight))
    assert rel_err(t2n(grad[:, :, ::5, ::5]), g["grad_sub"]) < 1e-6


def test_pamr_448_oracle_matches_reference():
    g = load_golden("pamr_448.npz")
    x = (synth.smooth_rgb(1, 448, 448, seed=4) - 120.0) / 58.0
    mask = synth.probabilities(1, 21, 28, 28, seed=4)
    out = orc.pamr(x, mask, 10, [1, 2, 4, 8, 12, 24])
    assert rel_err(t2n(out[:, :, ::7, ::7]), g["out_sub"]) < TOL
    assert rel_err(t2n(out.sum(dim=(2, 3))), g["out_sum"]) < 1e-4
