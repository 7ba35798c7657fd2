"""The head of the dense-CRF term (csrc/crf_head.cu) against an fp64 composition of library calls on the device, value by
value:
    seg = bilinear_down_0.5( softmax([0, bilinear_up(z -> S x S)]) )         crf_head_fwd_kernel
    d_up = d seg / d up  (autograd of that composition in fp64)             crf_head_bwd_kernel
    d_patch = bilinear_up^T d_up                                             bilinear_up_bwd_kernel (gather form)

Where the kernels branch: an output row of h = S/2 pixels takes ceil(h / 128) CTAs; the four full-resolution pixels of an
output pixel share one set of patch rows (Quad.shared) when the up-sampling ratio keeps them between the same patch
centres, as at ratio 16, and read their own rows otherwise; the bilinear backward loads d_up rows 16 bytes at a time when
S % 4 == 0 and one float at a time otherwise, and takes S <= 512.

The reference up-sampling is ATen's: its float32 tap weights (the kernels compute the same source index
scale * (dst + 0.5) - 0.5 in fp32), applied in fp64 as Wt . z . Wt^T.  At a ratio like 28 -> 450 the fp64 F.interpolate
puts its taps up to ~2^-19 elsewhere, which moves the interpolated logits by up to ~3e-5 relative (seen as 2.2e-5 in seg):
that is where the float32 operation places its taps, not an error of the kernels, and test_tap_weights_follow_fp64_taps
bounds it.

Tolerances are elementwise.  Probabilities: |ours - ref| <= rtol * ref (values below 1e-30 absolutely).  Gradients are
signed sums that can cancel, so each value is held against the sum of the magnitudes of its terms, computed in fp64 by the
same composition on |g|: |ours - ref| <= rtol * mag.  The rtol values are a small multiple of the maxima measured on a
B200 (RTOL below).
"""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from acr_wsss_b200 import _lib

TINY = 1e-30
# (B, P, C, S, logits): the training shape, the kernel limit S = 512, P = S, P = 1, C = 1, S = 2 mod 4 (scalar loads) with
# one and two CTAs per row, non-integer ratios (unshared Quad), and logits up to +-60 against the constant background logit.
CASES = [
    (8, 28, 80, 448, "randn"),
    (2, 32, 20, 512, "randn"),
    (2, 16, 5, 16, "randn"),
    (3, 1, 7, 32, "randn"),
    (2, 7, 1, 112, "randn"),
    (2, 5, 4, 46, "randn"),
    (1, 28, 8, 450, "randn"),
    (2, 12, 9, 100, "randn"),
    (1, 3, 2, 10, "randn"),
    (2, 28, 80, 448, "pm60"),
    (2, 9, 6, 18, "pm60"),
    (2, 28, 20, 448, "neg60"),
    (2, 28, 20, 448, "pos60"),
]
MEASURED = {}
# rtol per quantity, for logits N(0, 2^2) ("randn") and for logits up to +-60 ("large"), about 3x the largest value over
# CASES measured on a B200 (1000 W):
#   seg      1.6e-6 / 1.3e-5   (__expf of a logit difference near 120 carries ~2^-18 relative: the large-logit tier)
#   d_up     2.3e-6 / 1.4e-5
#   d_patch  9.4e-8 / 3.3e-7   (on the kernel's own d_up: fp32 sums of <= 2 x 2 x (S/P + 1)^2 taps)
#   z_grad   8.0e-7 / 6.9e-6
RTOL = {"seg": {"randn": 5e-6, "large": 4e-5}, "d_up": {"randn": 7e-6, "large": 4e-5},
        "d_patch": {"randn": 3e-7, "large": 1e-6}, "z_grad": {"randn": 2.5e-6, "large": 2e-5}}


def _logits(B, P, C, kind, seed):
    g = torch.Generator().manual_seed(seed)
    if kind == "randn":
        return torch.randn(B, P * P, C, generator=g) * 2.0
    if kind == "pm60":
        return torch.rand(B, P * P, C, generator=g) * 120.0 - 60.0
    base = -60.0 if kind == "neg60" else 60.0
    return base + torch.randn(B, P * P, C, generator=g)


def _aten_taps(P, S, dev, dtype=torch.float32):
    """ATen's tap weights of bilinear P -> S, align_corners=False, in `dtype`: Wt[Y, i] = weight of source row i in output
    row Y (a [P, 1] -> [S, 1] up-sampling of the unit vectors: the width taps of a 1 -> 1 resize are (1, 0)), as fp64."""
    eye = torch.eye(P, device=dev, dtype=dtype).reshape(1, P, P, 1)
    return F.interpolate(eye, size=(S, 1), mode="bilinear", align_corners=False)[0, :, :, 0].t().double()


def _up(z, Wt):
    """bilinear up-sampling [B,P*P,C] -> [B,C,S,S] with tap matrix Wt [S,P], in z's precision."""
    B, PP, C = z.shape
    P = Wt.shape[1]
    return Wt @ z.permute(0, 2, 1).reshape(B, C, P, P) @ Wt.t()


def _head(up):
    prob = torch.softmax(torch.cat([torch.zeros_like(up[:, :1]), up], dim=1), dim=1)
    return F.interpolate(prob, scale_factor=0.5, mode="bilinear", align_corners=False, recompute_scale_factor=True), prob


def _reference(z, Wt, g_seg):
    """fp64: seg, d_up, z's gradient for the cotangent g_seg, and the magnitudes mag_up / mag_patch of d_up and the gradient."""
    z64 = z.double().requires_grad_(True)
    up = _up(z64, Wt)
    up.retain_grad()
    seg, prob = _head(up)
    seg.backward(g_seg.double())
    with torch.no_grad():
        gf = 0.25 * g_seg.double().abs().repeat_interleave(2, 2).repeat_interleave(2, 3)
        mag_up = (prob * (gf + (prob * gf).sum(1, keepdim=True)))[:, 1:]
    zz = torch.zeros_like(z64, requires_grad=True)
    (mag_patch,) = torch.autograd.grad(_up(zz, Wt), zz, mag_up)
    return seg.detach(), up.grad, z64.grad, mag_up, mag_patch


def _check_prob(ours, ref, rtol, what):
    ours, ref = ours.detach().double(), ref.double()
    err = (ours - ref).abs()
    big = ref > TINY
    rel = float((err[big] / ref[big]).max()) if bool(big.any()) else 0.0
    assert rel <= rtol, f"{what}: elementwise relative error {rel:.3e} > {rtol:.1e}"
    if (~big).any():
        assert float(err[~big].max()) <= TINY, what
    return rel


def _check_grad(ours, ref, mag, rtol, what):
    ours, ref, mag = ours.double(), ref.double(), mag.double()
    r = (ours - ref).abs() / (mag + TINY)
    worst = float(r.max())
    if worst > rtol:
        i = tuple(int(v) for v in (r == r.max()).nonzero()[0])
        raise AssertionError(f"{what}: error {worst:.3e} x magnitude > {rtol:.1e} at {i}: {float(ours[i])!r} vs {float(ref[i])!r} "
                             f"(magnitude {float(mag[i]):.3e})")
    return worst


def _record(name, kind, v):
    key = (name, "randn" if kind == "randn" else "large")
    MEASURED[key] = max(MEASURED.get(key, 0.0), v)
    print(f"{name} [{kind}]: {v:.3e}   running max {key}: {MEASURED[key]:.3e}")


def _c(name, *args):
    from acr_wsss_b200 import ops
    ops._call(name, 1, *args)


@pytest.mark.gpu
@pytest.mark.parametrize("B,P,C,S,kind", CASES, ids=[f"B{b}-P{p}-C{c}-S{s}-{k}" for b, p, c, s, k in CASES])
def test_head_forward_backward_and_bilinear_backward_vs_fp64(B, P, C, S, kind):
    from acr_wsss_b200 import ops
    dev = torch.device("cuda:0")
    z = _logits(B, P, C, kind, seed=B * P * C + S).to(dev)
    g_seg = torch.randn(B, C + 1, S // 2, S // 2, generator=torch.Generator().manual_seed(S)).to(dev)
    Wt = _aten_taps(P, S, dev)
    seg_ref, d_up_ref, z_grad_ref, mag_up, mag_patch = _reference(z, Wt, g_seg)
    big = "randn" if kind == "randn" else "large"
    what = f"B={B} P={P} C={C} S={S} {kind}"

    zg = z.clone().requires_grad_(True)
    seg = ops.crf_head(zg, S)
    _record("seg", kind, _check_prob(seg, seg_ref, RTOL["seg"][big], "seg " + what))

    # the head's backward alone, through the C ABI
    d_up = torch.empty(B, C, S, S, device=dev)
    _c("acr_crf_head_bwd", ops._p(z.contiguous()), ops._p(g_seg), B, P, C, S, ops._p(d_up), ops._stream())
    _record("d_up", kind, _check_grad(d_up, d_up_ref, mag_up, RTOL["d_up"][big], "d_up " + what))

    # the gather-form bilinear backward alone, on the kernel's own d_up
    d_patch = torch.empty(B, C, P, P, device=dev)
    _c("acr_bilinear_up_bwd", ops._p(d_up), B * C, P, S, ops._p(d_patch), ops._stream())
    u = d_up.double()
    xx = torch.zeros(B, P * P, C, device=dev, dtype=torch.float64, requires_grad=True)
    (ref_patch,) = torch.autograd.grad(_up(xx, Wt), xx, u)
    (mag_u,) = torch.autograd.grad(_up(xx, Wt), xx, u.abs())
    got = d_patch.flatten(2).transpose(1, 2)
    _record("d_patch", kind, _check_grad(got, ref_patch, mag_u, RTOL["d_patch"][big], "d_patch " + what))

    # autograd end to end: ops.crf_head's backward = head backward + bilinear backward
    seg.backward(g_seg)
    _record("z_grad", kind, _check_grad(zg.grad, z_grad_ref, mag_patch, RTOL["z_grad"][big], "z.grad " + what))


@pytest.mark.gpu
@pytest.mark.parametrize("P,S", [(28, 448), (32, 512), (28, 450), (12, 100), (5, 46), (3, 10), (1, 32), (16, 16)])
def test_tap_weights_follow_fp64_taps(P, S):
    """The float32 tap matrix the references use is the fp64 one up to the fp32 rounding of the source index: equal at
    power-of-two ratios, within 2^-17 (a few ulps of an index below 32) otherwise; both are row-stochastic."""
    dev = torch.device("cuda:0")
    w32, w64 = _aten_taps(P, S, dev), _aten_taps(P, S, dev, torch.float64)
    d = float((w32 - w64).abs().max())
    assert d <= 2.0 ** -17, d
    if (S // P) * P == S and (S // P) & (S // P - 1) == 0:
        assert d == 0.0
    assert float((w64.sum(1) - 1).abs().max()) < 1e-12


@pytest.mark.gpu
@pytest.mark.parametrize("P,S", [(28, 448), (32, 512), (16, 16), (1, 32), (5, 46), (12, 100), (7, 112), (3, 10), (28, 450)])
def test_bilinear_up_bwd_one_hot_is_exact(P, S):
    """A one-hot d_up at (Y, X) comes back as the outer product of the two rows' tap weights: zero outside the <= 2 x 2 patch
    support, and inside it the fp64 product of ATen's float32 tap weights to 2^-22 relative.  The probes sweep the first
    and last rows and columns, the clamped border taps (source index < 0 or >= P - 1) and the group boundaries."""
    from acr_wsss_b200 import ops
    dev = torch.device("cuda:0")
    Wt = _aten_taps(P, S, dev)
    half = S // (2 * P)
    edge = sorted({v for v in (0, 1, 2, half - 1, half, half + 1, S // 2 - 1, S // 2, S - half - 2, S - half - 1, S - half,
                               S - 3, S - 2, S - 1) if 0 <= v < S})
    rng = np.random.default_rng(P * S)
    probes = [(y, x) for y in edge for x in edge] + [tuple(int(v) for v in rng.integers(0, S, 2)) for _ in range(64)]
    d_up = torch.zeros(len(probes), S, S, device=dev)
    for i, (y, x) in enumerate(probes):
        d_up[i, y, x] = 1.0
    out = torch.full((len(probes), P, P), float("nan"), device=dev)
    _c("acr_bilinear_up_bwd", ops._p(d_up), len(probes), P, S, ops._p(out), ops._stream())
    out = out.double()
    for i, (y, x) in enumerate(probes):
        exp = torch.outer(Wt[y], Wt[x])
        nz = exp != 0
        assert int(nz.sum()) <= 4, (y, x)
        assert bool((out[i][~nz] == 0).all()), f"P={P} S={S} one-hot at {(y, x)}: nonzero outside the tap support"
        rel = float(((out[i][nz] - exp[nz]).abs() / exp[nz]).max())
        assert rel <= 2.0 ** -22, f"P={P} S={S} one-hot at {(y, x)}: {rel:.3e} from the product of ATen's tap weights"


@pytest.mark.gpu
def test_dense_crf_loss_from_patch_logits_cfg4_vs_fp64_and_oracle_filter():
    """The whole term at the COCO-shaped step (B = 8, P = 28, C = 80, S = 448, sigma_rgb 15, sigma_xy 100 at scale 0.5):
    loss and logit gradient against the fp64 head composition followed by the C oracle's filter (fp32, on the fp64
    probabilities rounded once).  loss = -w/N <s, A s>, d loss / d s = -2 w/N A s."""
    from acr_wsss_b200 import dense_crf_loss_from_patch_logits, synth
    from oracle import bilateral_oracle as bo
    dev = torch.device("cuda:0")
    B, P, C, S, w, srgb, sxy = 8, 28, 80, 448, 1e-3, 15.0, 100.0
    z = _logits(B, P, C, "randn", seed=4).to(dev)
    img = synth.smooth_rgb(B, S, S, seed=4).to(dev)
    zg = z.clone().requires_grad_(True)
    loss = dense_crf_loss_from_patch_logits(img, zg, w, srgb, sxy, 0.5)
    loss.backward()

    img_s = F.interpolate(img, scale_factor=0.5, recompute_scale_factor=True)
    Wt = _aten_taps(P, S, dev)
    z64 = z.double().requires_grad_(True)
    seg64, prob = _head(_up(z64, Wt))
    AS = torch.from_numpy(bo.oracle_bilateral(img_s.cpu().numpy(), seg64.detach().float().cpu().numpy(), srgb, sxy * 0.5))
    AS = AS.to(dev).double()
    loss_ref = -w / B * float((seg64.detach() * AS).sum())
    g_seg = -2.0 * w / B * AS
    seg64.backward(g_seg)
    rel_loss = abs(float(loss) - loss_ref) / abs(loss_ref)
    with torch.no_grad():
        gf = 0.25 * g_seg.abs().repeat_interleave(2, 2).repeat_interleave(2, 3)
        mag_up = (prob * (gf + (prob * gf).sum(1, keepdim=True)))[:, 1:]
    zz = torch.zeros_like(z64, requires_grad=True)
    (mag,) = torch.autograd.grad(_up(zz, Wt), zz, mag_up)
    print(f"cfg4 loss relative error {rel_loss:.3e}")
    assert rel_loss <= 2e-7, rel_loss              # measured on a B200: 5.9e-8
    _record("cfg4_grad", "randn", _check_grad(zg.grad, z64.grad, mag, 2e-6, "cfg4 logit gradient"))      # measured: 5.2e-7


@pytest.mark.gpu
def test_crf_head_rejects_more_patches_than_pixels():
    """P > S (a down-sampling head) is rejected by the forward, so no backward can meet a shape the bilinear backward
    does not take."""
    from acr_wsss_b200 import ops
    z = torch.randn(1, 9 * 9, 3, device="cuda:0", requires_grad=True)
    with pytest.raises(RuntimeError, match="P <= S"):
        ops.crf_head(z, 8)
    seg = ops.crf_head(z, 10)                 # P <= S still runs both ways
    seg.sum().backward()
    assert z.grad is not None and torch.isfinite(z.grad).all()


def test_crf_head_abi_rejects_p_greater_than_s_before_any_launch():
    L = _lib.lib()
    buf = ctypes.create_string_buffer(4096)
    dev = ctypes.c_void_p((ctypes.addressof(buf) + 255) & ~255)      # never dereferenced
    assert L.acr_crf_head_fwd(dev, 1, 9, 3, 8, dev, None) == -1
    assert b"P <= S" in L.acr_last_error_string()
    assert L.acr_crf_head_bwd(dev, dev, 1, 9, 3, 8, dev, None) == -1
    assert L.acr_bilinear_up_bwd(dev, 3, 9, 8, dev, None) == -1
    assert L.acr_bilinear_up_bwd(dev, 3, 28, 514, dev, None) == -1
