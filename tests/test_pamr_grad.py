"""GPU tier (-m gpu): PAMR's backward (acr_pamr_fwd_save + acr_pamr_bwd through ops._Pamr) against torch.autograd of the
oracle restatement in float64, on every path the forward takes (tests/test_pamr_paths.py's table), at the mask ratios the
bilinear adjoint has to cover, and at the production shape; plus the properties the autograd Function promises: the forward
it wraps is unchanged bit for bit, the no-grad call launches what it always did, and the backward is deterministic, batch
independent and capturable in a CUDA graph.
"""
import pytest
import torch

from helpers import rel_err, t2n

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-3
STD_DIL = [1, 2, 4, 8, 12, 24]
MODES = ["mask", "image", "both"]


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def _inputs(B, C, H, W, mh, mw, seed):
    from acr_wsss_b200 import synth
    x = (synth.smooth_rgb(B, H, W, seed=seed) - 120.0) / 58.0
    mask = synth.probabilities(B, C, mh, mw, seed=seed)
    return x, mask


def _grads(fn, x, mask, g, mode):
    """(out, d_x, d_mask) of fn(x, mask) under the cotangent g, with the inputs `mode` names requiring grad."""
    xr = x.detach().clone().requires_grad_(mode in ("image", "both"))
    mr = mask.detach().clone().requires_grad_(mode in ("mask", "both"))
    out = fn(xr, mr)
    wrt = [t for t in (xr, mr) if t.requires_grad]
    if not out.requires_grad:                                      # num_iter = 0 and only the image asks: nothing reaches it
        return out, None, None
    grads = torch.autograd.grad(out, wrt, g, allow_unused=True)
    d = dict(zip([id(t) for t in wrt], grads))
    return out, d.get(id(xr)), d.get(id(mr))


def _check_against_oracle(x, mask, num_iter, dil, mode, seed=0):
    from acr_wsss_b200 import PAMR
    from oracle import acr_oracle as orc
    g = torch.randn(x.shape[0], mask.shape[1], *x.shape[-2:], generator=torch.Generator().manual_seed(seed)).to(x.device)
    out, dx, dm = _grads(PAMR(num_iter, dil), x, mask, g, mode)
    ref, rdx, rdm = _grads(lambda a, b: orc.pamr(a, b, num_iter, dil), x.double(), mask.double(), g.double(), mode)
    assert rel_err(t2n(out), t2n(ref)) < FP32_TOL
    if mode in ("mask", "both"):
        assert dm is not None and dm.shape == mask.shape
        assert torch.isfinite(dm).all()
        assert rel_err(t2n(dm), t2n(rdm)) <= FP32_TOL
    else:
        assert dm is None
    if mode in ("image", "both") and num_iter > 0:
        assert dx is not None and dx.shape == x.shape
        assert torch.isfinite(dx).all()
        assert rel_err(t2n(dx), t2n(rdx)) <= FP32_TOL
    else:
        assert dx is None and rdx is None                          # num_iter = 0: x is not connected to the output


PATHS = [
    (2, 5, 40, 45, 10, 12, 3, [1, 2, 4]),                     # odd width, tile kernel
    (1, 21, 97, 75, 7, 6, 4, STD_DIL),                        # odd width, standard dilations
    (1, 25, 64, 64, 8, 8, 3, STD_DIL),                        # channel groups of 21 and 4: the last chunk holds one channel
    (2, 25, 33, 51, 5, 5, 2, STD_DIL),                        # the same at an odd width
    (1, 4, 48, 64, 6, 8, 3, [1, 32]),                         # dilation above the tile halo: one thread per pixel
    (1, 4, 50, 37, 6, 8, 3, [1, 32]),
    (1, 6, 56, 60, 7, 6, 2, [1, 2, 3, 4, 5, 6, 7]),           # 7 and 8 dilations: one thread per pixel
    (2, 3, 45, 53, 6, 7, 2, [1, 2, 4, 6, 8, 12, 16, 24]),
    (1, 21, 40, 45, 10, 12, 0, STD_DIL),                      # num_iter = 0: the up-sampled mask
    (1, 21, 40, 48, 10, 12, 0, STD_DIL),
    (1, 4, 40, 45, 40, 45, 2, [1, 2, 4]),                     # mask ratios: identity
    (1, 3, 448, 448, 28, 28, 2, [1, 2, 4]),                   # 28 -> 448 (x16)
    (1, 5, 97, 97, 7, 7, 3, STD_DIL),                         # 7 -> 97 (non-integer)
    (1, 3, 40, 45, 1, 12, 2, [1, 2, 4]),                      # a one-row mask
    (1, 3, 40, 45, 10, 1, 2, [1, 2, 4]),                      # a one-column mask
]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("B,C,H,W,mh,mw,num_iter,dil", PATHS)
def test_pamr_grad_matches_fp64_autograd(dev, B, C, H, W, mh, mw, num_iter, dil, mode):
    x, mask = _inputs(B, C, H, W, mh, mw, seed=H * 1000 + W + mh)
    _check_against_oracle(x.to(dev), mask.to(dev), num_iter, dil, mode, seed=B + C + num_iter)


def test_pamr_grad_production_shape(dev):
    """cfg3: one image, 21 classes, 448 x 448, 10 iterations, the standard dilations.  The fp64 oracle runs on the GPU with
    every gather autograd saves kept (about 16 GB)."""
    x, mask = _inputs(1, 21, 448, 448, 28, 28, seed=3)
    _check_against_oracle(x.to(dev), mask.to(dev), 10, STD_DIL, "both", seed=3)


@pytest.mark.parametrize("dil", [[1, 2, 4], STD_DIL, [1, 32]])
def test_pamr_grad_flat_regions(dev, dil):
    """A constant block: sigma = 0 (std backward masked) and |x_c - x_n| = 0 (sign(0) = 0) occur; gradients stay finite and
    equal to the oracle's."""
    x, mask = _inputs(1, 6, 64, 72, 8, 9, seed=11)
    x[:, :, 8:40, 10:50] = 0.25
    x[:, 1, :, :] = -1.0                                           # a whole channel constant
    _check_against_oracle(x.to(dev), mask.to(dev), 3, dil, "both", seed=5)


@pytest.mark.parametrize("dil", [[1, 2, 4], STD_DIL, [1, 32]])
def test_pamr_forward_unchanged_by_grad_mode(dev, dil):
    from acr_wsss_b200 import PAMR, ops
    x, mask = _inputs(2, 21, 64, 72, 8, 9, seed=2)
    x, mask = x.to(dev), mask.to(dev)
    pamr = PAMR(4, dil)
    with torch.no_grad():
        plain = pamr(x, mask)
    for mode in MODES:
        out = pamr(x.clone().requires_grad_(mode != "mask"), mask.clone().requires_grad_(mode != "image"))
        assert out.requires_grad
        assert torch.equal(out.detach(), plain)
    # the no-grad path (grad mode off, or no input requiring grad) makes the one acr_pamr_fwd call it always made
    for ctx in (torch.no_grad, torch.enable_grad):
        ops.PROFILE.reset(True)
        try:
            with ctx():
                pamr(x, mask)
            prof = ops.PROFILE.summary()
        finally:
            ops.PROFILE.reset(False)
        assert prof["launches"] == 3
        assert list(prof["kernels"]) == ["acr_pamr_fwd"]


def _pamr_grads(x, mask, g, dil, num_iter):
    from acr_wsss_b200 import PAMR
    xr, mr = x.clone().requires_grad_(), mask.clone().requires_grad_()
    out = PAMR(num_iter, dil)(xr, mr)
    return torch.autograd.grad(out, [xr, mr], g)


@pytest.mark.parametrize("dil", [STD_DIL, [1, 32]])
def test_pamr_grad_deterministic_and_batch_independent(dev, dil):
    x, mask = _inputs(3, 21, 96, 88, 12, 11, seed=9)
    x, mask = x.to(dev), mask.to(dev)
    g = torch.randn(3, 21, 96, 88, generator=torch.Generator().manual_seed(1)).to(dev)
    a = _pamr_grads(x, mask, g, dil, 5)
    b = _pamr_grads(x, mask, g, dil, 5)
    for u, v in zip(a, b):
        assert torch.equal(u, v)
    one = _pamr_grads(x[1:2].contiguous(), mask[1:2].contiguous(), g[1:2].contiguous(), dil, 5)
    for u, v in zip(a, one):
        assert torch.equal(u[1:2], v)


def test_pamr_grad_cuda_graph_replay_matches_eager(dev):
    from acr_wsss_b200 import ops
    x, mask = _inputs(2, 21, 80, 72, 10, 9, seed=4)
    x, mask = x.to(dev), mask.to(dev)
    g = torch.randn(2, 21, 80, 72, generator=torch.Generator().manual_seed(2)).to(dev)
    eager = _pamr_grads(x, mask, g, STD_DIL, 4)
    sx, sm, sg = x.clone(), mask.clone(), g.clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):                                     # warm-up off the capture (kernel attributes, allocator)
        _pamr_grads(sx, sm, sg, STD_DIL, 4)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with ops.cuda_graph_capture(graph, s):
        captured = _pamr_grads(sx, sm, sg, STD_DIL, 4)
    sx.copy_(x), sm.copy_(mask), sg.copy_(g)
    graph.replay()
    torch.cuda.synchronize()
    for u, v in zip(captured, eager):
        assert torch.equal(u, v)


def test_pamr_in_a_mixed_loss_moves_the_mask_logits(dev):
    """A loss with a PAMR term and another term: the PAMR term now contributes its gradient to the mask logits (it used to
    contribute zero), and the total gradient is the oracle's."""
    from acr_wsss_b200 import PAMR
    from oracle import acr_oracle as orc
    x, _ = _inputs(2, 5, 48, 56, 6, 7, seed=8)
    x = x.to(dev)
    logits0 = torch.randn(2, 5, 6, 7, generator=torch.Generator().manual_seed(3)).to(dev)
    target = torch.rand(2, 5, 48, 56, generator=torch.Generator().manual_seed(4)).to(dev)

    def grad(pamr_fn, logits):
        logits = logits.clone().requires_grad_()
        refined = pamr_fn(x.to(logits.dtype), logits.softmax(1))
        loss = ((refined - target.to(logits.dtype)) ** 2).sum() + 1e-3 * (logits ** 2).sum()
        return torch.autograd.grad(loss, logits)[0] - 2e-3 * logits.detach()     # minus the other term's gradient

    ours = grad(PAMR(3, [1, 2, 4]), logits0)
    ref = grad(lambda a, b: orc.pamr(a, b, 3, [1, 2, 4]), logits0.double())
    assert float(ref.abs().max()) > 0.1 * float((2e-3 * logits0).abs().max())
    assert rel_err(t2n(ours), t2n(ref)) <= FP32_TOL
