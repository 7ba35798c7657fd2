"""GPU tier (-m gpu): every path through acr_pamr_fwd against the CPU oracle.

PAMR picks its iteration kernel from the input: the TMA-fed tile kernel for at most 6 dilations of at most 24 pixels, at any
width, and a one-thread-per-pixel kernel for everything else.  The shapes below take each side of that choice, odd widths,
a channel count whose last group ends in a one-channel chunk, zero iterations, and an output pointer that is only 4-byte
aligned.
"""
import ctypes

import pytest
import torch

from helpers import rel_err, t2n

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-3
STD_DIL = [1, 2, 4, 8, 12, 24]


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def _inputs(B, C, H, W, mh, mw, seed):
    from acr_wsss_b200 import synth
    x = (synth.smooth_rgb(B, H, W, seed=seed) - 120.0) / 58.0
    mask = synth.probabilities(B, C, mh, mw, seed=seed)
    return x, mask


@pytest.mark.parametrize("B,C,H,W,mh,mw,num_iter,dil", [
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
])
def test_pamr_paths_match_oracle(dev, B, C, H, W, mh, mw, num_iter, dil):
    from acr_wsss_b200 import PAMR
    from oracle import acr_oracle as orc
    x, mask = _inputs(B, C, H, W, mh, mw, seed=H * 1000 + W)
    out = PAMR(num_iter, dil)(x.to(dev), mask.to(dev))
    ref = orc.pamr(x, mask, num_iter, dil)
    assert out.shape == (B, C, H, W)
    assert rel_err(t2n(out), t2n(ref)) < FP32_TOL


def _pamr_fwd_into(x, mask, dil, num_iter, out):
    """acr_pamr_fwd straight through the C ABI, writing into `out` (any float32 device tensor of B*C*H*W elements)."""
    from acr_wsss_b200 import _lib
    B, K, H, W = x.shape
    _, C, mh, mw = mask.shape
    L = _lib.lib()
    wsb = L.acr_pamr_workspace(B, K, C, H, W, len(dil))
    ws = torch.empty(wsb, device=x.device, dtype=torch.uint8)
    rc = L.acr_pamr_fwd(ctypes.c_void_p(x.data_ptr()), ctypes.c_void_p(mask.data_ptr()), B, K, C, H, W, mh, mw,
                        (ctypes.c_int * len(dil))(*dil), len(dil), num_iter, ctypes.c_void_p(out.data_ptr()),
                        ctypes.c_void_p(ws.data_ptr()), wsb, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    _lib.check(rc, "acr_pamr_fwd")


def test_pamr_unaligned_out_matches_aligned(dev):
    """A C-ABI caller may hand in an output that is only 4-byte aligned; the result must not depend on it."""
    B, C, H, W = 1, 21, 64, 64
    x, mask = _inputs(B, C, H, W, 8, 8, seed=7)
    x, mask = x.to(dev).contiguous(), mask.to(dev).contiguous()
    n = B * C * H * W
    aligned = torch.empty(n, device=dev)
    buf = torch.full((n + 4,), float("nan"), device=dev)
    shifted = buf[1:1 + n]
    assert shifted.data_ptr() % 16 == 4
    _pamr_fwd_into(x, mask, STD_DIL, 3, aligned)
    _pamr_fwd_into(x, mask, STD_DIL, 3, shifted)
    torch.cuda.synchronize()
    assert torch.equal(shifted.cpu(), aligned.cpu())
