"""CPU tier: self-checks of the dense-CRF oracle (oracle/densecrf_oracle.c)."""
import numpy as np
import pytest
import torch

from acr_wsss_b200 import synth
from oracle import bilateral_oracle, densecrf_oracle


def _noise(H, W, seed):
    return (torch.randn(3, H, W, generator=torch.Generator().manual_seed(seed)) * 58 + 120).clamp(0, 255).numpy()


@pytest.mark.parametrize("H,W", [(16, 20), (40, 36), (64, 64)])
@pytest.mark.parametrize("kind", ["smooth", "noise"])
@pytest.mark.parametrize("srgb,sxy", [(13.0, 80.0), (5.0, 3.0)])
def test_d5_filter_is_bit_exact_with_the_pinned_bilateral_oracle(H, W, kind, srgb, sxy):
    """At H*W % 4 == 0 the SSE reference has no phantom pads, so densecrf 2.x's lattice is the same filter."""
    img = synth.smooth_rgb(1, H, W, seed=1)[0].numpy() if kind == "smooth" else _noise(H, W, 3)
    ins = synth.probabilities(1, 3, H, W, seed=2)[0].numpy()
    ours = densecrf_oracle.bilateral(img, ins, srgb, sxy)
    pinned = bilateral_oracle.oracle_bilateral(img[None], ins[None], srgb, sxy)[0]
    assert np.array_equal(ours, pinned)


def test_zero_compat_returns_the_initial_q_at_every_iteration():
    img = synth.smooth_rgb(1, 23, 31, seed=5)[0].numpy()
    P = synth.probabilities(1, 5, 23, 31, seed=5)[0].numpy()
    q0 = densecrf_oracle.dense_crf(img, P, 0)
    for t in (1, 4):
        assert np.array_equal(densecrf_oracle.dense_crf(img, P, t, compat_g=0.0, compat_b=0.0), q0)
    lp = np.log(np.maximum(P, 1e-5))
    ref = np.exp(lp - lp.max(0)) / np.exp(lp - lp.max(0)).sum(0)
    assert np.abs(q0 - ref).max() <= 1e-6


@pytest.mark.parametrize("C", [1, 2, 21])
def test_q_sums_to_one(C):
    img = _noise(19, 13, 7)
    P = synth.probabilities(1, C, 19, 13, seed=7)[0].numpy() * 0.7           # unnormalised scores
    q = densecrf_oracle.dense_crf(img, P, 5)
    assert np.isfinite(q).all() and np.abs(q.sum(0) - 1).max() <= 1e-6
