"""GPU tier: dense-CRF mean-field inference (ops.dense_crf, csrc/densecrf.cu) against the CPU oracle
(oracle/densecrf_oracle.c), its determinism, and the reference-shaped wrappers in cam.py."""
import numpy as np
import pytest
import torch

from acr_wsss_b200 import cam, ops, synth
from oracle import densecrf_oracle

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _image(kind, N, H, W, seed):
    if kind == "smooth":
        return synth.smooth_rgb(N, H, W, seed=seed)
    return (torch.randn(N, 3, H, W, generator=torch.Generator().manual_seed(seed)) * 58 + 120).clamp(0, 255)


def _scores(kind, N, C, H, W, seed):
    if kind == "prob":
        return synth.probabilities(N, C, H, W, seed=seed)
    # _crf_with_alpha: [(1 - max cam)^alpha, cams] with min-max normalised cams (unnormalised scores)
    out = []
    for n in range(N):
        cams = synth.probabilities(1, max(C - 1, 1), H, W, seed=seed + n)[0].numpy()
        cams = (cams - cams.min(axis=(1, 2), keepdims=True)) / (np.ptp(cams, axis=(1, 2), keepdims=True) + 1e-5)
        out.append(cam._bg_scores(dict(enumerate(cams)), 4.0) if C > 1 else cams)
    return torch.from_numpy(np.stack(out).astype(np.float32))


def _check(q, ref):
    q, ref = np.asarray(q, np.float64), np.asarray(ref, np.float64)
    assert np.isfinite(q).all()
    assert np.abs(q - ref).max() <= 1e-4, np.abs(q - ref).max()
    if ref.shape[0] > 1:
        top2 = np.sort(ref, axis=0)[-2:]
        sure = (top2[1] - top2[0]) > 1e-3
        assert (q.argmax(0) == ref.argmax(0))[sure].all()


BOTH, G_ONLY, B_ONLY = (3.0, 10.0), (3.0, 0.0), (0.0, 10.0)
CASES = [   # N, C, H, W, n_iter, image, scores, (compat_g, compat_b)
    (1, 2, 1, 1, 10, "smooth", "prob", BOTH),
    (1, 1, 1, 7, 10, "noise", "prob", BOTH),
    (1, 2, 7, 1, 1, "smooth", "alpha", BOTH),
    (3, 21, 13, 17, 10, "noise", "alpha", BOTH),
    (3, 21, 13, 17, 10, "smooth", "prob", G_ONLY),
    (3, 21, 13, 17, 10, "smooth", "prob", B_ONLY),
    (2, 81, 13, 17, 1, "noise", "prob", BOTH),
    (1, 81, 64, 64, 10, "noise", "prob", BOTH),
    (2, 21, 64, 64, 1, "smooth", "alpha", BOTH),
    (1, 21, 64, 64, 10, "noise", "alpha", G_ONLY),
    (1, 21, 64, 64, 10, "noise", "alpha", B_ONLY),
    (9, 2, 13, 17, 10, "smooth", "alpha", BOTH),
    (1, 21, 375, 500, 10, "smooth", "alpha", BOTH),
    (1, 21, 500, 375, 10, "smooth", "prob", BOTH),
]


@pytest.mark.parametrize("N,C,H,W,t,img_kind,sc_kind,compat", CASES)
def test_dense_crf_matches_the_oracle(N, C, H, W, t, img_kind, sc_kind, compat):
    img = _image(img_kind, N, H, W, seed=H + W)
    P = _scores(sc_kind, N, C, H, W, seed=C)
    q = ops.dense_crf(img.to(DEV), P.to(DEV), n_iter=t, compat_g=compat[0], compat_b=compat[1]).cpu().numpy()
    for n in range(N):
        ref = densecrf_oracle.dense_crf(img[n].numpy(), P[n].numpy(), t, compat_g=compat[0], compat_b=compat[1])
        _check(q[n], ref)


@pytest.mark.parametrize("N,C,H,W", [(1, 1, 1, 1), (3, 21, 13, 17), (2, 81, 64, 64), (1, 21, 375, 500)])
def test_zero_iterations_is_the_softmax_of_the_clipped_log_scores(N, C, H, W):
    img = _image("noise", N, H, W, seed=1)
    P = _scores("alpha", N, C, H, W, seed=2)
    q = ops.dense_crf(img.to(DEV), P.to(DEV), n_iter=0).cpu().numpy()
    lp = np.log(np.maximum(P.numpy().astype(np.float64), 1e-5))
    e = np.exp(lp - lp.max(1, keepdims=True))
    assert np.abs(q - e / e.sum(1, keepdims=True)).max() <= 1e-6


def test_deterministic_batch_independent_and_graph_capturable():
    img = torch.cat([_image("noise", 5, 64, 96, seed=3), _image("smooth", 4, 64, 96, seed=4)]).to(DEV)
    P = _scores("alpha", 9, 21, 64, 96, seed=5).to(DEV)
    a = ops.dense_crf(img, P)
    b = ops.dense_crf(img, P)
    assert torch.equal(a, b)
    for n in (0, 6, 8):                                      # the ninth image goes through the second internal batch
        assert torch.equal(ops.dense_crf(img[n:n + 1], P[n:n + 1]), a[n:n + 1])
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ops.dense_crf(img[:3], P[:3])                        # warm-up on the capture stream
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = ops.dense_crf(img[:3], P[:3])
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, a[:3])


def test_out_of_range_scores_make_only_that_image_nan():
    img = _image("smooth", 2, 16, 24, seed=6).to(DEV)
    P = _scores("prob", 2, 3, 16, 24, seed=6).to(DEV)
    P[0, 1, 5, 7] = float("inf")
    q = ops.dense_crf(img, P, n_iter=1)
    assert torch.isnan(q[0]).all()
    assert torch.equal(q[1:], ops.dense_crf(img[1:], P[1:], n_iter=1))


def test_crf_inference_and_crf_with_alpha_follow_the_reference_interface():
    H, W = 45, 61
    img = _image("smooth", 1, H, W, seed=7)[0].permute(1, 2, 0).round().to(torch.uint8).numpy()       # HWC uint8
    probs = _scores("prob", 1, 21, H, W, seed=7)[0].numpy()
    q = cam.crf_inference(img, probs, t=10, scale_factor=1, labels=21)
    assert q.shape == (21, H, W) and q.dtype == np.float32
    dev_img = torch.from_numpy(img.transpose(2, 0, 1).astype(np.float32))[None].to(DEV)
    assert np.array_equal(q, ops.dense_crf(dev_img, torch.from_numpy(probs)[None].to(DEV), n_iter=10)[0].cpu().numpy())
    q2 = cam.crf_inference(img, probs, t=3, scale_factor=2, labels=21)
    ref2 = densecrf_oracle.dense_crf(dev_img[0].cpu().numpy(), probs, 3, sxy_g=1.5, sxy_b=40.0)
    _check(q2, ref2)

    cams = _scores("alpha", 1, 4, H, W, seed=8)[0, 1:].numpy()
    cam_dict = {14: cams[0], 2: cams[1], 7: cams[2]}
    res = cam.crf_with_alpha(img, cam_dict, 32, t=10)
    assert list(res.keys()) == [0, 15, 3, 8]
    assert all(v.shape == (H, W) and v.dtype == np.float32 for v in res.values())
    scores = cam._bg_scores(cam_dict, 32)
    ref = cam.crf_inference(img, scores, t=10, labels=4)
    for i, k in enumerate(res):
        assert np.array_equal(res[k], ref[i])
    _check(np.stack(list(res.values())), densecrf_oracle.dense_crf(dev_img[0].cpu().numpy(), scores, 10))


def test_crf_with_alpha_batch_on_mixed_sizes_is_bitwise_per_image():
    sizes = [(37, 50), (50, 37), (37, 50), (20, 20), (37, 50)]
    imgs, dicts = [], []
    for m, (h, w) in enumerate(sizes):
        imgs.append(_image("smooth", 1, h, w, seed=m)[0].permute(1, 2, 0).round().to(torch.uint8).numpy())
        c = 3 if m != 4 else 2                                   # image 4: same size as 0 and 2, fewer classes
        cams = _scores("alpha", 1, c + 1, h, w, seed=10 + m)[0, 1:].numpy()
        dicts.append({k * 3 + 1: cams[k] for k in range(c)})
    batch = cam.crf_with_alpha_batch(imgs, dicts, 4, t=5)
    for m in range(len(sizes)):
        one = cam.crf_with_alpha(imgs[m], dicts[m], 4, t=5)
        assert list(batch[m].keys()) == list(one.keys())
        for k in one:
            assert np.array_equal(batch[m][k], one[k])
