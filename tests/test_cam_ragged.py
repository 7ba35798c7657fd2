"""GPU tier (-m gpu): batched CAM inference for images of different original sizes.

The finish kernel (ops.cam_finish, csrc/cam_finish.cu) against the reference's finish as torch ops, and
infer_cam_batch with per-image output sizes against infer_cam_image run image by image.
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from helpers import rel_err

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def _build(dev, C, precision, qkv_gain=2.0):
    from acr_wsss_b200 import ACR
    from oracle import acr_oracle as orc
    sd = orc.synth_state_dict(orc.vit_shapes(768, 12, C), qkv_gain=qkv_gain)
    m = ACR(C, "vitb", precision=precision).to(dev)
    m.load_state_dict(sd, strict=True)
    m.eval()
    return m


def _reference_finish(cams_s, patch_s, grids, labels, present, sizes):
    """The reference's finish (infer_cam.py:153-215: F.interpolate per view, label multiply, flip, sums over views and
    scales, normalize_cam) as torch ops for each image of the batch: returns per image (GETAM planes [n_m,rows,cols],
    patch-CAM planes [n_m,rows,cols])."""
    from acr_wsss_b200.cam import normalize_cam
    M, C = labels.shape
    out = []
    for m, (rows, cols) in enumerate(sizes):
        nm = len(present[m])
        if nm == 0:
            out.append(None)
            continue
        cam_list, patch_list = [], []
        for cams, patch, (ph, pw) in zip(cams_s, patch_s, grids):
            for v in range(2):
                pc = patch[v * M + m:v * M + m + 1].permute(0, 2, 1).reshape(1, C, ph, pw)
                pc = F.interpolate(pc, [rows, cols], mode="bilinear", align_corners=False)[0] * labels[m].view(C, 1, 1)
                cm = cams[v * M + m, :, :nm].t().reshape(nm, 1, ph, pw)
                cm = F.interpolate(cm, (rows, cols), mode="bilinear", align_corners=True)[:, 0]
                if v == 0:
                    pc, cm = pc.flip(-1), cm.flip(-1)
                patch_list.append(pc[present[m]])
                cam_list.append(cm)
        out.append((normalize_cam(torch.stack(cam_list).sum(0), 1e-6), normalize_cam(torch.stack(patch_list).sum(0), 1e-5)))
    return out


def test_cam_finish_kernel_matches_torch_composition(dev):
    """Two scales (7x7, 14x14), C = 20, M = 5, output sizes from 1x7 to 500x375, 3 / 1 / 0 real copies of n = 3; the planes
    packed in reverse order with gaps (the kernel writes where the table says); two calls bitwise equal."""
    from acr_wsss_b200 import ops
    g = torch.Generator().manual_seed(0)
    M, C, n = 5, 20, 3
    grids = [(7, 7), (14, 14)]
    sizes = [(375, 500), (500, 375), (333, 500), (1, 7), (17, 1)]
    present = [[3, 7, 14], [1], [], [0, 5], [2, 11, 19]]
    labels = torch.zeros(M, C)
    for m, p in enumerate(present):
        labels[m, p] = 0.5 + 0.5 * torch.rand(len(p), generator=g)
    labels = labels.to(dev)
    cams_s = [torch.rand(2 * M, ph * pw, n, generator=g).to(dev) for ph, pw in grids]
    patch_s = [(torch.randn(2 * M, ph * pw, C, generator=g) + 0.5).relu().to(dev) for ph, pw in grids]
    planes, where, total = [], {}, 0
    for m in reversed(range(M)):
        rows, cols = sizes[m]
        for kind in (1, 0):
            for k in reversed(range(len(present[m]))):
                planes.append((total, m, present[m][k] if kind else k, kind, rows, cols))
                where[(m, kind, k)] = total
                total += rows * cols + 3
    out = ops.cam_finish(cams_s, patch_s, grids, labels, planes, total)
    again = ops.cam_finish(cams_s, patch_s, grids, labels, planes, total)
    torch.cuda.synchronize()
    ref = _reference_finish(cams_s, patch_s, grids, labels, present, sizes)
    for m, (rows, cols) in enumerate(sizes):
        for kind in (0, 1):
            for k in range(len(present[m])):
                o = where[(m, kind, k)]
                got = out[o:o + rows * cols].view(rows, cols)
                want = ref[m][kind][k]
                assert rel_err(got.cpu().numpy(), want.cpu().numpy()) <= 1e-5, (m, kind, k)
                assert torch.equal(got, again[o:o + rows * cols].view(rows, cols)), (m, kind, k)


SETS = [(3, 7, 14), (1,), (0, 5), ()]
SIZES = [(75, 100), (100, 75), (100, 67), (56, 100)]


def _batch_inputs(dev, C=20):
    from acr_wsss_b200 import synth
    imgs = torch.cat([synth.images(1, 128, seed=10 + i) for i in range(len(SETS))]).to(dev)
    labels = torch.cat([synth.labels(1, C, present=p) for p in SETS]).to(dev)
    return imgs, labels


def test_infer_cam_batch_ragged_matches_per_image(dev):
    """infer_cam_batch with one original size per image == infer_cam_image per image at that size, eager and as a CUDA graph
    (two warm-ups, capture, replay), on the precision / affinity matrix of test_infer_cam_batch_matches_per_image; an image
    without a present class gives empty dicts; >= 99.9 % pseudo-label agreement (fp32, t = 1)."""
    from acr_wsss_b200 import infer_cam_image, infer_cam_batch, pseudo_label
    imgs, labels = _batch_inputs(dev)
    for prec, tol, t_, nrm in (("fp32", 1e-4, 1, False), ("fp32", 1e-2, 2, True), ("bf16", 2e-2, 1, False)):
        m = _build(dev, 20, prec)
        kw = dict(scales=(1.0, 0.5), start_layer=10, getam_func="cam_grad_s", t=t_, normalize=nrm)
        ref = [infer_cam_image(m, imgs[i:i + 1], labels[i:i + 1], SIZES[i], **kw) for i in range(len(SETS))]
        for graph in (False, True, True, True):
            res = infer_cam_batch(m, imgs, labels, SIZES, cuda_graph=graph, **kw)
            assert len(res) == len(SETS)
            for i, p in enumerate(SETS):
                a, pa, _ = ref[i]
                assert sorted(res[i][0]) == sorted(a) == sorted(p) and sorted(res[i][1]) == sorted(pa) == sorted(p)
                for c in p:
                    assert res[i][0][c].shape == SIZES[i] and res[i][0][c].dtype == np.float32
                    assert rel_err(res[i][0][c], a[c]) < tol and rel_err(res[i][1][c], pa[c]) < tol, (prec, graph, i, c)
                if prec == "fp32" and t_ == 1 and p:
                    for thr in (0.25, 0.40):
                        agree = (pseudo_label(res[i][0], 20, thr) == pseudo_label(a, 20, thr)).mean()
                        assert agree >= 0.999, (graph, i, thr, agree)


def test_infer_cam_batch_list_of_equal_sizes_is_the_pair_form(dev):
    from acr_wsss_b200 import infer_cam_batch
    imgs, labels = _batch_inputs(dev)
    m = _build(dev, 20, "fp32")
    kw = dict(scales=(1.0, 0.5), start_layer=10, getam_func="cam_grad_s")
    pair = infer_cam_batch(m, imgs, labels, (40, 56), **kw)
    lst = infer_cam_batch(m, imgs, labels, [(40, 56)] * len(SETS), **kw)
    for (a, pa), (b, pb) in zip(pair, lst):
        assert sorted(a) == sorted(b) and sorted(pa) == sorted(pb)
        for c in a:
            assert np.array_equal(a[c], b[c]) and np.array_equal(pa[c], pb[c]), c


def test_infer_cam_batch_graph_with_a_repeated_scale(dev):
    """Two scales of one input shape replay the same CUDA graph: the first scale's maps must survive the second replay."""
    from acr_wsss_b200 import infer_cam_batch
    imgs, labels = _batch_inputs(dev)
    m = _build(dev, 20, "bf16")
    kw = dict(scales=(0.5, 1.0, 0.5), start_layer=10, getam_func="grad")
    eager = infer_cam_batch(m, imgs, labels, SIZES, **kw)
    for _ in range(4):
        res = infer_cam_batch(m, imgs, labels, SIZES, cuda_graph=True, **kw)
        for (a, pa), (b, pb) in zip(eager, res):
            for c in a:
                assert rel_err(b[c], a[c]) < 1e-5 and rel_err(pb[c], pa[c]) < 1e-5, c


def test_cam_graphs_go_with_the_model(dev):
    """The graph cache does not keep the model alive in a reference cycle: dropping the last reference frees the model and
    its CUDA graphs at once, not whenever the cyclic collector runs (which may be during another stream's graph capture)."""
    import gc
    import weakref
    from acr_wsss_b200 import infer_cam_batch
    imgs, labels = _batch_inputs(dev)
    m = _build(dev, 20, "bf16")
    for _ in range(3):
        infer_cam_batch(m, imgs, labels, SIZES, start_layer=10, getam_func="grad", cuda_graph=True)
    assert any(g.graph is not None for g in m._cam_graphs.values())
    ref = weakref.ref(m)
    gc.collect()
    gc.disable()
    try:
        del m
        assert ref() is None
    finally:
        gc.enable()
