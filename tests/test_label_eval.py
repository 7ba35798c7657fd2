"""Pseudo-label evaluation at every background threshold (csrc/label_eval.cu, ops.cam_label_counts / label_map_counts,
cam.LabelEvaluator, scripts/evaluate_cams.py).

The oracle is the repository's numpy restatement of evaluation.py: pseudo_label then label_iou, run once per threshold.  The
int64 P / T / TP must be equal, and IoU / mIoU bitwise equal.  CPU tier: a numpy model of the one-pass histogram form (the
same finish, cam._curve_counts) equals the oracle, and three wrong variants of it (thresholds compared in float64, ties broken
by dict order, ignore pixels counted) do not.  GPU tier (marked gpu): the kernels against the oracle.
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from acr_wsss_b200 import cam, ops
from acr_wsss_b200.cam import label_iou, pseudo_label

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEFAULT = [i / 100 for i in range(100)]
ROUNDED_UP = [t for t in DEFAULT if float(np.float32(t)) > t]


# ---------------------------------------------------------------------------------------------------------------- oracle
def _pseudo(d, gt, K, t):
    """pseudo_label for one image; a dict without planes is the all-zero CAM (an explicit zero plane of class 0 is exactly
    pseudo_label's implicit one; with K = 1 there is no class, and key -1 only gives pseudo_label the size of the map)."""
    return pseudo_label(d if d else {0 if K > 1 else -1: np.zeros(gt.shape, np.float32)}, K - 1, t)


def _oracle_counts(preds, gts, K):
    """label_iou's accumulation (evaluation.py:33-67), kept as int64 counts."""
    P, T, TP = (np.zeros(K, np.int64) for _ in range(3))
    for predict, gt in zip(preds, gts):
        cal = gt < 255
        mask = (predict == gt) * cal
        for i in range(K):
            P[i] += np.sum((predict == i) * cal)
            T[i] += np.sum((gt == i) * cal)
            TP[i] += np.sum((gt == i) * mask)
    return P, T, TP


def oracle(dicts, gts, K, thresholds):
    """Per threshold: (P, T, TP) int64 [T, K] and label_iou's (iou [T, K], miou [T])."""
    P, T, TP, iou, miou = [], [], [], [], []
    for t in thresholds:
        preds = [_pseudo(d, g, K, t) for d, g in zip(dicts, gts)]
        c = _oracle_counts(preds, gts, K)
        i, m = label_iou(preds, gts, K)
        for acc, v in zip((P, T, TP, iou, miou), (*c, i, m)):
            acc.append(v)
    return np.array(P), np.array(T), np.array(TP), np.array(iou), np.array(miou)


# ------------------------------------------------------------------------------------------------ one-pass model (CPU)
def model_counts(dicts, gts, K, thresholds, thr_dtype=np.float32, dict_order_ties=False, count_ignore=False):
    """The counters acr_cam_label_counts fills, in numpy.  The keyword arguments select the wrong variants."""
    thr = np.asarray(thresholds, np.float64).astype(thr_dtype)
    Tn, Tp = len(thr), len(thr) + 1
    n = (K - 1) * Tp
    counts = np.zeros(ops.cam_label_counts_len(K, Tn), np.int64)
    for d, gt in zip(dicts, gts):
        valid = np.ones(gt.shape, bool) if count_ignore else gt != 255
        g = gt[valid].astype(np.int64)
        if K > 1:
            labels = list(range(1, K))
            if dict_order_ties:                       # present classes in dict order first, then the absent ones
                labels = [k + 1 for k in d] + [c for c in labels if c - 1 not in d]
            stack = np.stack([np.asarray(d[c - 1], np.float32) if c - 1 in d else np.zeros(gt.shape, np.float32) for c in labels])
            arg = np.argmax(stack, axis=0)
            bc = np.asarray(labels)[arg][valid]
            m = np.take_along_axis(stack, arg[None], 0)[0][valid]
            j = np.searchsorted(thr, m, side="left")   # thresholds < m; NaN sorts last: j = T
            np.add.at(counts, (bc - 1) * Tp + j, 1)
            hit = g == bc
            np.add.at(counts, n + (bc[hit] - 1) * Tp + j[hit], 1)
        else:
            j = np.zeros(g.shape, np.int64)
        np.add.at(counts, 2 * n + j[g == 0], 1)
        np.add.at(counts, 2 * n + Tp + np.minimum(np.where(g == 255, K, g), K), 1)
    return counts


def finish(counts, K, Tn):
    P, T, TP = cam._curve_counts(torch.as_tensor(counts), K, Tn)
    return P.numpy(), T.numpy(), TP.numpy()


# ------------------------------------------------------------------------------------------------------------ fixtures
def make_image(rng, h, w, K, classes, special=False, negative=False):
    """One image: CAM planes mixing smooth values with exact float32 thresholds (ties between classes and values equal to
    float32(tau), including the thresholds float32 rounds upward), dict order shuffled; ground truth with 255, with labels of
    its classes, with background and with values in [K, 255)."""
    grid = np.float32(DEFAULT + [0.5, 1.0])
    d = {}
    for c in rng.permutation(classes):
        v = np.where(rng.random((h, w)) < 0.5, rng.choice(grid, (h, w)), rng.random((h, w), dtype=np.float32))
        v = v.astype(np.float32)
        if negative:
            v = v - np.float32(0.75)
        if special:
            u = rng.random((h, w))
            v[u < 0.01] = np.nan
            v[(u >= 0.01) & (u < 0.03)] = np.inf
            v[(u >= 0.03) & (u < 0.05)] = -np.inf
        d[int(c)] = v
    choices = [0, 0, 255] + [c + 1 for c in classes] + ([K, 254] if K < 254 else [])
    gt = rng.choice(np.array(choices), (h, w)).astype(np.uint8)
    return d, gt


SIZES = [(1, 1), (1, 23), (19, 1), (7, 13), (37, 29)]


def make_set(seed, K, sizes=SIZES, special=False, negative=False):
    rng = np.random.default_rng(seed)
    dicts, gts = [], []
    counts = [0, 1, 3, K - 1]
    for k, (h, w) in enumerate(sizes):
        classes = sorted(rng.choice(K - 1, size=min(counts[k % 4], K - 1), replace=False).tolist())
        d, g = make_image(rng, h, w, K, classes, special, negative)
        dicts.append(d)
        gts.append(g)
    return dicts, gts


THRESHOLD_SETS = {
    "T1": [0.1], "T2": [0.1, 0.35], "T100": DEFAULT,
    "negative": [-1.0, -0.5, -0.25, -0.01, 0.0, 0.1, 0.29, 0.5],
}


def cap_thresholds(K):
    """The most thresholds whose histograms fit 200 KB, with equal neighbours after float32 rounding."""
    T = (200 * 1024 - 4 * K) // (4 * (2 * K - 1)) - 1
    base = np.linspace(-0.05, 1.05, T)
    base[1::7] = base[0::7][:len(base[1::7])] + 1e-12       # equal to the previous one in float32
    return np.maximum.accumulate(base).tolist()


def assert_equal_to_oracle(P, T, TP, iou, miou, dicts, gts, K, thresholds):
    oP, oT, oTP, oiou, omiou = oracle(dicts, gts, K, thresholds)
    np.testing.assert_array_equal(P, oP)
    np.testing.assert_array_equal(T, oT)
    np.testing.assert_array_equal(TP, oTP)
    if iou is not None:
        assert iou.dtype == np.float64 and iou.tobytes() == oiou.tobytes()
        assert miou.dtype == np.float64 and miou.tobytes() == omiou.tobytes()


# ------------------------------------------------------------------------------------------------------------ CPU tier
def test_fixtures_hit_the_float32_rounding():
    assert len(ROUNDED_UP) == 46 and 0.1 in ROUNDED_UP
    dicts, gts = make_set(0, 21)
    vals = np.concatenate([v.ravel() for d in dicts for v in d.values()])
    assert np.isin(np.float32(ROUNDED_UP), vals).sum() > 30


@pytest.mark.parametrize("K", [21, 81])
@pytest.mark.parametrize("case", ["T1", "T2", "T100", "negative", "special"])
def test_one_pass_model_equals_oracle(K, case):
    thr = THRESHOLD_SETS.get(case, DEFAULT)
    dicts, gts = make_set(1, K, special=case == "special", negative=case == "negative")
    P, T, TP = finish(model_counts(dicts, gts, K, thr), K, len(thr))
    assert_equal_to_oracle(P, T, TP, None, None, dicts, gts, K, thr)


def test_one_pass_model_with_one_class():
    dicts, gts = [{}, {}], [np.array([[0, 1, 255, 7]], np.uint8), np.zeros((3, 2), np.uint8)]
    P, T, TP = finish(model_counts(dicts, gts, 1, [-0.5, 0.5]), 1, 2)
    assert_equal_to_oracle(P, T, TP, None, None, dicts, gts, 1, [-0.5, 0.5])


@pytest.mark.parametrize("variant", ["float64 thresholds", "dict-order ties", "ignore counted"])
def test_negative_controls_fail_the_oracle(variant):
    K, thr = 21, DEFAULT
    dicts, gts = make_set(2, K)
    kw = {"float64 thresholds": dict(thr_dtype=np.float64), "dict-order ties": dict(dict_order_ties=True),
          "ignore counted": dict(count_ignore=True)}[variant]
    P, T, TP = finish(model_counts(dicts, gts, K, thr, **kw), K, len(thr))
    oP, oT, oTP, _, _ = oracle(dicts, gts, K, thr)
    assert not (np.array_equal(P, oP) and np.array_equal(T, oT) and np.array_equal(TP, oTP)), variant


def test_evaluate_script_fails_without_a_gpu(tmp_path):
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "evaluate_cams.py"), "--list", str(tmp_path / "x.txt"),
                        "--predict_dir", str(tmp_path), "--gt_dir", str(tmp_path), "--curve"], capture_output=True, text=True)
    assert r.returncode != 0 and "GPU" in r.stderr


# ------------------------------------------------------------------------------------------------------------ GPU tier
gpu = pytest.mark.gpu


def evaluate(dicts, gts, K, thr, chunks=1):
    ev = cam.LabelEvaluator(K, thr)
    step = -(-len(dicts) // chunks)
    for i in range(0, len(dicts), step):
        ev.add(dicts[i:i + step], gts[i:i + step])
    return ev.counts(), ev.result()


@gpu
@pytest.mark.parametrize("K", [21, 81])
@pytest.mark.parametrize("case", ["T1", "T2", "T100", "negative", "special", "cap"])
def test_curve_equals_oracle(K, case):
    thr = cap_thresholds(K) if case == "cap" else THRESHOLD_SETS.get(case, DEFAULT)
    sizes = SIZES if case == "cap" else SIZES + [(375, 500), (500, 375)]
    dicts, gts = make_set(10 + K, K, sizes, special=case == "special", negative=case == "negative")
    if case != "cap":                                  # the two VOC-size images carry 1 and 3 classes
        assert [len(d) for d in dicts[-2:]] == [1, 3]
    (P, T, TP), (iou, miou, best_t, best_m) = evaluate(dicts, gts, K, thr)
    assert_equal_to_oracle(P, T, TP, iou, miou, dicts, gts, K, thr)
    b = int(np.argmax(miou))
    assert best_t == thr[b] and best_m == miou[b] and best_m == miou.max() and (miou[:b] < best_m).all()


@gpu
def test_one_class_and_implicit_zero_planes():
    """num_cls 1 (everything is background), and images with no plane where a negative threshold lets the zero planes win."""
    gts = [np.array([[0, 1, 255, 7]], np.uint8), np.zeros((3, 2), np.uint8)]
    (P, T, TP), (iou, miou, _, _) = evaluate([{}, {}], gts, 1, [-0.5, 0.5])
    assert_equal_to_oracle(P, T, TP, iou, miou, [{}, {}], gts, 1, [-0.5, 0.5])
    dicts, gts = make_set(5, 21, [(4, 9)] * 4, negative=True)
    dicts[1] = {}
    thr = [-2.0, -0.9, -0.75, -0.5, -1e-3, 0.0, 1e-3]
    (P, T, TP), (iou, miou, _, _) = evaluate(dicts, gts, 21, thr)
    assert_equal_to_oracle(P, T, TP, iou, miou, dicts, gts, 21, thr)


@gpu
def test_streaming_and_determinism():
    K = 21
    dicts, gts = make_set(3, K, SIZES * 3 + [(500, 375)], special=True)
    one = evaluate(dicts, gts, K, DEFAULT)
    for chunks in (3, len(dicts)):
        many = evaluate(dicts, gts, K, DEFAULT, chunks)
        for a, b in zip(one[0], many[0]):
            np.testing.assert_array_equal(a, b)
        assert one[1][0].tobytes() == many[1][0].tobytes()
    again = evaluate(dicts, gts, K, DEFAULT)
    for a, b in zip(one[0], again[0]):
        np.testing.assert_array_equal(a, b)
    assert_equal_to_oracle(*one[0], one[1][0], one[1][1], dicts, gts, K, DEFAULT)


@gpu
def test_counts_beyond_32_bits():
    """Five calls over one 2^30-pixel constant image: class counts of 5 * 2^30 > 2^32, checked analytically."""
    dev = torch.device("cuda:0")
    side = 1 << 15
    N = side * side
    cams = torch.full((N,), 0.5, device=dev, dtype=torch.float32)
    gt = torch.ones(N, device=dev, dtype=torch.uint8)
    counts, maps = None, None
    for _ in range(5):
        counts = ops.cam_label_counts(cams, [(0, 0, 0)], gt, [(0, side, side)], DEFAULT, 21, counts)
        maps = ops.label_map_counts(gt, gt, [(0, side, side)], 21, maps)
    del cams
    P, T, TP = (x.cpu().numpy() for x in cam._curve_counts(counts, 21, 100))
    total = 5 * N
    assert total > 1 << 32
    below = np.arange(100) < 50                         # float32(i/100) < 0.5 for i < 50
    exp_P = np.zeros((100, 21), np.int64)
    exp_P[:, 1] = np.where(below, total, 0)
    exp_P[:, 0] = np.where(below, 0, total)
    exp_T = np.zeros((100, 21), np.int64)
    exp_T[:, 1] = total
    np.testing.assert_array_equal(P, exp_P)
    np.testing.assert_array_equal(T, exp_T)
    np.testing.assert_array_equal(TP, np.where(np.arange(21) == 1, exp_P, 0))
    m = maps.cpu().numpy()
    np.testing.assert_array_equal(m, np.stack([exp_T[0]] * 3))


@gpu
def test_label_maps_equal_oracle():
    K = 21
    rng = np.random.default_rng(4)
    preds, gts = [], []
    for h, w in SIZES + [(500, 375)]:
        preds.append(rng.choice(np.array([0, 1, 5, 20, K, 100, 255], np.uint8), (h, w)))
        gts.append(rng.choice(np.array([0, 1, 5, 20, K, 200, 255], np.uint8), (h, w)))
    ev = cam.LabelEvaluator(K, [0.5])
    ev.add_labels(preds[:3], gts[:3])
    ev.add_labels(preds[3:], gts[3:])
    P, T, TP = ev.counts()
    oP, oT, oTP = _oracle_counts(preds, gts, K)
    np.testing.assert_array_equal(P[0], oP)
    np.testing.assert_array_equal(T[0], oT)
    np.testing.assert_array_equal(TP[0], oTP)
    iou, miou, _, _ = ev.result()
    oiou, omiou = label_iou(preds, gts, K)
    assert iou[0].tobytes() == oiou.tobytes() and miou[0] == omiou


@gpu
def test_counting_cam_finish_output_on_the_device():
    """ops.cam_finish's packed output counted where it lies equals counting its host copy."""
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(6)
    M, C, n = 3, 20, 3
    present = [[2, 7, 14], [0], [5, 19]]
    sizes = [(375, 500), (1, 7), (33, 17)]
    grids = [(7, 7), (14, 14)]
    cams_s = [torch.rand(2 * M, ph * pw, n, generator=g).to(dev) for ph, pw in grids]
    patch_s = [torch.rand(2 * M, ph * pw, C, generator=g).to(dev) for ph, pw in grids]
    labels = torch.zeros(M, C)
    for m, p in enumerate(present):
        labels[m, p] = 1.0
    planes, total = cam._finish_planes(present, sizes)
    out = ops.cam_finish(cams_s, patch_s, grids, labels.to(dev), planes, total)
    rng = np.random.default_rng(6)
    gts = [rng.choice(np.array([0, 1, 3, 6, 8, 15, 20, 255], np.uint8), s) for s in sizes]
    gt_dev = torch.from_numpy(np.concatenate([x.ravel() for x in gts])).to(dev)
    offs = np.cumsum([0] + [r * c for r, c in sizes])
    eval_planes = [(o, m, present[m][ch]) for o, m, ch, kind, _, _ in planes if kind == 0]
    counts = ops.cam_label_counts(out, eval_planes, gt_dev, [(offs[m], r, c) for m, (r, c) in enumerate(sizes)], DEFAULT, 21)
    host = out.cpu().numpy()
    dicts = [{} for _ in range(M)]
    for o, m, ch, kind, r, c in planes:
        if kind == 0:
            dicts[m][present[m][ch]] = host[o:o + r * c].reshape(r, c)
    (P, T, TP), _ = evaluate(dicts, gts, 21, DEFAULT)
    for a, b in zip(cam._curve_counts(counts, 21, 100), (P, T, TP)):
        np.testing.assert_array_equal(a.cpu().numpy(), b)
    assert_equal_to_oracle(P, T, TP, None, None, dicts, gts, 21, DEFAULT)


def _write_set(tmp_path, dicts, gts, preds=None):
    from PIL import Image
    pal = sum(([i, i, i] for i in range(256)), [])
    names = [f"img_{i:03d}" for i in range(len(gts))]
    (tmp_path / "pred").mkdir()
    (tmp_path / "gt").mkdir()
    for i, nm in enumerate(names):
        cam.save_cam_dict(str(tmp_path / "pred" / f"{nm}.npy"), dicts[i])
        im = Image.fromarray(gts[i], mode="P")
        im.putpalette(pal)
        im.save(tmp_path / "gt" / f"{nm}.png")
        if preds is not None:
            Image.fromarray(preds[i], mode="L").save(tmp_path / "pred" / f"{nm}.png")
    (tmp_path / "list.txt").write_text("".join(f"{nm}\n" for nm in names))
    return names


def _run_script(tmp_path, *extra):
    cmd = [sys.executable, os.path.join(ROOT, "scripts", "evaluate_cams.py"), "--list", str(tmp_path / "list.txt"),
           "--predict_dir", str(tmp_path / "pred"), "--gt_dir", str(tmp_path / "gt"), "--json", str(tmp_path / "out.json"),
           "--batch", "3", *extra]
    r = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0, r.stderr
    return json.loads((tmp_path / "out.json").read_text()), r.stdout


@gpu
def test_evaluate_script_end_to_end(tmp_path):
    K = 21
    dicts, gts = make_set(8, K, SIZES + [(50, 40), (9, 9), (12, 30)])
    dicts = [{k: v for k, v in d.items()} for d in dicts]
    rng = np.random.default_rng(8)
    preds = [rng.choice(np.array([0, 1, 3, 20, 30], np.uint8), g.shape) for g in gts]
    _write_set(tmp_path, dicts, gts, preds)

    res, out = _run_script(tmp_path, "--curve")
    _, _, _, oiou, omiou = oracle(dicts, gts, K, DEFAULT)
    assert res["thresholds"] == DEFAULT and res["miou"] == omiou.tolist()
    b = int(np.argmax(omiou))
    assert res["best_threshold"] == DEFAULT[b] and res["iou_at_best"] == oiou[b].tolist()
    assert "best" in out

    res, _ = _run_script(tmp_path, "--t", "0.1")
    _, _, _, oiou, omiou = oracle(dicts, gts, K, [0.1])
    assert res["miou"] == omiou.tolist() and res["iou_at_best"] == oiou[0].tolist()

    res, _ = _run_script(tmp_path, "--type", "png")
    oiou, omiou = label_iou(preds, gts, K)
    assert res["miou"] == [omiou] and res["iou_at_best"] == oiou.tolist()
