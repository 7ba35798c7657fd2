"""CAM inference with affinity refinement: the inline block infer_cam.py:145-215, lifted into functions.

`infer_cam_image` reproduces the per-image loop body (scales x flips x present classes) with the hot pieces
on this repo's kernels: head-mean stack (fused attention), GETAM from row-0 quantities, A = sum_l attn[:,l,1:,1:]
and ONE [Np x Np]x[Np x C'] contraction for all present classes instead of C' matrix-vector products.
`infer_cam_batch` runs M images per trunk pass; `infer_cam_image` is the same pass with M = 1.  Both finish every image
(bilinear resizes to its own size, flips, sums over views and scales, min-max normalisation) in one kernel (ops.cam_finish).
"""
import numbers
import weakref

import numpy as np
import torch
import torch.nn.functional as F

from . import ops


def affinity_refine(attn, cam, t=1, normalize=False):
    """infer_cam.py:164-165,184.  attn [B,L,N,N]; cam [B,N-1,C] or [B,N-1] -> same shape as cam.

    t=1, normalize=False is the reference (A is the plain sum over blocks, applied once, SURVEY Q7);
    t>1 / normalize=True is the generalisation named by the north star (row-normalised affinity power).
    """
    squeeze = cam.dim() == 2
    c3 = cam.unsqueeze(-1) if squeeze else cam
    if c3.shape[-1] + int(bool(normalize)) <= 128:
        out = ops.affinity_refine_tc(attn, c3, t, normalize)        # tensor cores: block sum + contraction + normalisation fused
    else:                                                           # more classes than one UMMA tile: exact CUDA-core kernels
        out = ops.affinity_apply(ops.affinity_sum(attn, normalize), c3, t)
    return out.squeeze(-1) if squeeze else out


def normalize_cam(sum_cam, eps):
    """Per-class min-max normalisation, infer_cam.py:202,209 (eps 1e-5 patch CAM / 1e-6 GETAM).  [C,H,W]."""
    mn = sum_cam.amin(dim=(1, 2), keepdim=True)
    mx = sum_cam.amax(dim=(1, 2), keepdim=True)
    return (sum_cam - mn) / (mx - mn + eps)


def pseudo_label(cam_dict, num_classes, threshold):
    """evaluation.py:30-36: argmax over [threshold, cam_1..cam_C] -> uint8 label map."""
    h, w = next(iter(cam_dict.values())).shape
    tensor = np.zeros((num_classes + 1, h, w), np.float32)
    for key, v in cam_dict.items():
        tensor[key + 1] = v
    tensor[0, :, :] = threshold
    return np.argmax(tensor, axis=0).astype(np.uint8)


def save_cam_dict(path, cam_dict):
    """Pseudo-label writer, infer_cam.py:227-228: `np.save(path, {class_index: float32 [rows,cols]})` -- the pickled-dict
    .npy that evaluation.py:28-31 (and the downstream segmentation training) reads back with allow_pickle."""
    np.save(path, {int(k): np.ascontiguousarray(v, dtype=np.float32) for k, v in cam_dict.items()})


def crf_inference(img, probs, t=10, scale_factor=1, labels=21):
    """Drop-in for the reference's crf_inference (tool/imutils.py, pydensecrf): img HWC uint8 [H,W,3], probs [labels,H,W]
    scores -> numpy float32 [labels,H,W], the marginals after t mean-field iterations of a Gaussian (sxy 3/scale_factor,
    compat 3) and a bilateral kernel (sxy 80/scale_factor, srgb 13, compat 10), on the current CUDA device."""
    h, w = img.shape[:2]
    dev = torch.device("cuda", torch.cuda.current_device())
    image = torch.from_numpy(np.ascontiguousarray(np.asarray(img).transpose(2, 0, 1), dtype=np.float32)).to(dev)[None]
    scores = torch.from_numpy(np.ascontiguousarray(probs, dtype=np.float32).reshape(labels, h, w)).to(dev)[None]
    q = ops.dense_crf(image, scores, n_iter=t, sxy_g=3 / scale_factor, compat_g=3, sxy_b=80 / scale_factor, srgb=13, compat_b=10)
    return q[0].cpu().numpy()


def _bg_scores(cam_dict, alpha):
    """_crf_with_alpha's scores (myTool.py): [(1 - max_c cam)^alpha, cams in dict order]."""
    v = np.array(list(cam_dict.values()))
    bg = np.power(1 - np.max(v, axis=0, keepdims=True), alpha)
    return np.concatenate((bg, v), axis=0)


def crf_with_alpha(img, cam_dict, alpha, t=10):
    """The reference's _crf_with_alpha (myTool.py) for one image: img HWC uint8, cam_dict {class: [H,W]} ->
    {0: background marginal, class + 1: marginal of class} (numpy float32 [H,W])."""
    return crf_with_alpha_batch([img], [cam_dict], alpha, t)[0]


def crf_with_alpha_batch(imgs, cam_dicts, alpha, t=10):
    """crf_with_alpha for a list of images of any sizes: images with the same size and the same number of classes go
    through one ops.dense_crf call; the results are bitwise those of one call per image.  Returns one dict per image."""
    scores = [_bg_scores(d, alpha) for d in cam_dicts]
    groups = {}
    for m, (img, sc) in enumerate(zip(imgs, scores)):
        groups.setdefault((img.shape[0], img.shape[1], sc.shape[0]), []).append(m)
    dev = torch.device("cuda", torch.cuda.current_device())
    out = [None] * len(imgs)
    for (h, w, c), idx in groups.items():
        image = torch.from_numpy(np.stack([np.asarray(imgs[m]).transpose(2, 0, 1) for m in idx]).astype(np.float32)).to(dev)
        probs = torch.from_numpy(np.stack([scores[m] for m in idx]).astype(np.float32)).to(dev)
        q = ops.dense_crf(image, probs, n_iter=t).cpu().numpy()
        for j, m in enumerate(idx):
            res = {0: q[j, 0]}
            for i, key in enumerate(cam_dicts[m].keys()):
                res[key + 1] = q[j, i + 1]
            out[m] = res
    return out


def load_cam_dict(path):
    """evaluation.py:28-29."""
    return np.load(path, allow_pickle=True).item()


def label_iou(pred_labels, gt_labels, num_cls=21):
    """evaluation.py:33-67 without its 8 worker processes: per-class IoU over a list of (prediction, ground truth) uint8
    label maps (255 = ignore) and the mean.  Returns (iou [num_cls], miou)."""
    P = np.zeros(num_cls, np.float64)
    T = np.zeros(num_cls, np.float64)
    TP = np.zeros(num_cls, np.float64)
    for predict, gt in zip(pred_labels, gt_labels):
        cal = gt < 255
        mask = (predict == gt) * cal
        for i in range(num_cls):
            P[i] += np.sum((predict == i) * cal)
            T[i] += np.sum((gt == i) * cal)
            TP[i] += np.sum((gt == i) * mask)
    iou = TP / (T + P - TP + 1e-10)
    return iou, float(np.mean(iou))


def _above(h):
    """[..., t] = sum over j > t of h[..., j], for t = 0..J-2 (int64 on the device: exact)."""
    return h.flip(-1).cumsum(-1).flip(-1)[..., 1:]


def _curve_counts(counts, num_cls, num_thresholds):
    """ops.cam_label_counts' counters -> label_iou's P, T, TP at every threshold, int64 [T, num_cls] each.  A pixel with
    best class c and j thresholds below its value is labelled c at thresholds 0..j-1 and background above; so class c >= 1
    gets the pixels with j > t, and background the rest of the valid pixels."""
    K, T = num_cls, num_thresholds
    n = (K - 1) * (T + 1)
    by_class = counts[:n].view(K - 1, T + 1)
    hit = counts[n:2 * n].view(K - 1, T + 1)
    bg_gt = counts[2 * n:2 * n + T + 1]
    gt = counts[2 * n + T + 1:]
    pc, tpc = _above(by_class).t(), _above(hit).t()
    P = torch.cat([(gt.sum() - pc.sum(1)).unsqueeze(1), pc], 1)
    TP = torch.cat([(gt[0] - _above(bg_gt)).unsqueeze(1), tpc], 1)
    return P, gt[:K].expand(T, K), TP


class LabelEvaluator:
    """evaluation.py's mIoU at every background threshold of a sweep, on the current CUDA device (csrc/label_eval.cu).

    The result is exactly that of pseudo_label then label_iou run once per threshold: the counts are integers, and IoU and
    mIoU are computed with label_iou's float64 formula.  thresholds: ascending floats (default i/100 for i in 0..99), compared
    in float32 as pseudo_label compares them.  Counts accumulate over add / add_labels calls, so a dataset streams through in
    batches; add_labels' label maps count the same at every threshold."""

    def __init__(self, num_cls=21, thresholds=None):
        self.num_cls = int(num_cls)
        self.thresholds = [i / 100 for i in range(100)] if thresholds is None else [float(t) for t in thresholds]
        self.device = torch.device("cuda", torch.cuda.current_device())
        self._cam = torch.zeros(ops.cam_label_counts_len(self.num_cls, len(self.thresholds)), device=self.device, dtype=torch.int64)
        self._map = torch.zeros(3, self.num_cls, device=self.device, dtype=torch.int64)

    def add(self, cam_dicts, gt_maps):
        """cam_dicts: {class: float [rows, cols]} per image (as load_cam_dict or infer_cam_batch return them); gt_maps: uint8
        [rows, cols] per image (255 = ignore).  Images may differ in size.  One pinned buffer, one host-to-device copy."""
        gt_maps = [np.asarray(g) for g in gt_maps]
        assert len(cam_dicts) == len(gt_maps)
        npix = [g.size for g in gt_maps]
        nf = sum(len(d) * n for d, n in zip(cam_dicts, npix))
        host = torch.empty(4 * nf + sum(npix), dtype=torch.uint8, pin_memory=True)
        buf = host.numpy()
        f, g = buf[:4 * nf].view(np.float32), buf[4 * nf:]
        planes, images, fo, go = [], [], 0, 0
        for m, (d, gt) in enumerate(zip(cam_dicts, gt_maps)):
            assert gt.dtype == np.uint8 and gt.ndim == 2, "ground truth: uint8 [rows, cols]"
            n = gt.size
            g[go:go + n] = gt.reshape(-1)
            images.append((go, gt.shape[0], gt.shape[1]))
            go += n
            for key, v in d.items():
                assert np.shape(v) == gt.shape, f"image {m}: class {key} plane {np.shape(v)} vs ground truth {gt.shape}"
                f[fo:fo + n] = np.asarray(v).reshape(-1)          # float32, as pseudo_label's tensor holds it
                planes.append((fo, m, int(key)))
                fo += n
        dev = host.to(self.device, non_blocking=True)
        ops.cam_label_counts(dev[:4 * nf].view(torch.float32), planes, dev[4 * nf:], images, self.thresholds, self.num_cls, self._cam)

    def add_labels(self, pred_maps, gt_maps):
        """Label-map predictions (uint8 [rows, cols], e.g. the argmax of crf_with_alpha's marginals) with their ground truth."""
        pred_maps, gt_maps = [np.asarray(p) for p in pred_maps], [np.asarray(g) for g in gt_maps]
        assert len(pred_maps) == len(gt_maps)
        total = sum(g.size for g in gt_maps)
        host = torch.empty(2 * total, dtype=torch.uint8, pin_memory=True)
        buf = host.numpy()
        images, o = [], 0
        for p, gt in zip(pred_maps, gt_maps):
            assert p.dtype == gt.dtype == np.uint8 and gt.ndim == 2 and p.shape == gt.shape, "label maps: uint8 [rows, cols]"
            buf[o:o + gt.size] = p.reshape(-1)
            buf[total + o:total + o + gt.size] = gt.reshape(-1)
            images.append((o, gt.shape[0], gt.shape[1]))
            o += gt.size
        dev = host.to(self.device, non_blocking=True)
        ops.label_map_counts(dev[:total], dev[total:], images, self.num_cls, self._map)

    def counts(self):
        """label_iou's P, T, TP at every threshold: int64 numpy [T, num_cls] each."""
        P, T, TP = _curve_counts(self._cam, self.num_cls, len(self.thresholds))
        return tuple((x + self._map[i]).cpu().numpy() for i, x in enumerate((P, T, TP)))

    def result(self):
        """(iou [T, num_cls] float64, miou [T] float64, best_threshold, best_miou): label_iou's values at every threshold; the
        best threshold is the first one with the highest mIoU."""
        P, T, TP = (x.astype(np.float64) for x in self.counts())
        iou = TP / (T + P - TP + 1e-10)
        miou = np.array([np.mean(r) for r in iou], dtype=np.float64)
        best = int(np.argmax(miou))
        return iou, miou, self.thresholds[best], float(miou[best])


def label_iou_curve(cam_dicts, gt_maps, num_cls=21, thresholds=None):
    """evaluation.py --curve in one call: LabelEvaluator(num_cls, thresholds), add, result."""
    ev = LabelEvaluator(num_cls, thresholds)
    ev.add(cam_dicts, gt_maps)
    return ev.result()


def _lowres_pass(model, both, idx, n, start_layer, getam_func, aff, t, normalize):
    """Device-only part of one scale for M images: both [2M,3,h,w] (flipped views first) through the trunk, the blocks
    >= start_layer on n copies of every sample, ONE backward, one batched GETAM, one affinity refinement.  idx [2M*n] is the
    class of every (view, image, copy); images with fewer present classes carry dummy copies.  Which classes are present only
    reaches the pass through that device tensor, so the pass is CUDA-graph capturable per (shape, n).
    Returns (patch_cam [2M,Np,C], cams [2M,Np,n])."""
    cls_rep, _, attn, patch_cam = model.forward_cam_batched(both, n, start_layer)
    model.backward_for_getam_batched(cls_rep, idx)
    cams = model.getam_batch(start_layer=start_layer, func=getam_func)           # [2M*n, Np]
    cams = cams.view(both.shape[0], n, -1).transpose(1, 2).contiguous()           # [2M, Np, n]
    if aff:
        cams = affinity_refine(attn.detach(), cams, t=t, normalize=normalize)
    return patch_cam.detach(), cams


class _LowresGraph:
    """CUDA graph of _lowres_pass for one (model, input shape, copies per image, options) key: the pass is hundreds of
    launches of small kernels and is CPU-launch bound when run eagerly.
    It lives in model._cam_graphs and holds the model weakly: a strong reference would make model and graphs cyclic garbage,
    and the cyclic collector could then destroy the graphs and free their memory pool in the middle of an unrelated CUDA graph
    capture, which invalidates that capture.  Without the cycle they go when the last reference to the model does."""

    def __init__(self, model, shape, n, args):
        dev = next(model.parameters()).device
        self.both = torch.empty(shape, device=dev)
        self.idx = torch.zeros(shape[0] * n, device=dev, dtype=torch.long)
        self.model, self.n, self.args = weakref.ref(model), n, args
        self.graph = None
        self.calls = 0
        self.stream = torch.cuda.Stream(device=dev)

    def run(self, both, idx):
        self.both.copy_(both)
        self.idx.copy_(idx)
        self.calls += 1
        cur = torch.cuda.current_stream()
        if self.graph is None and self.calls <= 2:          # warm up eagerly on the capture stream (lazy inits, cuBLAS workspaces)
            self.stream.wait_stream(cur)
            with torch.cuda.stream(self.stream):
                out = _lowres_pass(self.model(), self.both, self.idx, self.n, *self.args)
            cur.wait_stream(self.stream)
            return out
        if self.graph is None:
            torch.cuda.synchronize()
            self.graph = torch.cuda.CUDAGraph()
            with ops.cuda_graph_capture(self.graph, self.stream):
                self.out = _lowres_pass(self.model(), self.both, self.idx, self.n, *self.args)
        self.graph.replay()
        return self.out


def infer_cam_image(model, img, label, out_size, scales=(1,), start_layer=9, getam_func="cam_grad_s", aff=True, t=1,
                    normalize=False, cuda_graph=False):
    """One image of the infer_cam.py loop body (:145-215): infer_cam_batch's pass and finish with M = 1.

    img [1,3,h,w] (normalised), label [1,C] multi-hot, out_size = (rows, cols) of the original image (the
    reference calls these W,H at infer_cam.py:136).  Returns (cam_dict, patch_cam_dict, norm_cam): {class_index: float32
    [rows,cols]} dicts as saved by np.save at :227-228 (views of one pinned host buffer), and the normalised GETAM maps on the
    device, fp32 [C,rows,cols] with zeros for the absent classes.
    cuda_graph (on a GPU): replay the device-only part as a CUDA graph, cached on the model per (input shape,
    number of present classes, options); the first two calls of a key run eagerly.  In-place weight updates are picked
    up by the replays (the graph reads the parameter storage); re-allocating parameters (e.g. model.to(...)) needs
    `model._cam_graphs.clear()`.
    """
    assert img.shape[0] == 1, "the reference infers one image at a time (infer_cam.py:122)"
    rows, cols = int(out_size[0]), int(out_size[1])
    out, _, (present,) = _infer_cams(model, img, label, [(rows, cols)], scales, start_layer, getam_func, aff, t, normalize,
                                     cuda_graph)
    k = len(present)
    norm_cam = torch.zeros(label.shape[1], rows, cols, device=img.device)
    norm_cam.index_copy_(0, torch.tensor(present, device=img.device, dtype=torch.long), out[:k * rows * cols].view(k, rows, cols))
    host = _to_host(out).reshape(2, k, rows, cols)            # GETAM planes, then patch-CAM planes
    return {ci: host[0, i] for i, ci in enumerate(present)}, {ci: host[1, i] for i, ci in enumerate(present)}, norm_cam


def _to_host(t):
    """Device tensor -> numpy array through a pinned buffer of torch's caching host allocator.  The array is a VIEW of that
    buffer and keeps it alive (no second host-side copy: np.copy of the 4.8 MB per image cost 1 ms, a third of the whole call);
    the allocator recycles the block once the caller drops the arrays."""
    if not t.is_cuda:
        return t.detach().cpu().numpy()
    host = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    host.copy_(t, non_blocking=True)
    torch.cuda.current_stream().synchronize()
    return host.numpy()


def _finish_planes(present, sizes):
    """Plane table of ops.cam_finish for a batch: per image its GETAM planes (copy k = k-th present class), then its patch-CAM
    planes, packed back to back.  Returns (rows {offset, image, channel, kind, rows, cols}, total elements)."""
    planes, total = [], 0
    for m, (rows, cols) in enumerate(sizes):
        for kind in (0, 1):
            for k, ci in enumerate(present[m]):
                planes.append((total, m, ci if kind else k, kind, rows, cols))
                total += rows * cols
    return planes, total


def _infer_cams(model, imgs, labels, sizes, scales, start_layer, getam_func, aff, t, normalize, cuda_graph):
    """infer_cam_batch on the device: sizes holds (rows, cols) per image.  Returns (ops.cam_finish's fp32 output buffer, its
    plane table from _finish_planes, the present classes of every image)."""
    M, C = labels.shape
    assert imgs.shape[0] == M
    nblocks = len(model.pretrained.model.blocks)
    assert 0 <= start_layer < nblocks, "the backward stops at the input of block start_layer"
    lab_host = labels.tolist()                                   # one device->host read
    present = [[ci for ci in range(C) if lab_host[m][ci] > 1e-5] for m in range(M)]
    n = max(1, max(len(p) for p in present))
    padded = [p + [p[0] if p else 0] * (n - len(p)) for p in present]            # dummy copies repeat a class; never finished
    idx = torch.tensor(padded, device=imgs.device, dtype=torch.long).repeat(2, 1).reshape(-1)   # sample (v, m), copy k
    b, c, h, w = imgs.shape
    cams_s, patch_s, grids, live = [], [], [], {}
    for scale in scales:
        inp = F.interpolate(imgs, size=(int(h * scale), int(w * scale)), mode="bilinear", align_corners=False)
        ph, pw = int((h * scale) // 16), int((w * scale) // 16)
        both = torch.cat([inp.flip(-1), inp], dim=0)             # hflip = 1 (flipped) first, then 2, as infer_cam.py:148-151
        args = (start_layer, getam_func, aff, t, normalize)
        if cuda_graph and imgs.is_cuda:
            cache = model.__dict__.setdefault("_cam_graphs", {})
            key = (tuple(both.shape), n) + args
            if key not in cache:
                if len(cache) >= 8:
                    cache.clear()
                cache[key] = _LowresGraph(model, tuple(both.shape), n, args)
            if key in live:            # a replay overwrites the graph's outputs: keep those of the earlier scale
                j = live[key]
                patch_s[j], cams_s[j] = patch_s[j].clone(), cams_s[j].clone()
            live[key] = len(cams_s)
            patch_cam, cams = cache[key].run(both, idx)
        else:
            patch_cam, cams = _lowres_pass(model, both, idx, n, *args)
        patch_s.append(patch_cam)
        cams_s.append(cams)
        grids.append((ph, pw))
    planes, total = _finish_planes(present, sizes)
    return ops.cam_finish(cams_s, patch_s, grids, labels, planes, total), planes, present


def infer_cam_batch(model, imgs, labels, out_size, scales=(1,), start_layer=9, getam_func="cam_grad_s", aff=True, t=1,
                    normalize=False, cuda_graph=False):
    """infer_cam_image for M images of one input shape in ONE pass per scale (the reference loops over images,
    infer_cam.py:122-215): both flips of all images go through the trunk as a batch of 2M, the blocks >= start_layer run on n
    copies per image (n = the largest number of present classes in the batch; images with fewer classes carry dummy copies),
    one backward, one batched GETAM, one batched affinity contraction.  Then ONE kernel (ops.cam_finish) resizes every
    present class's GETAM map and patch CAM to its image's original size, adds the flips and scales and min-max normalises
    them; dummy copies are never computed.
    imgs [M,3,h,w] (the reference resizes every image to crop_size x crop_size first), labels [M,C]; out_size is the
    original size (rows, cols) of every image, or a sequence of M such pairs when the originals differ.
    Returns a list of (cam_dict, patch_cam_dict) per image, the same contents as infer_cam_image; the arrays are views of
    one pinned host buffer.  An image without a present class gets two empty dicts."""
    M = labels.shape[0]
    if len(out_size) == 2 and all(isinstance(v, numbers.Integral) for v in out_size):
        sizes = [(int(out_size[0]), int(out_size[1]))] * M
    else:
        sizes = [(int(r), int(c)) for r, c in out_size]
        assert len(sizes) == M, "out_size: (rows, cols) or one such pair per image"
    out, planes, present = _infer_cams(model, imgs, labels, sizes, scales, start_layer, getam_func, aff, t, normalize,
                                       cuda_graph)
    host = _to_host(out)
    maps = iter(host[o:o + r * cl].reshape(r, cl) for o, _, _, _, r, cl in planes)
    res = []
    for m in range(M):
        cam_dict = {ci: next(maps) for ci in present[m]}
        res.append((cam_dict, {ci: next(maps) for ci in present[m]}))
    return res
