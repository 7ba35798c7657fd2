"""CAM inference with affinity refinement: the inline block infer_cam.py:145-215, lifted into functions.

`infer_cam_image` reproduces the per-image loop body (scales x flips x present classes) with the hot pieces
on this repo's kernels: head-mean stack (fused attention), GETAM from row-0 quantities, A = sum_l attn[:,l,1:,1:]
and ONE [Np x Np]x[Np x C'] contraction for all present classes instead of C' matrix-vector products.
Bilinear resizes are library calls (F.interpolate), exactly the ones the reference makes.  `infer_cam_batch` runs M images
per trunk pass and finishes all of them (resizes to each image's own size, flips, sums, normalisation) in one kernel.
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


def _lowres_pass(model, both, present_idx, n_present, start_layer, getam_func, aff, t, normalize, max_replicas):
    """Device-only part of one scale of the batched path: trunk forward on both flips, blocks >= start_layer on one copy
    per present class, ONE backward, GETAM rows, affinity refinement.  Everything that depends on WHICH classes are present
    goes through the device tensor `present_idx`, so the pass is CUDA-graph capturable per (shape, n_present).
    Returns (patch_cam [2,Np,C], cams [2,Np,n_present])."""
    rows_v = [[], []]
    attn = patch_cam = None
    for c0 in range(0, n_present, max_replicas):
        n = min(max_replicas, n_present - c0)
        cls_rep, _, attn, patch_cam = model.forward_cam_batched(both, n, start_layer)
        model.backward_for_getam_batched(cls_rep, present_idx[c0:c0 + n].repeat(2))
        for v in range(2):
            for k in range(n):
                cam, _, _ = model.getam(v * n + k, start_layer=start_layer, func=getam_func)
                rows_v[v].append(cam[0])
    cams = torch.stack([torch.stack(rows_v[v], dim=1) for v in range(2)])            # [2,Np,C']
    if aff:
        cams = torch.cat([affinity_refine(attn[v:v + 1].detach(), cams[v:v + 1], t=t, normalize=normalize) for v in range(2)])
    return patch_cam.detach(), cams


def _lowres_pass_batch(model, both, idx, n, start_layer, getam_func, aff, t, normalize):
    """_lowres_pass for M images at once.  both [2M,3,h,w] (flipped views first), idx [2M*n] class of every (view, image, copy);
    n copies per image (images with fewer present classes carry dummy copies).  Returns (patch_cam [2M,Np,C], cams [2M,Np,n])."""
    cls_rep, _, attn, patch_cam = model.forward_cam_batched(both, n, start_layer)
    model.backward_for_getam_batched(cls_rep, idx)
    cams = model.getam_batch(start_layer=start_layer, func=getam_func)           # [2M*n, Np]
    cams = cams.view(both.shape[0], n, -1).transpose(1, 2).contiguous()           # [2M, Np, n]
    if aff:
        cams = affinity_refine(attn.detach(), cams, t=t, normalize=normalize)
    return patch_cam.detach(), cams


class _LowresGraph:
    """CUDA graph of _lowres_pass for one (model, input shape, number of present classes, options) key: the pass is ~270
    launches of small kernels at batch 2 and is CPU-launch bound when run eagerly (8.4 ms per image, 2.8 ms of GPU time).
    It lives in model._cam_graphs and holds the model weakly: a strong reference would make model and graphs cyclic garbage,
    and the cyclic collector could then destroy the graphs and free their memory pool in the middle of an unrelated CUDA graph
    capture, which invalidates that capture.  Without the cycle they go when the last reference to the model does."""

    def __init__(self, model, shape, n_present, args, batch=False):
        dev = next(model.parameters()).device
        self.both = torch.empty(shape, device=dev)
        self.idx = torch.zeros(shape[0] * n_present if batch else n_present, device=dev, dtype=torch.long)
        self.model, self.n, self.args = weakref.ref(model), n_present, args
        self.fn = _lowres_pass_batch if batch else _lowres_pass
        self.graph = None
        self.calls = 0
        self.stream = torch.cuda.Stream(device=dev)

    def run(self, both, present_idx):
        self.both.copy_(both)
        self.idx.copy_(present_idx)
        self.calls += 1
        cur = torch.cuda.current_stream()
        if self.graph is None and self.calls <= 2:          # warm up eagerly on the capture stream (lazy inits, cuBLAS workspaces)
            self.stream.wait_stream(cur)
            with torch.cuda.stream(self.stream):
                out = self.fn(self.model(), self.both, self.idx, self.n, *self.args)
            cur.wait_stream(self.stream)
            return out
        if self.graph is None:
            torch.cuda.synchronize()
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph, stream=self.stream):
                self.out = self.fn(self.model(), self.both, self.idx, self.n, *self.args)
        self.graph.replay()
        return self.out


def infer_cam_image(model, img, label, out_size, scales=(1,), start_layer=9, getam_func="cam_grad_s",
                    aff=True, t=1, normalize=False, truncate_backward=True, batch_classes=True, max_replicas=8,
                    cuda_graph=False):
    """One image of the infer_cam.py loop body (:145-215).

    img [1,3,h,w] (normalised), label [1,C] multi-hot, out_size = (rows, cols) of the original image (the
    reference calls these W,H at infer_cam.py:136).  Returns (cam_dict, patch_cam_dict, norm_cam [C,rows,cols])
    with {class_index: float32 [rows,cols]} dicts as saved by np.save at :227-228.
    truncate_backward: stop each per-class backward at block `start_layer` (identical GETAM; SURVEY section 8f rank 1).
    batch_classes (needs truncate_backward): both flips go through the trunk as one batch of 2, the blocks >= start_layer
    run on one copy of the token stream per present class (at most max_replicas per pass) and ONE backward delivers every
    class's attention gradients for both flips.
    cuda_graph (batched path on a GPU): replay the device-only part as a CUDA graph, cached on the model per (input shape,
    number of present classes, options); the first two calls of a key run eagerly.  In-place weight updates are picked
    up by the replays (the graph reads the parameter storage); re-allocating parameters (e.g. model.to(...)) needs
    `model._cam_graphs.clear()`.
    """
    assert img.shape[0] == 1, "the reference infers one image at a time (infer_cam.py:122)"
    C = label.shape[1]
    b, c, h, w = img.shape
    rows, cols = out_size
    lab_host = label[0].tolist()                       # one device->host read (the reference tests the labels one by one)
    present = [ci for ci in range(C) if lab_host[ci] > 1e-5]
    cam_list, patch_cam_list = [], []
    nblocks = len(model.pretrained.model.blocks)
    batched = truncate_backward and batch_classes and len(present) > 0 and 0 < start_layer < nblocks
    present_idx = torch.tensor(present, device=img.device, dtype=torch.long) if present else None

    def finish_view(attn, patch_cam, cams, flipped, ph, pw):
        """infer_cam.py:153-199 for one flip: patch CAM and (affinity-refined) GETAM maps at the original image size.
        cams [1,Np,C'] (already refined when attn is None)."""
        patch_cam = patch_cam.permute(0, 2, 1).reshape(1, C, ph, pw)
        patch_cam = F.interpolate(patch_cam, [rows, cols], mode="bilinear", align_corners=False)[0]
        patch_cam = patch_cam.detach() * label[0, :].view(C, 1, 1)
        if flipped:
            patch_cam = patch_cam.flip(-1)
        patch_cam_list.append(patch_cam)
        cam_matrix = torch.zeros(C, rows, cols, device=img.device)
        if present:
            if aff and attn is not None:
                cams = affinity_refine(attn.detach(), cams, t=t, normalize=normalize)
            cams = cams[0].t().reshape(len(present), 1, ph, pw)
            cams = F.interpolate(cams, (rows, cols), mode="bilinear", align_corners=True)[:, 0]
            cam_matrix.index_copy_(0, present_idx, cams)
        if flipped:
            cam_matrix = cam_matrix.flip(-1)
        cam_list.append(cam_matrix)

    for scale in scales:
        inp = F.interpolate(img, size=(int(h * scale), int(w * scale)), mode="bilinear", align_corners=False)
        ph, pw = int((h * scale) // 16), int((w * scale) // 16)
        if batched:
            # both flips as one batch of 2, every present class as a copy of the token stream from block start_layer on:
            # one forward and ONE backward per scale (the reference: 2 forwards and 2*C' full backwards)
            both = torch.cat([inp.flip(-1), inp], dim=0)          # hflip = 1 (flipped) first, then 2, as infer_cam.py:148-151
            args = (start_layer, getam_func, aff, t, normalize, max_replicas)
            if cuda_graph and img.is_cuda:
                cache = model.__dict__.setdefault("_cam_graphs", {})
                key = (tuple(both.shape), len(present)) + args
                if key not in cache:
                    if len(cache) >= 8:
                        cache.clear()
                    cache[key] = _LowresGraph(model, tuple(both.shape), len(present), args)
                patch_cam, cams = cache[key].run(both, present_idx)
            else:
                patch_cam, cams = _lowres_pass(model, both, present_idx, len(present), *args)
            for v in range(2):
                finish_view(None, patch_cam[v:v + 1], cams[v:v + 1], v == 0, ph, pw)
            continue
        for hflip in (1, 2):
            view = inp.flip(-1) if hflip % 2 == 1 else inp
            cls_pred, _, attn, patch_cam = model.forward_cam(view)
            output = cls_pred[0, :]
            rows0 = []
            for ci in present:
                if truncate_backward:
                    model.backward_for_getam(output[ci], start_layer)
                else:
                    # (set_to_none=False: a Trainer-attached model keeps its .grad views of the flat gradient buffer)
                    model.zero_grad(set_to_none=False)
                    output[ci].backward(retain_graph=True)      # one_hot * output, infer_cam.py:173-179
                cam, _, _ = model.getam(0, start_layer=start_layer, func=getam_func)
                rows0.append(cam[0])
            cams = torch.stack(rows0, dim=1).unsqueeze(0) if present else None        # [1,Np,C']
            finish_view(attn, patch_cam, cams, hflip % 2 == 1, ph, pw)
    patch_sum = torch.stack(patch_cam_list).sum(0)
    patch_norm = normalize_cam(patch_sum, 1e-5)
    sum_cam = torch.stack(cam_list).sum(0)
    norm_cam = normalize_cam(sum_cam, 1e-6)
    # only the present classes go to the host (what the reference keeps, infer_cam.py:217-228), through one pinned buffer
    if present:
        both = torch.stack([norm_cam.index_select(0, present_idx), patch_norm.index_select(0, present_idx)])     # [2,C',rows,cols]
        host_np = _to_host(both)
    cam_dict = {ci: host_np[0, k] for k, ci in enumerate(present)}
    patch_cam_dict = {ci: host_np[1, k] for k, ci in enumerate(present)}
    return cam_dict, patch_cam_dict, norm_cam


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
    M, C = labels.shape
    assert imgs.shape[0] == M
    if len(out_size) == 2 and all(isinstance(v, numbers.Integral) for v in out_size):
        sizes = [(int(out_size[0]), int(out_size[1]))] * M
    else:
        sizes = [(int(r), int(c)) for r, c in out_size]
        assert len(sizes) == M, "out_size: (rows, cols) or one such pair per image"
    nblocks = len(model.pretrained.model.blocks)
    assert 0 < start_layer < nblocks, "the batched path stops the backward at block start_layer"
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
            key = ("batch", tuple(both.shape), n) + args
            if key not in cache:
                if len(cache) >= 8:
                    cache.clear()
                cache[key] = _LowresGraph(model, tuple(both.shape), n, args, batch=True)
            if key in live:            # a replay overwrites the graph's outputs: keep those of the earlier scale
                j = live[key]
                patch_s[j], cams_s[j] = patch_s[j].clone(), cams_s[j].clone()
            live[key] = len(cams_s)
            patch_cam, cams = cache[key].run(both, idx)
        else:
            patch_cam, cams = _lowres_pass_batch(model, both, idx, n, *args)
        patch_s.append(patch_cam)
        cams_s.append(cams)
        grids.append((ph, pw))
    planes, total = _finish_planes(present, sizes)
    host = _to_host(ops.cam_finish(cams_s, patch_s, grids, labels, planes, total))
    maps = iter(host[o:o + r * cl].reshape(r, cl) for o, _, _, _, r, cl in planes)
    out = []
    for m in range(M):
        cam_dict = {ci: next(maps) for ci in present[m]}
        out.append((cam_dict, {ci: next(maps) for ci in present[m]}))
    return out
