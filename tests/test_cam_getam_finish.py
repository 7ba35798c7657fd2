"""GPU tier (-m gpu): the GETAM row-0 kernel (csrc/cam.cu: acr_getam_row0, acr_getam_row0_batch) and the batched CAM finish
(csrc/cam_finish.cu: acr_cam_finish) against fp64 numpy oracles written from the reference, at the token counts, block and
head counts, sample counts, grid sets, output sizes and shared-memory sizes CAM inference meets, plus exact probes.

GETAM oracle (DPT/ACR.py:177-215, row 0 of each block): pos = mean_h max(g, 0), gp = mean_h max(g p, 0); the block value is
pos, pos^2, gp or gp pos for func 0..3; the blocks l >= start_layer are summed, relu'd, and the first `skip` tokens dropped.
max(., 0) propagates NaN, as clamp(min=0) and relu do.

Finish oracle (infer_cam.py:153-215): ATen's upsample_bilinear2d for an explicit output size, per axis
  align_corners=True:  scale = (in-1)/(out-1) (0 when out = 1), src = scale dst
  align_corners=False: scale = in/out, src = max(scale (dst+0.5) - 0.5, 0)
  i0 = floor(src), i1 = min(i0+1, in-1), l1 = src - i0;
GETAM planes with align_corners=True and eps 1e-6, patch-CAM planes times the label with align_corners=False and eps 1e-5,
view 0 flipped horizontally, summed over scales and views, then (x - min) / (max - min + eps) with a NaN-propagating min/max
(cam.normalize_cam uses amin/amax).  Everything is fp64.  The kernel, like ATen on fp32 tensors, places its taps in fp32;
bilinear interpolation is continuous in the source position, so that moves the normalised planes of these cases by at
most 1.6e-6 (at the 160-wide grid), well inside the 2e-5 tolerance.
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from helpers import rel_err

pytestmark = pytest.mark.gpu

FUNCS = ["grad", "grad_s", "cam_grad", "cam_grad_s"]
SENTINEL = 0x7FD1A5A5             # a quiet NaN with a payload no computation produces
TESTS = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def _bits(t):
    return t.contiguous().view(torch.int32)


# ------------------------------------------------------------------ GETAM oracle and inputs
def getam_blocks(p, g):
    """p, g [L,S,H,N] -> fp64 (pos, gp) [L,S,N]: the head means of max(g, 0) and max(g p, 0)."""
    p = np.asarray(p, np.float64)
    g = np.asarray(g, np.float64)
    return np.maximum(g, 0.0).mean(2), np.maximum(g * p, 0.0).mean(2)


def getam_oracle(pos, gp, start_layer, func, skip):
    """-> (cam [S,N-skip], per-block rows [L,S,N]) in fp64."""
    rows = {"grad": pos, "grad_s": pos * pos, "cam_grad": gp, "cam_grad_s": gp * pos}[func]
    return np.maximum(rows[start_layer:].sum(0), 0.0)[:, skip:], rows


# (S samples, L blocks, H heads, N tokens).  N: 2 (one token left), 26, 197 (224 px), 785 (448 px: one CTA of 256 tokens
# and a tail of 17), 1025 (ViT-L 512 px), 3137 (scale 2.0 at 448 px).  S = 2 M n: 320 is M = 8 images of 20 classes.
GETAM_CASES = [
    (1, 1, 1, 2),
    (1, 4, 3, 26),
    (6, 12, 12, 197),
    (48, 12, 12, 785),
    (320, 2, 12, 785),
    (320, 1, 1, 1025),
    (16, 24, 16, 1025),
    (6, 12, 12, 3137),
    (48, 2, 16, 3137),
    (1, 24, 16, 3137),
]


def _getam_id(c):
    return "S{}_L{}_H{}_N{}".format(*c)


def _getam_inputs(S, L, H, N, dev):
    """p: softmax rows; g: mixed signs, about one element in eight exactly zero.  Both fp32 on `dev`."""
    gen = torch.Generator(device="cuda").manual_seed(S * 7919 + L * 131 + H * 17 + N)
    p = torch.softmax(2.0 * torch.randn(L, S, H, N, generator=gen, device=dev), -1)
    g = torch.randn(L, S, H, N, generator=gen, device=dev) * 1e-2
    g = torch.where(torch.rand(L, S, H, N, generator=gen, device=dev) < 0.125, torch.zeros_like(g), g)
    assert p.numel() * 4 <= 256 << 20
    return p, g


def _starts(L):
    return sorted({0, L // 2, L - 1})


def _skips(N):
    return [1, 2] if N > 2 else [1]


@pytest.mark.parametrize("case", GETAM_CASES, ids=[_getam_id(c) for c in GETAM_CASES])
def test_getam_batch_matches_fp64(dev, case):
    """acr_getam_row0_batch for every func, start_layer in {0, L/2, L-1} and skip in {1, 2}."""
    from acr_wsss_b200 import ops
    S, L, H, N = case
    p, g = _getam_inputs(S, L, H, N, dev)
    pos, gp = getam_blocks(p.cpu().numpy(), g.cpu().numpy())
    for func in FUNCS:
        for start in _starts(L):
            for skip in _skips(N):
                ref, _ = getam_oracle(pos, gp, start, func, skip)
                got = ops.getam_row0_batch(p, g, start, func, skip)
                assert got.shape == (S, N - skip)
                assert rel_err(got.cpu().numpy(), ref) <= 1e-5, (func, start, skip)


@pytest.mark.parametrize("case", GETAM_CASES, ids=[_getam_id(c) for c in GETAM_CASES])
def test_getam_single_entry_rows_and_batch_rows(dev, case):
    """acr_getam_row0 on one sample: its per-block rows against the fp64 block values, and its CAM bitwise equal to that
    sample's row of the batch entry (the same kernel with the same summation order)."""
    from acr_wsss_b200 import ops
    S, L, H, N = case
    p, g = _getam_inputs(S, L, H, N, dev)
    pos, gp = getam_blocks(p.cpu().numpy(), g.cpu().numpy())
    start, skip = L // 2, _skips(N)[-1]
    for func in FUNCS:
        batch = ops.getam_row0_batch(p, g, start, func, skip)
        ref, ref_rows = getam_oracle(pos, gp, start, func, skip)
        for s in sorted({0, S // 2, S - 1}):
            cam, rows = ops.getam_row0(p[:, s], g[:, s], start, func, skip, want_rows=True)
            assert torch.equal(_bits(cam[0]), _bits(batch[s])), (func, s)
            assert rel_err(rows.cpu().numpy(), ref_rows[:, s]) <= 1e-5, (func, s)
            assert rel_err(cam[0].cpu().numpy(), ref[s]) <= 1e-5, (func, s)


def test_getam_non_finite_gradients(dev):
    """NaN and infinities in the gradient behave as in torch: a NaN at a summed block makes that token's CAM NaN, a NaN at a
    block below start_layer shows only in that block's row, +inf gives +inf, -inf counts as 0, and inf * 0 (cam_grad) is NaN.
    Nothing else changes: every other element equals the clean run bit for bit."""
    from acr_wsss_b200 import ops
    S, L, H, N, start, skip = 3, 4, 3, 300, 2, 1          # 300 tokens: the probes sit in both CTAs
    p, g = _getam_inputs(S, L, H, N, dev)

    def run(gg, pp=p, func="grad"):
        return ops.getam_row0_batch(pp, gg, start, func, skip)

    def others_equal(a, b, s, j):
        keep = torch.ones_like(a, dtype=torch.bool)
        keep[s, j - skip] = False
        return torch.equal(_bits(a[keep]), _bits(b[keep]))

    for func in FUNCS:
        clean = run(g, func=func)
        # NaN at a summed block
        gn = g.clone()
        gn[3, 1, 0, 260] = float("nan")
        got = run(gn, func=func)
        assert torch.isnan(got[1, 260 - skip]), func
        assert others_equal(got, clean, 1, 260), func
        # NaN below start_layer: the CAM is unchanged, the block's row is NaN at that token only
        gn = g.clone()
        gn[0, 0, 2, 5] = float("nan")
        assert torch.equal(_bits(run(gn, func=func)), _bits(clean)), func
        cam, rows = ops.getam_row0(p[:, 0], gn[:, 0], start, func, skip, want_rows=True)
        _, rows_clean = ops.getam_row0(p[:, 0], g[:, 0], start, func, skip, want_rows=True)
        assert torch.equal(_bits(cam[0]), _bits(clean[0])), func
        assert torch.isnan(rows[0, 5]), func
        nan_rows = torch.isnan(rows)
        assert int(nan_rows.sum()) == 1, func
        assert torch.equal(_bits(rows[~nan_rows]), _bits(rows_clean[~nan_rows])), func
        # -inf counts as 0: the same bits as a zero gradient there; a token whose gradients are all -inf has a CAM of 0
        gi, gz = g.clone(), g.clone()
        gi[2, 2, 1, 7], gz[2, 2, 1, 7] = float("-inf"), 0.0
        assert torch.equal(_bits(run(gi, func=func)), _bits(run(gz, func=func))), func
        gi = g.clone()
        gi[:, 2, :, 9] = float("-inf")
        got = run(gi, func=func)
        assert float(got[2, 9 - skip]) == 0.0 and others_equal(got, clean, 2, 9), func
    # +inf: 'grad' is +inf at that token
    gi = g.clone()
    gi[3, 2, 1, 7] = float("inf")
    got = run(gi)
    assert float(got[2, 7 - skip]) == float("inf")
    assert others_equal(got, run(g), 2, 7)
    # inf * 0 in cam_grad: NaN as in torch (and still +inf for 'grad', which does not read p)
    pz = p.clone()
    pz[2, 0, 2, 40] = 0.0
    gi = g.clone()
    gi[2, 0, 2, 40] = float("inf")
    for func in ("cam_grad", "cam_grad_s"):
        got = run(gi, pz, func)
        assert torch.isnan(got[0, 40 - skip]), func
        assert others_equal(got, run(g, pz, func), 0, 40), func
    assert float(run(gi, pz, "grad")[0, 40 - skip]) == float("inf")


# ------------------------------------------------------------------ finish oracle and inputs
def _axis(n_in, n_out, align):
    """[n_out, n_in] fp64 interpolation matrix of one axis (see the module docstring)."""
    dst = np.arange(n_out, dtype=np.float64)
    if align:
        src = dst * ((n_in - 1) / (n_out - 1) if n_out > 1 else 0.0)
    else:
        src = np.maximum(n_in / n_out * (dst + 0.5) - 0.5, 0.0)
    i0 = np.floor(src).astype(np.int64)
    i1 = np.minimum(i0 + 1, n_in - 1)
    l1 = src - i0
    w = np.zeros((n_out, n_in))
    np.add.at(w, (np.arange(n_out), i0), 1.0 - l1)
    np.add.at(w, (np.arange(n_out), i1), l1)
    return w


def finish_oracle(cams_s, patch_s, grids, labels, plane):
    """One plane {offset, image, channel, kind, rows, cols} -> (normalised plane, max - min of the sum), fp64."""
    _, m, ch, kind, rows, cols = plane
    M = labels.shape[0]
    align = kind == 0
    acc = np.zeros((rows, cols))
    for cams, patch, (ph, pw) in zip(cams_s, patch_s, grids):
        wr, wc = _axis(ph, rows, align), _axis(pw, cols, align)
        for v in range(2):
            x = (patch if kind else cams)[v * M + m, :, ch].astype(np.float64).reshape(ph, pw)
            y = wr @ x @ wc.T
            if kind:
                y = y * np.float64(labels[m, ch])
            acc += y[:, ::-1] if v == 0 else y
    mn, mx = acc.min(), acc.max()
    return (acc - mn) / (mx - mn + (1e-5 if kind else 1e-6)), mx - mn


def _maps(rng, V, ph, pw, K):
    """[V, ph*pw, K] fp32 low-res maps: a row ramp (both views), a column ramp (view 1 only, so the flip does not cancel it)
    and uniform noise.  The ramps keep max - min of every plane of two or more pixels well above 1e-2."""
    x = 0.25 * rng.random((V, ph, pw, K)) + np.linspace(0.0, 1.0, ph)[None, :, None, None]
    x[V // 2:] += np.linspace(0.0, 1.0, pw)[None, None, :, None]
    return x.reshape(V, ph * pw, K).astype(np.float32)


def _finish_inputs(grids, sizes, C, npresent, seed):
    """M = len(sizes) images; image m has max(1, npresent - m % 2) present classes.  Returns numpy inputs and the plane table
    (per image its GETAM planes, then its patch-CAM planes, packed in order)."""
    rng = np.random.default_rng(seed)
    M = len(sizes)
    present = [[(3 * m + 7 * k) % C for k in range(max(1, npresent - m % 2))] for m in range(M)]
    n = max(len(q) for q in present)
    labels = np.zeros((M, C), np.float32)
    for m, q in enumerate(present):
        labels[m, q] = 0.5 + 0.5 * rng.random(len(q))
    cams_s = [_maps(rng, 2 * M, ph, pw, n) for ph, pw in grids]
    patch_s = [_maps(rng, 2 * M, ph, pw, C) for ph, pw in grids]
    planes, off = [], 0
    for m, (rows, cols) in enumerate(sizes):
        for kind in (0, 1):
            for k, c in enumerate(present[m]):
                planes.append((off, m, c if kind else k, kind, rows, cols))
                off += rows * cols
    return cams_s, patch_s, labels, planes, off


def _to(dev, xs):
    return [torch.from_numpy(x).to(dev) for x in xs]


def _lowres_bytes(grids):
    return 8 * sum(ph * pw for ph, pw in grids)


VOC = [(375, 500), (500, 375), (333, 500)]
SCALES_448 = [(14, 14), (28, 28), (42, 42), (56, 56)]              # 0.5 / 1.0 / 1.5 / 2.0 at 448
SCALES_512 = [(16, 16), (32, 32), (48, 48), (64, 64)]              # the same at 512: opt-in shared memory
# name: (grids, output sizes, C, present classes per image, low-res bytes).  The kernel's static shared memory (240 bytes on
# sm_100a) and the dynamic low-res maps share the 48 KB a block gets without the opt-in: the three smem_* sets sit just
# below that, inside the window where only the sum exceeds it, and at the 200 KB cap.
FINISH_CASES = {
    "1_scale_voc": ([(28, 28)], VOC, 20, 3, 6272),
    "2_scales_coco_and_smaller_than_grid": ([(28, 28), (56, 56)], [(480, 640), (20, 30), (1, 1)], 80, 3, 31360),
    "3_scales_non_square": ([(28, 37), (21, 28), (14, 19)], [(375, 500), (1, 13), (13, 1), (2, 40), (3, 37), (7, 5)], 20, 2,
                            15120),
    "4_scales_448": (SCALES_448, VOC + [(480, 640), (20, 30)], 20, 3, 47040),
    "4_scales_448_with_1.61": ([(14, 14), (28, 28), (45, 45), (56, 56)], [(375, 500), (20, 30), (4, 6)], 20, 2, 49128),
    "4_scales_512": (SCALES_512, [(500, 375), (333, 500), (6, 40), (1, 64)], 20, 2, 61440),
    "8_scales_short_outputs": ([(7 * k, 7 * k) for k in range(1, 9)],
                               [(h, 41) for h in range(1, 8)] + [(13, 1), (375, 500)], 20, 2, 79968),
    "8_images_C80_312_planes": ([(28, 28), (14, 14)],
                                [(37, 50), (50, 37), (33, 50), (48, 64), (20, 30), (64, 48), (7, 9), (45, 45)], 80, 20, 7840),
    "smem_78x78": ([(78, 78)], [(375, 500), (100, 100)], 20, 1, 48672),
    "smem_96x64": ([(96, 64)], [(333, 500), (1, 1)], 20, 1, 49152),
    "smem_160x160": ([(160, 160)], [(375, 500), (3, 2)], 20, 1, 204800),
}


def _check_planes(out, cams_s, patch_s, grids, labels, planes, what):
    for pl in planes:
        off, m, ch, kind, rows, cols = pl
        ref, spread = finish_oracle(cams_s, patch_s, grids, labels, pl)
        assert spread >= 1e-2 or rows * cols == 1, (what, pl, spread)
        got = out[off:off + rows * cols].view(rows, cols).cpu().numpy().astype(np.float64)
        err = np.abs(got - ref).max()
        assert err <= 2e-5, (what, pl, err)


@pytest.mark.parametrize("name", list(FINISH_CASES))
def test_cam_finish_matches_fp64(dev, name):
    from acr_wsss_b200 import ops
    grids, sizes, C, npresent, nbytes = FINISH_CASES[name]
    assert _lowres_bytes(grids) == nbytes
    cams_s, patch_s, labels, planes, total = _finish_inputs(grids, sizes, C, npresent, seed=nbytes)
    out = ops.cam_finish(_to(dev, cams_s), _to(dev, patch_s), grids, torch.from_numpy(labels).to(dev), planes, total)
    _check_planes(out, cams_s, patch_s, grids, labels, planes, name)


@pytest.mark.parametrize("name", [k for k, v in FINISH_CASES.items() if 48 * 1024 - 240 < v[4] <= 48 * 1024])
def test_cam_finish_in_window_as_the_first_launch(name):
    """The shared-memory opt-in is a per-process, per-device attribute: once any finish over 48 KB has run, every later size
    launches.  So each in-window set also runs as the first finish of a fresh process."""
    code = ("import sys, torch; sys.path[:0] = [{!r}, {!r}]; import test_cam_getam_finish as t; "
            "t.test_cam_finish_matches_fp64(torch.device('cuda:0'), {!r})").format(os.path.dirname(TESTS), TESTS, name)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]


def _finish_raw(dev, cams, patch, grids, labels, planes, out):
    """acr_cam_finish straight into a caller's buffer (ops.cam_finish allocates its own)."""
    from acr_wsss_b200 import _lib
    ns = len(grids)
    table = np.ascontiguousarray(np.asarray(planes, dtype=np.int64).reshape(-1, 6))
    ws = torch.empty(table.nbytes, device=dev, dtype=torch.uint8)
    rc = _lib.lib().acr_cam_finish(
        (ctypes.c_void_p * ns)(*[c.data_ptr() for c in cams]), (ctypes.c_void_p * ns)(*[c.data_ptr() for c in patch]),
        (ctypes.c_int * (2 * ns))(*[v for gr in grids for v in gr]), ns, labels.shape[0], cams[0].shape[-1], labels.shape[1],
        ctypes.c_void_p(labels.data_ptr()), table.ctypes.data_as(ctypes.POINTER(ctypes.c_longlong)), len(table),
        ctypes.c_void_p(out.data_ptr()), out.numel(), ctypes.c_void_p(ws.data_ptr()), table.nbytes,
        ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, _lib.lib().acr_last_error_string()
    torch.cuda.synchronize()


def test_cam_finish_exact_probes(dev):
    """Two calls are bitwise equal; a GETAM plane whose maps are all zero (a class with zero gradient) comes out exactly 0; with
    the planes packed out of order and gaps between them, the kernel writes each plane where the table says and nothing else:
    every gap element keeps a NaN sentinel."""
    from acr_wsss_b200 import ops
    grids, sizes = SCALES_448, [(375, 500), (20, 30), (7, 41)]
    cams_s, patch_s, labels, planes, total = _finish_inputs(grids, sizes, 20, 3, seed=1)
    for c in cams_s:
        c[[0, len(sizes)], :, 1] = 0.0                    # GETAM copy 1 of image 0, both views
    cams, patch, lab = _to(dev, cams_s), _to(dev, patch_s), torch.from_numpy(labels).to(dev)
    a = ops.cam_finish(cams, patch, grids, lab, planes, total)
    b = ops.cam_finish(cams, patch, grids, lab, planes, total)
    assert torch.equal(_bits(a), _bits(b))
    zero = next(pl for pl in planes if pl[1] == 0 and pl[3] == 0 and pl[2] == 1)
    assert torch.equal(_bits(a[zero[0]:zero[0] + zero[4] * zero[5]]), torch.zeros(zero[4] * zero[5], dtype=torch.int32, device=dev))

    # out of order, a gap of 1 + 37 i elements before plane i and after the last one
    order = list(range(len(planes)))[::-1]
    moved, off, mask = [], 0, []
    for i in order:
        off += 1 + 37 * i
        pl = planes[i]
        moved.append((off,) + tuple(pl[1:]))
        mask.append((off, off + pl[4] * pl[5]))
        off += pl[4] * pl[5]
    off += 1 + 37 * len(planes)
    out = torch.full((off,), SENTINEL, dtype=torch.int32, device=dev).view(torch.float32)
    _finish_raw(dev, cams, patch, grids, lab, moved, out)
    gap = torch.ones(off, dtype=torch.bool, device=dev)
    for lo, hi in mask:
        gap[lo:hi] = False
    assert bool((_bits(out)[gap] == SENTINEL).all())
    for pl, mv in zip([planes[i] for i in order], moved):
        n = pl[4] * pl[5]
        assert torch.equal(_bits(out[mv[0]:mv[0] + n]), _bits(a[pl[0]:pl[0] + n])), pl


def test_cam_finish_nan_cell_makes_its_plane_nan(dev):
    """A NaN in one low-res cell makes its whole plane NaN, as normalize_cam's amin/amax do, and leaves every other plane
    bit for bit as it was.  Probed in a GETAM plane and a patch-CAM plane, at a scale over the 48 KB default (crop 512)."""
    from acr_wsss_b200 import ops
    grids, sizes = SCALES_512, [(333, 500), (5, 40), (500, 375)]
    cams_s, patch_s, labels, planes, total = _finish_inputs(grids, sizes, 20, 3, seed=2)
    cams, patch, lab = _to(dev, cams_s), _to(dev, patch_s), torch.from_numpy(labels).to(dev)
    clean = ops.cam_finish(cams, patch, grids, lab, planes, total)
    M = len(sizes)
    # (kind, image, channel, scale, view, low-res cell)
    for kind, m, ch, s, v, cell in [(0, 1, 0, 3, 0, 64 * 63 + 5), (1, 2, planes[-1][2], 0, 1, 17), (0, 0, 1, 1, 1, 0)]:
        src = [t.clone() for t in (patch if kind else cams)]
        src[s][v * M + m, cell, ch] = float("nan")
        got = ops.cam_finish(cams if kind else src, src if kind else patch, grids, lab, planes, total)
        hit = 0
        for pl in planes:
            o, n = pl[0], pl[4] * pl[5]
            if (pl[1], pl[2], pl[3]) == (m, ch, kind):
                assert bool(torch.isnan(got[o:o + n]).all()), pl
                hit += 1
            else:
                assert torch.equal(_bits(got[o:o + n]), _bits(clean[o:o + n])), pl
        assert hit == 1
