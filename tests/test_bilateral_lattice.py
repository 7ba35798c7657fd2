"""The permutohedral bilateral filter (csrc/bilateral.cu, csrc/lattice.cuh) against the C oracle (oracle/permuto_oracle.c),
value by value, at every plane count, tile tail and batch chunk the kernels distinguish.

Where the kernels branch: the splat works on 16 x 8 pixel tiles with an odd float4 row stride Q|1 (Q = ceil(K/4)) and sends
a pair whose slot table neighbourhood is full (kSlotProbes probes) straight to global memory; the slice serves a pixel
with 8, 16 or 32 lanes for Q <= 8, <= 16, <= 24; K <= 96; images go through 8 at a time, so N > 8 reads a second chunk's
pointers and lattice sizes; an image whose H*W is not a multiple of 4 has phantom pad pixels (all-zero features) whose
vertices take part in the blur.

Exact probes.  The kernels differ from the oracle only in the order of the splat additions (header of bilateral.cu): the
embedding, the six blur passes and the slice use the same roundings in the same order (__fmul_rn / __fadd_rn; the oracle is
built with -ffp-contract=off).  When every plane holds a single nonzero pixel, every (vertex, plane) of the lattice receives
at most one product, fmaf(w, x, 0) rounds like w*x and adding zeros is exact, so the GPU result must be BITWISE equal to the
oracle's.  Any error in plane routing, neighbour ids, tile tails or chunk offsets breaks that.

Dense probes.  With nonnegative planes every output is a sum of nonnegative terms, so an elementwise relative error is
well defined; its size is set by the splat's float-atomic order only (DENSE_TOL below).

Noise images at sxy = srgb = 1 put nearly 768 distinct vertices into the 1024 splat slots of a tile; replaying the slot
table's linear probing with 768 distinct ids on the CPU, about two thirds of such tiles have a pair that finds no slot
within 32 probes, so the 224 x 224 noise cases run the splat's global-memory fallback on hundreds of tiles.

The negative controls at the end need no GPU: applied to oracle outputs, each error these tests target must fail the
check that targets it.
"""
import numpy as np
import pytest
import torch

from oracle import bilateral_oracle as bo

KS = (1, 2, 3, 4, 5, 8, 31, 32, 33, 63, 64, 65, 93, 96)
SIZES = ((1, 1), (1, 17), (7, 15), (8, 16), (9, 17), (33, 31), (224, 224))     # H*W mod 4 = 1, 1, 1, 0, 1, 3, 0
NS = (1, 8, 9, 17)
# (image kind, sigma_rgb, sigma_xy): the cfg4 sigmas (15, 100 * 0.5) on smooth images, moderate and near-worst-case
# lattices on white noise, and one colour per image (hundreds of pairs in one splat slot).
KINDS = (("smooth", 15.0, 50.0), ("noise", 5.0, 3.0), ("noise", 1.0, 1.0), ("const", 15.0, 50.0))

# Largest elementwise relative error of the dense probes, measured on a B200 (1000 W): 1.7e-6 (test_dense_elementwise,
# at 224 x 224; 1.1e-6 at 33 x 31, <= 7e-7 on the smaller sizes) and 5.5e-7 at the cfg4 shape N = 8, K = 81, 224 x 224.
DENSE_TOL = 5e-6


def _images(kind, N, H, W, seed):
    g = torch.Generator().manual_seed(seed)
    if kind == "smooth":
        from acr_wsss_b200 import synth
        return synth.smooth_rgb(N, H, W, seed=seed).numpy()
    if kind == "noise":
        return (torch.rand(N, 3, H, W, generator=g) * 255).numpy()
    return (torch.rand(N, 3, 1, 1, generator=g) * 255).expand(N, 3, H, W).contiguous().numpy()


def _positions(H, W):
    """Pixel indices, the ones where the kernels change behaviour first: image corners, splat tile corners, the last pixels
    (next to the phantom pads), then every other pixel in a seeded order."""
    HW = H * W
    special = [0, W - 1, (H - 1) * W, HW - 1, HW - 2, HW - 3, HW - 4]
    for y in (7, 8, 15, 16):
        for x in (15, 16, 31, 32):
            special.append(y * W + x if y < H and x < W else -1)
    seen, order = set(), []
    for p in special:
        if 0 <= p < HW and p not in seen:
            seen.add(p)
            order.append(p)
    rest = np.random.default_rng(HW).permutation(HW)
    return order + [int(p) for p in rest if int(p) not in seen]


def _impulses(N, K, H, W, seed):
    """ins [N,K,H,W]: plane k of image n is zero except at one pixel, a different pixel for every plane while K <= H*W."""
    order = _positions(H, W)
    rng = np.random.default_rng(seed)
    ins = np.zeros((N, K, H * W), np.float32)
    for n in range(N):
        for k in range(K):
            ins[n, k, order[(k + n) % len(order)]] = rng.uniform(0.5, 2.0)
    return ins.reshape(N, K, H, W)


def _dense(N, K, H, W, seed):
    return np.random.default_rng(seed).uniform(0.05, 1.0, (N, K, H, W)).astype(np.float32)


def _case(iK, iS):
    """(N, kind) of grid point (KS[iK], SIZES[iS]): every K meets every N and kind across the sizes."""
    return NS[(iK + iS) % len(NS)], KINDS[iK % len(KINDS)]


def _gpu(images, ins, srgb, sxy):
    from acr_wsss_b200 import ops
    out, m = ops.bilateral_filter(torch.from_numpy(images).cuda(), torch.from_numpy(np.ascontiguousarray(ins)).cuda(), srgb, sxy,
                                  return_lattice_size=True)
    return out.cpu().numpy(), m


# ------------------------------------------------------------------ the checks (shared with the negative controls)
def check_bitwise(ours, ref, what):
    ours, ref = np.ascontiguousarray(ours, np.float32), np.ascontiguousarray(ref, np.float32)
    assert ours.shape == ref.shape, what
    diff = ours.view(np.uint32) != ref.view(np.uint32)
    if diff.any():
        i = tuple(int(v) for v in np.argwhere(diff)[0])
        raise AssertionError(f"{what}: {int(diff.sum())} of {diff.size} values differ from the oracle's bits, "
                             f"first at {i}: {ours[i]!r} vs {ref[i]!r}")


def max_rel(ours, ref):
    ref = np.asarray(ref, np.float64)
    assert (ref > 0).all(), "dense probes: every reference value is a positive sum"
    return float((np.abs(np.asarray(ours, np.float64) - ref) / ref).max())


def check_dense(ours, ref, what):
    e = max_rel(ours, ref)
    assert e <= DENSE_TOL, f"{what}: elementwise relative error {e:.3e} > {DENSE_TOL:.0e}"
    return e


def check_sizes(ours, ref, what):
    assert list(ours) == list(ref), f"{what}: lattice vertex counts {list(ours)} != oracle {list(ref)}"


# ------------------------------------------------------------------ GPU tier
@pytest.mark.gpu
@pytest.mark.parametrize("iS", range(len(SIZES)), ids=[f"{h}x{w}" for h, w in SIZES])
def test_impulses_bitwise_equal_to_oracle(iS):
    H, W = SIZES[iS]
    for iK, K in enumerate(KS):
        N, (kind, srgb, sxy) = _case(iK, iS)
        what = f"K={K} N={N} {H}x{W} {kind} srgb={srgb} sxy={sxy}"
        img, ins = _images(kind, N, H, W, seed=100 * iS + iK), _impulses(N, K, H, W, seed=iK)
        out, m = _gpu(img, ins, srgb, sxy)
        check_bitwise(out, bo.oracle_bilateral(img, ins, srgb, sxy), what)
        check_sizes(m, bo.oracle_lattice_sizes(img, srgb, sxy), what)


@pytest.mark.gpu
@pytest.mark.parametrize("iS", range(len(SIZES)), ids=[f"{h}x{w}" for h, w in SIZES])
def test_dense_elementwise(iS):
    H, W = SIZES[iS]
    worst = 0.0
    for iK, K in enumerate(KS):
        N, (kind, srgb, sxy) = _case(iK, iS)
        img, ins = _images(kind, N, H, W, seed=100 * iS + iK + 7), _dense(N, K, H, W, seed=iK)
        out, _ = _gpu(img, ins, srgb, sxy)
        worst = max(worst, check_dense(out, bo.oracle_bilateral(img, ins, srgb, sxy), f"K={K} N={N} {H}x{W} {kind}"))
    print(f"dense {H}x{W}: max elementwise relative error {worst:.3e}")


@pytest.mark.gpu
def test_dense_elementwise_cfg4_shape():
    """The filter of the COCO-shaped step: N = 8 images, K = 81 planes (softmax over background + 80 classes), 224 x 224."""
    from acr_wsss_b200 import synth
    img = synth.smooth_rgb(8, 224, 224, seed=4).numpy()
    ins = synth.probabilities(8, 81, 224, 224, seed=4).numpy()
    out, m = _gpu(img, ins, 15.0, 50.0)
    e = check_dense(out, bo.oracle_bilateral(img, ins, 15.0, 50.0), "cfg4")
    check_sizes(m, bo.oracle_lattice_sizes(img, 15.0, 50.0), "cfg4")
    print(f"dense cfg4: max elementwise relative error {e:.3e}")


@pytest.mark.gpu
@pytest.mark.parametrize("kind,srgb,sxy,N,H,W", [
    ("smooth", 15.0, 50.0, 9, 224, 224),
    ("noise", 1.0, 1.0, 9, 224, 224),            # near-worst case: almost 6 vertices per pixel
    ("const", 15.0, 50.0, 9, 224, 224),
    ("const", 15.0, 50.0, 17, 1, 1),
] + [("noise", 5.0, 3.0, 17, H, W) for H, W in SIZES[:-1]])
def test_lattice_size_equals_oracle(kind, srgb, sxy, N, H, W):
    """M of every image, in both batch chunks, is the oracle's exact vertex count (a zero input must also come out zero)."""
    img = _images(kind, N, H, W, seed=H * W + N)
    zeros = np.zeros((N, 1, H, W), np.float32)
    out, m = _gpu(img, zeros, srgb, sxy)
    ref = bo.oracle_lattice_sizes(img, srgb, sxy)
    check_sizes(m, ref, f"{kind} N={N} {H}x{W}")
    assert not out.any()
    if kind == "noise" and sxy == 1.0:
        assert min(ref) > 5.9 * H * W


@pytest.mark.gpu
def test_host_drop_in_grow_only_cache_is_bitwise_equal_to_device_entry():
    """bilateralfilter_batch (host buffers, device buffers and workspace cached per device, grow-only) at sizes small ->
    large -> small -> larger K on fewer pixels: every call bit for bit the device entry's result, and the oracle's."""
    from acr_wsss_b200 import bilateralfilter_batch
    for i, (N, K, H, W) in enumerate([(1, 3, 7, 15), (17, 33, 224, 224), (2, 5, 9, 17), (9, 96, 33, 31), (1, 1, 1, 1),
                                      (3, 21, 8, 16)]):
        img, ins = _images("smooth", N, H, W, seed=i), _impulses(N, K, H, W, seed=i)
        host = np.full(ins.size, np.nan, np.float32)
        bilateralfilter_batch(img.reshape(-1), ins.reshape(-1), host, N, K, H, W, 15.0, 50.0)
        dev, _ = _gpu(img, ins, 15.0, 50.0)
        what = f"call {i}: N={N} K={K} {H}x{W}"
        check_bitwise(host.reshape(N, K, H, W), dev, what)
        check_bitwise(dev, bo.oracle_bilateral(img, ins, 15.0, 50.0), what)


# ------------------------------------------------------------------ negative controls (CPU: oracle only)
def _control_inputs():
    N, K, H, W = 9, 5, 9, 17
    img = _images("noise", N, H, W, seed=3)
    return img, _impulses(N, K, H, W, seed=3), _dense(N, K, H, W, seed=3), 5.0, 3.0


def test_controls_swapped_planes_fail():
    img, imp, dense, srgb, sxy = _control_inputs()
    for ins, check in ((imp, check_bitwise), (dense, check_dense)):
        ref = bo.oracle_bilateral(img, ins, srgb, sxy)
        check(ref, ref, "unchanged")
        bad = ref.copy()
        bad[:, [1, 3]] = ref[:, [3, 1]]
        with pytest.raises(AssertionError):
            check(bad, ref, "planes 1 and 3 swapped")


def test_controls_impulse_moved_by_one_pixel_fails():
    img, imp, _, srgb, sxy = _control_inputs()
    ref = bo.oracle_bilateral(img, imp, srgb, sxy)
    for n, k in ((0, 0), (8, 4)):
        moved = imp.copy()
        (y, x), = np.argwhere(imp[n, k] != 0)
        moved[n, k, y, x] = 0.0
        moved[n, k, y, x + 1 if x + 1 < imp.shape[3] else x - 1] = imp[n, k, y, x]
        with pytest.raises(AssertionError):
            check_bitwise(bo.oracle_bilateral(img, moved, srgb, sxy), ref, f"impulse of image {n} plane {k} moved")


def test_controls_dropped_blur_pass_fails():
    img, imp, dense, srgb, sxy = _control_inputs()
    for ins, check in ((imp, check_bitwise), (dense, check_dense)):
        ref = bo.oracle_bilateral(img, ins, srgb, sxy)
        for j in range(6):
            with pytest.raises(AssertionError):
                check(bo.oracle_bilateral(img, ins, srgb, sxy, skip_blur_axis=j), ref, f"blur pass {j} dropped")


def test_controls_image_replaced_by_its_neighbour_fails():
    """Image 8 (the first of the second chunk of 8) replaced by image 7."""
    img, imp, dense, srgb, sxy = _control_inputs()
    for ins, check in ((imp, check_bitwise), (dense, check_dense)):
        ref = bo.oracle_bilateral(img, ins, srgb, sxy)
        bad = ref.copy()
        bad[8] = ref[7]
        with pytest.raises(AssertionError):
            check(bad, ref, "image 8 <- image 7")
    m = bo.oracle_lattice_sizes(img, srgb, sxy)
    assert m[8] != m[7]
    with pytest.raises(AssertionError):
        check_sizes(m[:8] + [m[7]], m, "image 8 <- image 7")
