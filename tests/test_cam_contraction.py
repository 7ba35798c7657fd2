"""GPU tier (-m gpu): the tensor-core CAM contractions at the K-splits, chunk counts and batch sizes CAM inference runs, the
batched CAM finish at multi-scale grid sets, and the batched GETAM row-0 kernel at its production shape.

csrc/refine_tc.cu is one tcgen05 kernel for two jobs: ops.affinity_refine_tc, (sum_l attn[:,l,1:,1:])^t . cam (optionally
row-normalised), and ops.patch_cam, relu(tokens . W^T + b).  launch_refine splits K over a cluster of ks in {1, 2, 4, 8}
CTAs; each CTA walks its share of 64-wide K-chunks through a two-stage shared-memory ring.  Its third chunk is the first to
reuse a stage, after an mbarrier wait whose parity flips every second trip, and the wait after the loop takes its parity from
the chunk count.  _plan mirrors launch_refine, and test_cases_reach_every_split_and_ring_path names any of these paths
(and any padded column count) that the cases below stop reaching when the heuristic changes.

Exact probes: with dyadic inputs every product and every partial sum is exact in fp32, so the kernel must reproduce the
fp64 result bit for bit, and column c of the right-hand side is nonzero on K-chunk c mod nchunks only, so a stale stage, a
chunk skipped or counted twice by the K split, or a misplaced row shows as an O(1) error in a known column.
"""
import pytest
import torch
import torch.nn.functional as F

from helpers import rel_err

pytestmark = pytest.mark.gpu

TM, TK, SMS = 128, 64, 148          # refine_tc.cu: output rows per CTA, K per chunk; the SM count launch_refine plans for


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def _plan(B, M, K):
    """launch_refine's K split of out[B, M x Nc] = A[B, M x K] . Bm[B, K x Nc]: fewest (waves of CTAs) x (chunks per CTA)."""
    mt, nch = -(-M // TM), -(-K // TK)
    ks, best, c = 1, None, 1
    while c <= 8 and c <= nch:
        cost = -(-(mt * B * c) // SMS) * -(-nch // c)
        if best is None or cost < best:
            best, ks = cost, c
        c *= 2
    per = [nch * (r + 1) // ks - nch * r // ks for r in range(ks)]
    ctas = mt * B * ks
    return dict(ks=ks, chunks=nch, nloc=(min(per), max(per)), ctas=ctas, waves=-(-ctas // SMS))


def _ncp(C, normalize):
    """Padded column count (UMMA N) of the refinement: C classes plus the all-ones row-sum column."""
    return -(-(C + int(normalize)) // 32) * 32


def _classes(C, normalize):
    return min(C, 127) if normalize else C


# (B views, L slabs, N tokens, C classes; C = 128 runs as 127 with normalisation).  L = 12 at the production shapes:
# 448 px batch of 16 views (N = 785) and configs[2] multi-scale at scale 2.0 (N = 3137).  The rest use L = 2.
CASES = [
    (16, 12, 785, 20),              # ks 1, 13 chunks
    (48, 2, 577, 40),               # ks 1, 9 chunks, 2 waves
    (12, 2, 401, 33),               # ks 2, 3-4 chunks
    (32, 2, 577, 80),               # ks 2, 4-5 chunks, 3 waves
    (4, 2, 577, 128),               # ks 4, 2-3 chunks
    (1, 12, 3137, 63),              # ks 4, 12-13 chunks
    (16, 2, 1297, 21),              # ks 4, 5-6 chunks, 5 waves
    (1, 2, 1765, 28),               # ks 8, 3-4 chunks
    (3, 2, 2305, 100),              # ks 8, 4-5 chunks, 3 waves
]
C_SWEEP_SHAPE = (12, 2, 401)
C_SWEEP = [(C, nrm) for C in (1, 31, 32, 33, 63, 64, 65, 95, 96, 127) for nrm in (False, True)] + [(128, False)]
PATCH_SHAPES = [(16, 784, 768, 20), (2, 3136, 768, 20), (8, 784, 1024, 80)]       # (B, M, E, C): 448 px ViT-B and ViT-L, scale 2.0


def _case_id(c):
    return "B%d-L%d-N%d-C%d" % c


def _patch_id(c):
    return "B%d-M%d-E%d-C%d" % c


def test_cases_reach_every_split_and_ring_path():
    rows, reached = [], []
    for B, L, N, C in CASES:
        p = _plan(B, N - 1, N - 1)
        ncps = sorted({_ncp(_classes(C, n), n) for n in (False, True)})
        rows.append("refine B=%-3d L=%-3d N=%-5d C=%-4d ks=%d chunks=%-3d per CTA=%d-%-3d CTAs=%-4d waves=%d ncp=%s"
                    % (B, L, N, C, p["ks"], p["chunks"], *p["nloc"], p["ctas"], p["waves"], ncps))
        reached.append((p, ncps))
    for B, M, E, C in PATCH_SHAPES:
        p = _plan(B, M, E)
        rows.append("patch  B=%-3d M=%-4d E=%-5d C=%-4d ks=%d chunks=%-3d per CTA=%d-%-3d CTAs=%-4d waves=%d"
                    % (B, M, E, C, p["ks"], p["chunks"], *p["nloc"], p["ctas"], p["waves"]))
    print("\n" + "\n".join(rows))
    missing = []
    for ks in (1, 2, 4, 8):
        if not any(p["ks"] == ks and p["nloc"][0] >= 3 for p, _ in reached):
            missing.append("ks=%d with >= 3 chunks on every CTA (second trip around the ring)" % ks)
        if not any(p["ks"] == ks and p["waves"] >= 2 for p, _ in reached):
            missing.append("ks=%d with >= 2 waves of CTAs" % ks)
    if not any(p["ks"] == 1 and p["nloc"][0] >= 12 for p, _ in reached):
        missing.append("ks=1 with >= 12 chunks per CTA (the 448 px batch)")
    if not any(n >= 3 and n % 2 == 1 for p, _ in reached for n in p["nloc"]):
        missing.append("an odd chunk count >= 3 on a CTA (final wait on stage 0 after a phase flip)")
    for ncp in (32, 64, 96, 128):
        if not any(ncp in n for _, n in reached):
            missing.append("ncp=%d" % ncp)
    assert not missing, missing


# ------------------------------------------------------------------ affinity refinement: exact probe
def _dyadic_attn(B, L, N, dev, seed):
    """Slabs on a 2^-8 grid in [0, 1): the sum of L <= 12 has at most 12 significant bits, so it is exact in fp32 and its bf16
    hi and lo parts are exact too (lo is nonzero for most elements, so the lo . hi products are exercised)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randint(0, 256, (B, L, N, N), generator=g, device=dev, dtype=torch.float32).div_(256)


def _chunk_local(w, nch):
    """Zero w[..., k, c] unless K-chunk k // 64 is c mod nch: output column c is then a sum over exactly one chunk."""
    K, C = w.shape[-2:]
    keep = (torch.arange(K, device=w.device) // TK)[:, None] == (torch.arange(C, device=w.device) % nch)[None, :]
    return w * keep


def _probe_cam(B, K, C, dev, seed):
    """Weights j/8, j in 1..15: exact in bf16 (their lo part is zero, so the product that the kernel drops, lo . lo, is 0)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    w = torch.randint(1, 16, (B, K, C), generator=g, device=dev, dtype=torch.float32).div_(8)
    return _chunk_local(w, -(-K // TK))


def _where(bad, nch, ks):
    """Where a mismatch [B, M, C] lies: the K-chunks of the bad columns as (chunk, CTA rank, chunk index on that CTA), and the
    views and 128-row tiles that have a bad element."""
    chunks = set()
    for c in bad.flatten(0, 1).any(0).nonzero().flatten().tolist():
        ch = c % nch
        rank = next(r for r in range(ks) if nch * r // ks <= ch < nch * (r + 1) // ks)
        chunks.add((ch, rank, ch - nch * rank // ks))
    views = bad.flatten(1).any(1).nonzero().flatten().tolist()
    tiles = sorted({i // TM for i in bad.any(2).any(0).nonzero().flatten().tolist()})
    return dict(chunk_rank_index=sorted(chunks)[:16], views=views[:16], row_tiles=tiles[:16])


def _check_exact(got, ref, normalize, nch, ks, what):
    """t = 1: bitwise equal without normalisation; within one ulp with it (one rounded division).  All values are >= 0, so the
    ulp distance is the difference of the bit patterns."""
    want = ref.float()
    if normalize:
        bad = (got.view(torch.int32).long() - want.view(torch.int32).long()).abs() > 1
    else:
        assert torch.equal(want.double(), ref), (what, "the fp64 reference is not exact in fp32: the probe's bound is broken")
        bad = got != want
    n = int(bad.sum())
    assert n == 0, (what, "%d elements differ" % n,
                    _where(bad, nch, ks), "max abs err %.3e" % float((got.double() - ref).abs().max()))


def _refine_exact(dev, B, L, N, C, normalize, seed, attn=None):
    from acr_wsss_b200 import ops
    K = N - 1
    p = _plan(B, K, K)
    attn = _dyadic_attn(B, L, N, dev, seed) if attn is None else attn
    cam = _probe_cam(B, K, C, dev, seed + 1)
    A = attn[:, :, 1:, 1:].sum(1, dtype=torch.float64)
    # Exactness bound, in units of the 2^-8 grid of A: every partial sum of the row-sum column is at most the row sum, which
    # must stay below 2^24 units (at N = 3137, L = 12: <= 3136 * 12 * 255 = 9.6e6 units).  A product column sums at most
    # 64 products, each <= 12 * 15/8 on a 2^-11 grid: <= 64 * 12 * 15 * 256 = 2.9e6 units of 2^-11.
    assert float(A.sum(-1).max()) * 256 < 2 ** 24
    assert float(A.max()) * (15 / 8) * TK * 2048 < 2 ** 24
    ref = A @ cam.double()
    if normalize:
        ref = ref / A.sum(-1, keepdim=True)
    got = ops.affinity_refine_tc(attn, cam, 1, normalize)
    _check_exact(got, ref, normalize, p["chunks"], p["ks"], ("refine", B, L, N, C, normalize))
    return attn


@pytest.mark.parametrize("B,L,N,C", CASES, ids=[_case_id(c) for c in CASES])
def test_refine_tc_exact_probe(dev, B, L, N, C):
    attn = None
    for normalize in (False, True):
        attn = _refine_exact(dev, B, L, N, _classes(C, normalize), normalize, seed=N + C, attn=attn)


@pytest.mark.parametrize("C,normalize", C_SWEEP)
def test_refine_tc_exact_probe_class_count_sweep(dev, C, normalize):
    B, L, N = C_SWEEP_SHAPE
    _refine_exact(dev, B, L, N, C, normalize, seed=1000 + C)


# ------------------------------------------------------------------ affinity refinement: realistic inputs against fp64
def _softmax_attn(B, L, N, dev, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.softmax(2.0 * torch.randn(B, L, N, N, generator=g, device=dev), -1)


def _rand_cam(B, K, C, dev, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.rand(B, K, C, generator=g, device=dev)


def _check_fp64(got, ref, what):
    """Scale-normalised max error < 5e-5 (as test_affinity_refine_tc_shapes) and, since every term is >= 0, element-wise
    relative error < 1e-4."""
    e_max = rel_err(got.cpu().numpy(), ref.cpu().numpy())
    e_elem = float(((got.double() - ref).abs() / ref.abs()).max())
    assert e_max < 5e-5 and e_elem < 1e-4, (what, e_max, e_elem)
    return e_max, e_elem


@pytest.mark.parametrize("B,L,N,C", CASES, ids=[_case_id(c) for c in CASES])
def test_refine_tc_powers_match_fp64(dev, B, L, N, C):
    """t in {1, 2, 3} with and without normalisation: later powers read back the A the first pass wrote (L = 1 path)."""
    from acr_wsss_b200 import ops
    attn = _softmax_attn(B, L, N, dev, seed=N + C)
    A = attn[:, :, 1:, 1:].sum(1, dtype=torch.float64)
    errs = {}
    for normalize in (False, True):
        Cn = _classes(C, normalize)
        cam = _rand_cam(B, N - 1, Cn, dev, seed=N + Cn)
        An = A / A.sum(-1, keepdim=True) if normalize else A
        ref = cam.double()
        for t in (1, 2, 3):
            ref = An @ ref
            got = ops.affinity_refine_tc(attn, cam, t, normalize)
            errs[(normalize, t)] = _check_fp64(got, ref, (B, L, N, Cn, normalize, t))
    print({k: "%.1e / %.1e" % v for k, v in errs.items()})


@pytest.mark.parametrize("C,normalize", C_SWEEP)
def test_refine_tc_class_count_sweep_matches_fp64(dev, C, normalize):
    from acr_wsss_b200 import ops
    B, L, N = C_SWEEP_SHAPE
    attn = _softmax_attn(B, L, N, dev, seed=2000 + C)
    cam = _rand_cam(B, N - 1, C, dev, seed=3000 + C)
    A = attn[:, :, 1:, 1:].sum(1, dtype=torch.float64)
    if normalize:
        A = A / A.sum(-1, keepdim=True)
    ref = A @ (A @ cam.double())
    _check_fp64(ops.affinity_refine_tc(attn, cam, 2, normalize), ref, (C, normalize))


def test_refine_tc_agrees_with_cuda_core_path(dev):
    """t = 2, normalised, ks = 2 over 3 waves: the tensor-core kernel against ops.affinity_apply(ops.affinity_sum(...))."""
    from acr_wsss_b200 import ops
    B, L, N, C = 32, 2, 577, 80
    attn = _softmax_attn(B, L, N, dev, seed=7)
    cam = _rand_cam(B, N - 1, C, dev, seed=8)
    got = ops.affinity_refine_tc(attn, cam, 2, True)
    old = ops.affinity_apply(ops.affinity_sum(attn, True), cam, 2)
    assert rel_err(got.cpu().numpy(), old.cpu().numpy()) < 5e-5


def test_refine_tc_is_deterministic_across_the_k_split(dev):
    """ks = 8, 3 waves: the cluster's partial tiles are reduced in rank order, so two calls give the same bits."""
    from acr_wsss_b200 import ops
    B, L, N, C = 3, 2, 2305, 100
    assert _plan(B, N - 1, N - 1)["ks"] == 8
    attn = _softmax_attn(B, L, N, dev, seed=9)
    cam = _rand_cam(B, N - 1, C, dev, seed=10)
    for t, normalize in ((1, False), (2, True)):
        a = ops.affinity_refine_tc(attn, cam, t, normalize)
        b = ops.affinity_refine_tc(attn, cam, t, normalize)
        assert torch.equal(a, b), (t, normalize)


# ------------------------------------------------------------------ patch CAM (forward; the backward is a tested closed form)
def _token_view(buf, layout, B):
    """Token 1.. of B views: every third view of a [3B, M+1, E] buffer, or rows of E+5 floats sliced to E."""
    if layout == "every_third_view":
        return buf[::3, 1:, :]
    return buf[:, 1:, :buf.shape[-1] - 5]


def _token_buffer(B, M, E, layout, dev, gen, fill):
    shape = (3 * B, M + 1, E) if layout == "every_third_view" else (B, M + 1, E + 5)
    return fill(shape, gen)


@pytest.mark.parametrize("layout", ["every_third_view", "wide_rows"])
@pytest.mark.parametrize("B,M,E,C", PATCH_SHAPES, ids=[_patch_id(c) for c in PATCH_SHAPES])
def test_patch_cam_exact_probe(dev, B, M, E, C, layout):
    """Tokens j/16 (|j| <= 128) and weights j/8 (|j| <= 15) are exact in bf16, so only hi . hi products are nonzero and each is
    exact on a 2^-7 grid.  A column sums at most 64 of them (weights chunk-local as in the refinement probe), each <= 15, so every
    partial sum stays below 64 * 15 * 128 = 122,880 units of 2^-7; the bias is on the same grid.  Pre-activations of both signs:
    the relu zeroes about half of them."""
    from acr_wsss_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(M + E + C)
    fill = lambda shape, gen: torch.randint(-128, 129, shape, generator=gen, device=dev, dtype=torch.float32).div_(16)
    tok = _token_view(_token_buffer(B, M, E, layout, dev, g, fill), layout, B)
    assert tok.shape == (B, M, E) and (tok.stride(0) != M * E or tok.stride(1) != E)
    nch = -(-E // TK)
    W = _chunk_local(torch.randint(-15, 16, (E, C), generator=g, device=dev, dtype=torch.float32).div_(8), nch).t().contiguous()
    bias = torch.randint(-256, 257, (C,), generator=g, device=dev, dtype=torch.float32).div_(128)
    pre = tok.double() @ W.double().t() + bias.double()
    assert float(pre.abs().max()) * 128 < 2 ** 24 and 0.2 < float((pre < 0).double().mean()) < 0.8
    ref = torch.relu(pre)
    got = ops.patch_cam(tok, W, bias)
    p = _plan(B, M, E)
    _check_exact(got, ref, False, nch, p["ks"], ("patch_cam", B, M, E, C, layout))


@pytest.mark.parametrize("layout", ["every_third_view", "wide_rows"])
@pytest.mark.parametrize("B,M,E,C", PATCH_SHAPES, ids=[_patch_id(c) for c in PATCH_SHAPES])
def test_patch_cam_matches_fp64(dev, B, M, E, C, layout):
    from acr_wsss_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(M + E + C + 1)
    tok = _token_view(_token_buffer(B, M, E, layout, dev, g, lambda s, gen: torch.randn(s, generator=gen, device=dev)), layout, B)
    W = torch.randn(C, E, generator=g, device=dev) * 0.05
    bias = torch.randn(C, generator=g, device=dev) * 0.1
    ref = torch.relu(tok.double() @ W.double().t() + bias.double())
    got = ops.patch_cam(tok, W, bias)
    assert rel_err(got.cpu().numpy(), ref.cpu().numpy()) < 5e-5


# ------------------------------------------------------------------ cam_finish at multi-scale grid sets
def _lowres_bytes(grids):
    return 2 * sum(ph * pw for ph, pw in grids) * 4


def _reference_finish(cams_s, patch_s, grids, labels, present, sizes):
    """The reference's finish (infer_cam.py:153-215) as torch ops, for any grid set (non-square grids included): per image
    (GETAM planes [n_m,rows,cols], patch-CAM planes [n_m,rows,cols]) summed over scales, then views (view 0 = flipped input,
    first), then min-max normalised."""
    from acr_wsss_b200.cam import normalize_cam
    M, C = labels.shape
    out = []
    for m, (rows, cols) in enumerate(sizes):
        nm = len(present[m])
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


FINISH_SETS = {
    # configs[2] multi-scale (0.5 / 1.0 / 1.5 / 2.0) at 448 px: 47,040 bytes, under the 48 KB default
    "configs2_448": ([(14, 14), (28, 28), (42, 42), (56, 56)], [(375, 500), (500, 375), (448, 448)], 47040),
    # the same scales at crop 512: 61,440 bytes, over 48 KB (opt-in shared memory)
    "crop512": ([(16, 16), (32, 32), (48, 48), (64, 64)], [(512, 512), (333, 500)], 61440),
    # 8 scales, exactly at the 200 KB cap
    "eight_scales_at_cap": ([(8, 8), (16, 16), (24, 24), (32, 32), (40, 40), (48, 48), (64, 64), (112, 140)],
                            [(300, 400), (64, 40)], 204800),
    # non-square grids; output sizes below, between and above the grid sizes
    "non_square": ([(6, 11), (12, 22), (9, 5)], [(4, 7), (3, 40), (50, 2), (123, 77), (1, 1)], 3000),
}


@pytest.mark.parametrize("name", list(FINISH_SETS))
def test_cam_finish_multi_scale_grid_sets(dev, name):
    from acr_wsss_b200 import ops
    grids, sizes, nbytes = FINISH_SETS[name]
    assert _lowres_bytes(grids) == nbytes
    M, C = len(sizes), 20
    present = [[(3 * m + 7 * k) % C for k in range(1 + m % 3)] for m in range(M)]
    n = max(len(p) for p in present)
    g = torch.Generator().manual_seed(len(grids) * 100 + M)
    labels = torch.zeros(M, C)
    for m, p in enumerate(present):
        labels[m, p] = 0.5 + 0.5 * torch.rand(len(p), generator=g)
    labels = labels.to(dev)
    cams_s = [torch.rand(2 * M, ph * pw, n, generator=g).to(dev) for ph, pw in grids]
    patch_s = [(torch.randn(2 * M, ph * pw, C, generator=g) + 0.5).relu().to(dev) for ph, pw in grids]
    planes, where, total = [], {}, 0
    for m, (rows, cols) in enumerate(sizes):
        for kind in (0, 1):
            for k in range(len(present[m])):
                planes.append((total, m, present[m][k] if kind else k, kind, rows, cols))
                where[(m, kind, k)] = total
                total += rows * cols
    out = ops.cam_finish(cams_s, patch_s, grids, labels, planes, total)
    ref = _reference_finish(cams_s, patch_s, grids, labels, present, sizes)
    for m, (rows, cols) in enumerate(sizes):
        for kind in (0, 1):
            for k in range(len(present[m])):
                o = where[(m, kind, k)]
                got = out[o:o + rows * cols].view(rows, cols)
                assert rel_err(got.cpu().numpy(), ref[m][kind][k].cpu().numpy()) <= 1e-5, (name, m, kind, k, rows, cols)


# ------------------------------------------------------------------ batched GETAM row 0 at the production shape
@pytest.mark.parametrize("L", [2, 12])
def test_getam_row0_batch_matches_fp64(dev, L):
    """S = 48 samples (16 views x 3 classes), H = 12, N = 785, every func, start_layer 0 and > 0, against an fp64 evaluation of
    DPT/ACR.py:177-215 restricted to row 0."""
    from acr_wsss_b200 import ops
    S, H, N = 48, 12, 785
    g = torch.Generator(device="cuda").manual_seed(L)
    p = torch.softmax(torch.randn(L, S, H, N, generator=g, device=dev), -1)
    dp = torch.randn(L, S, H, N, generator=g, device=dev) * 1e-2
    pos_g = dp.double().clamp(min=0).mean(2)                     # [L,S,N]
    pos_gp = (dp.double() * p.double()).clamp(min=0).mean(2)
    per = {"grad": pos_g, "grad_s": pos_g * pos_g, "cam_grad": pos_gp, "cam_grad_s": pos_gp * pos_g}
    for func, c in per.items():
        for start in (0, L // 2):
            ref = torch.relu(c[start:].sum(0))[:, 1:]
            got = ops.getam_row0_batch(p, dp, start, func, 1)
            assert got.shape == (S, N - 1)
            assert rel_err(got.cpu().numpy(), ref.cpu().numpy()) < 1e-5, (func, start)
