"""GPU tier: the bf16 attention forward (acr_attn_fwd_bf16, csrc/attn_tc.cu: attn_fwd_kernel, then attn_mean_kernel<0>) against
an fp64 reference computed on the device, element by element, and exact probes of its addressing at every tile tail, head
count and batch size the launcher accepts.

The tests call the C ABI directly, so they set every buffer, stride and pre-fill.  Every output buffer is pre-filled with a
NaN-payload sentinel and followed by a guard region: an element the kernels do not write fails every comparison, and a write
past the end fails the guard check.

Reference (fp64, from the exact bf16 inputs, one head at a time): S = q k^T, lse = logsumexp(S scale), P = exp(S scale - lse),
O = P V, A-bar = mean_h P, p_row0 = P[0].  Element-wise bounds, derived from the kernels (u = 2^-24, s2 = scale log2 e, M = the
row's max |S s2|, R = an upper bound on the row's lazy rescales, nt = key tiles, e2 = 2^-21 for ex2.approx, dS = 2^-22 sum_d
|q_d k_d|: an allowance for the tensor core's fp32 accumulation, whose rounding is not specified):
  forward terms t_j = ex2(S_j s2 - m s2) (m: the stabiliser), relative error per term
      eta = ln2 (s2 dS + 5u M) + e2 + R (ln2 6u M + e2 + u)      (s2, m s2 and the fma rounded; each rescale's alpha)
  l = sum_j t_j: 32 fp32x2 adds per lane and tile, two combines, one add per tile, one multiply per rescale
      eps_l = ln2 s2 sum_j P_j dS_j + ln2 5u M + e2 + R (...) + (33 + nt + R) u
  lse = (m s2 + log2f(l)) ln2:  |err| <= eps_l + ln2 u (2M + 2 (log2 N + 8)) + 3u |lse|           (l <= N 2^8)
  P in the mean kernel, ex2(fma(S, s2, -lse log2e)) with the kernel's own lse (its measured error d_lse):
      |err| <= P (ln2 (s2 dS + 2u |S s2| + 3u |lse log2e|) + |d_lse| + e2) + 2^-126              (ftz)
  A-bar = (sum of H terms in fp32) * fl(1/H):  (1/H) (sum_h bound_P + (H+1) u sum_h P) + 2^-126
  out: P rounded to bf16 before the P.V MMA (l sums the unrounded P), fp32 accumulation, 1/l, the bf16 store:
      |err| <= (eta + 2^-8 + 2^-20 8 nt + R u) sum_j P_j |V_jd| + (eps_l + 3u) |O_d| + 2^-8 |O_d|
Each bound carries a (1 + 2^-10) or (1 + 2^-7) factor for second-order terms.  The test prints the worst err / bound of every
output and case.  out's worst ratio is close to 1 by construction: the bf16 store reaches its half-ulp bound 2^-8 |O_d| when
O_d lies just above a power of two; the other outputs stay well below 1.  test_negative_controls shows that a dropped key column, a head missing from the mean, P rounded to bf16
before the mean and lse off by 2^-12 each land at least 10x outside these bounds.

Exact probe: keys are +-1 vectors with |k_j . k_j'| <= 48 (j != j'), queries q_i = 16 k_pi(i), so the target's score beats every
other by >= 256 scale = 32 nat: out must be V[pi(i)] bit for bit, A-bar the count of heads with pi_h(i) = j over H.
"""
import ctypes
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

D = 64
SCALE = D ** -0.5                   # 1/8, exact
BM = 128                            # attn_tc.cuh: query rows and key columns of a tile
MEAN_COLS = 32                      # attn_mean_kernel: key columns of one softmax thread (a 32-column slice of a tile)
LOG2E, LN2 = 1.0 / math.log(2.0), math.log(2.0)
S2 = SCALE * LOG2E
U = 2.0 ** -24
E2 = 2.0 ** -21                     # ex2.approx.ftz.f32 relative error allowance
C_MMA = 2.0 ** -22                  # fp32 accumulation allowance of the QK^T MMA, relative to sum |q_d k_d|
TINY = 2.0 ** -126
SENT16, SENT32 = 0x7FA5, 0x7FC0DEAD  # NaN payloads no kernel computes
GUARD = 1024
EXISTING_TOL = {"out": 1e-2, "mean": 2e-3, "row0": 2e-3}     # test_gpu_parity.test_attention_bf16_forward_vs_oracle


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def _lib():
    from acr_wsss_b200 import _lib
    return _lib


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


# ------------------------------------------------------------------ the C-ABI call, with sentinels and guards
def _sentinel(n, dev, bits=32):
    if bits == 16:
        return torch.full((n + GUARD,), SENT16, dtype=torch.int16, device=dev)
    return torch.full((n + GUARD,), SENT32, dtype=torch.int32, device=dev)


def _run(qkv, H, mean=True, row0=True, mean_view=None, mbs=None):
    """acr_attn_fwd_bf16 on fresh sentinel-filled buffers.  mean_view: a caller-owned [B,N,N] fp32 view (any batch stride mbs);
    otherwise mean=True gives a dense one.  Returns the outputs as out [B,N,H,D] bf16, lse / row0 [B,H,N], mean [B,N,N]."""
    B, N, _ = qkv.shape
    dv = qkv.device
    out_f, lse_f = _sentinel(B * N * H * D, dv, 16), _sentinel(B * H * N, dv)
    row0_f = _sentinel(B * H * N, dv) if row0 else None
    mean_f = None
    if mean_view is None and mean:
        mean_f = _sentinel(B * N * N, dv)
        mean_view, mbs = mean_f[:B * N * N].view(torch.float32).view(B, N, N), N * N
    out = out_f[:B * N * H * D].view(torch.bfloat16)
    lse = lse_f[:B * H * N].view(torch.float32)
    r0 = None if row0_f is None else row0_f[:B * H * N].view(torch.float32)
    L = _lib().lib()
    rc = L.acr_attn_fwd_bf16(_p(qkv), B, N, H, D, SCALE, _p(out), _p(lse), _p(mean_view), int(mbs or 0), _p(r0),
                             ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, f"acr_attn_fwd_bf16 failed (rc={rc}): {_lib().last_error()}"
    for name, f, s in (("out", out_f, SENT16), ("lse", lse_f, SENT32), ("p_row0", row0_f, SENT32), ("mean", mean_f, SENT32)):
        if f is not None:
            assert bool((f[-GUARD:] == s).all()), f"a write past the end of {name}"
    return dict(out=out.view(B, N, H, D), lse=lse.view(B, H, N), mean=mean_view,
                row0=None if r0 is None else r0.view(B, H, N))


# ------------------------------------------------------------------ inputs
def _inputs(dev, B, N, H, sigma, kind, seed):
    """qkv [B,N,3HD] bf16 at N(0, sigma^2); kind 'grow': keys whose norm grows with the key tile, so the forward's lazy rescale
    fires between tiles, in rows of both signs of every warp (as test_gpu_parity's lazy-rescale test)."""
    g = torch.Generator(device=dev).manual_seed(seed)
    x = torch.randn(B, N, 3, H, D, generator=g, device=dev) * sigma
    if kind == "grow":
        u = torch.randn(H, D, generator=g, device=dev)
        u = u / u.norm(dim=-1, keepdim=True)
        tile = (torch.arange(N, device=dev) // BM).float().view(1, N, 1, 1)
        x[:, :, 0] += 6.0 * torch.sign(torch.randn(B, N, H, 1, generator=g, device=dev)) * u
        x[:, :, 1] += (4.0 + 14.0 * tile) * u
    return x.reshape(B, N, 3 * H * D).to(torch.bfloat16)


# (B, N, H, sigma, kind).  N mod 128 in {0, 1, 17, 31, 32, 33, 65, 69, 96, 97, 127}; N = 129, 161, 257: dead softmax warps in the
# last query tile; 197 / 785 / 1025 / 3137: 224 / 448 / 512 px crops and scale 2.0 at 448.  H: the 3-stage Q/K ring of the
# mean kernel (h % 3, phase flips at h = 3, 6), its TMEM double buffer (h & 1, odd H) and the second LSE staging round (H > 16).
CASES = [
    (1, 1, 1, 1.5, "normal"),
    (2, 129, 3, 1.5, "normal"),
    (3, 161, 5, 3.0, "normal"),
    (2, 159, 7, 3.0, "normal"),
    (1, 160, 2, 1.5, "normal"),
    (2, 197, 12, 1.5, "normal"),
    (1, 224, 17, 3.0, "normal"),
    (2, 225, 32, 1.5, "normal"),
    (3, 255, 16, 3.0, "normal"),
    (1, 256, 4, 1.5, "normal"),
    (1, 257, 1, 3.0, "normal"),
    (1, 193, 32, 3.0, "normal"),
    (2, 785, 12, 1.5, "normal"),
    (1, 1025, 16, 3.0, "normal"),
    (1, 3137, 12, 1.5, "normal"),
    (1, 785, 3, 1.5, "grow"),
    (2, 161, 2, 1.5, "grow"),
]
PROBE_EXTRA = [(48, 785, 12), (16, 1025, 16)]      # model.forward_cam_batched: 16 views x class replicas at 448 and 512 px
PROBES = sorted({c[:3] for c in CASES} | set(PROBE_EXTRA))


def _case_id(c):
    return "B%d-N%d-H%d-s%g-%s" % c


def _probe_id(c):
    return "B%d-N%d-H%d" % c


def _shape_facts(N, H):
    nt = -(-N // BM)
    tail = N - (nt - 1) * BM
    return dict(mod=N % BM, qtiles=nt, fwd_live_quads=-(-tail // 32), mean_live_slices=-(-tail // MEAN_COLS),
                ring_laps=-(-H // 3), lse_rounds=-(-H // 16))


def test_cases_reach_every_tail_and_ring_path():
    rows = []
    for B, N, H, sigma, kind in CASES:
        f = _shape_facts(N, H)
        rows.append("B=%d N=%-5d H=%-3d sigma=%-3g %-6s N%%128=%-4d tiles=%-3d live quads / slices of the last tile=%d/%d "
                    "ring laps=%-3d lse rounds=%d" % (B, N, H, sigma, kind, f["mod"], f["qtiles"], f["fwd_live_quads"],
                                                      f["mean_live_slices"], f["ring_laps"], f["lse_rounds"]))
    rows += ["probe B=%d N=%d H=%d" % p for p in PROBES]
    print("\n" + "\n".join(rows))
    missing = []
    mods = {c[1] % BM for c in CASES}
    for m in (0, 1, 17, 31, 32, 33, 65, 69, 96, 97, 127):
        if m not in mods:
            missing.append("N mod 128 = %d" % m)
    for n in (129, 161, 257, 256, 197, 785, 1025, 3137):
        if n not in {c[1] for c in CASES}:
            missing.append("N = %d" % n)
    for h in (1, 2, 3, 4, 5, 7, 12, 16, 17, 32):
        if h not in {c[2] for c in CASES}:
            missing.append("H = %d" % h)
    if not any(c[2] % 2 == 1 and c[2] >= 7 for c in CASES):
        missing.append("odd H >= 7 (the ring's stage parity flips twice, odd count on the TMEM double buffer)")
    if max(c[0] for c in CASES) != 3:
        missing.append("B = 3 (and B <= 3) in the fp64 cases")
    for s in (1.5, 3.0):
        if s not in {c[3] for c in CASES}:
            missing.append("sigma = %g" % s)
    if not any(c[4] == "grow" and c[1] > 2 * BM for c in CASES):
        missing.append("keys growing over >= 3 key tiles (lazy rescale between tiles)")
    for n in range(1, 5):
        if not any(_shape_facts(c[1], c[2])["fwd_live_quads"] == n and c[1] > BM for c in CASES):
            missing.append("a last query tile with %d live softmax quadrant(s)" % n)
    for p in PROBE_EXTRA + [(None, None, 32)]:
        if not any(q[2] == p[2] and (p[0] is None or q[:2] == p[:2]) for q in PROBES):
            missing.append("probe %s" % (p,))
    assert not missing, missing


# ------------------------------------------------------------------ fp64 reference and bounds
class _Worst:
    """Worst err / bound per output, where it is, and max |got - ref| and max |ref| for the scale-normalised error."""

    def __init__(self):
        self.ratio, self.where, self.diff, self.ref = {}, {}, {}, {}

    def add(self, name, got, ref, bound, loc):
        err = (got.double() - ref).abs()
        r = torch.nan_to_num(err / bound, nan=float("inf"))
        k = int(r.argmax())
        v = float(r.flatten()[k])
        if v >= self.ratio.get(name, -1.0):
            self.ratio[name] = v
            self.where[name] = _locate(name, loc, k, r.shape)
        self.diff[name] = max(self.diff.get(name, 0.0), float(torch.nan_to_num(err, nan=float("inf")).max()))
        self.ref[name] = max(self.ref.get(name, 0.0), float(ref.abs().max()))

    def rel(self, name):
        return self.diff[name] / (self.ref[name] + 1e-300)

    def report(self):
        return {k: "%.3g at %s" % (v, self.where[k]) for k, v in self.ratio.items()}


def _locate(name, loc, k, shape):
    idx = list(torch.unravel_index(torch.tensor(k), shape))
    idx = [int(i) for i in idx]
    if name == "out":             # [N, D] of image b, head h
        i, d = idx
        return dict(image=loc[0], head=loc[1], query=i, query_tile=i // BM, dim=d)
    if name == "lse":
        return dict(image=loc[0], head=loc[1], query=idx[0], query_tile=idx[0] // BM)
    if name == "row0":
        j = idx[0]
        return dict(image=loc[0], head=loc[1], key=j, key_tile=j // BM, slice=(j % BM) // MEAN_COLS)
    i, j = idx
    return dict(image=loc[0], query=i, query_tile=i // BM, key=j, key_tile=j // BM, slice=(j % BM) // MEAN_COLS)


def _compare(qkv, H, got, perturb=None):
    """Every output against the fp64 reference (optionally perturbed, for the negative controls) with the bounds of the
    module docstring, which always come from the unperturbed reference."""
    B, N, _ = qkv.shape
    x = qkv.view(B, N, 3, H, D)
    nt = -(-N // BM)
    w = _Worst()
    for b in range(B):
        A = torch.zeros(N, N, dtype=torch.float64, device=qkv.device)
        Ab, Asum = torch.zeros_like(A), torch.zeros_like(A)
        for h in range(H):
            q, k, v = (x[b, :, s, h].double() for s in range(3))
            S = q @ k.t()
            dS = C_MMA * (q.abs() @ k.abs().t())
            lse = torch.logsumexp(S * SCALE, -1)
            P = torch.exp(S * SCALE - lse[:, None])
            S2a = (S * S2).abs()
            dSmax = dS.amax(-1)
            M = (S2a + S2 * dS).amax(-1)
            # each rescale raises the stabiliser by more than 8 / s2, from the first key tile's maximum to the row's
            R = ((S.amax(-1) - S[:, :BM].amax(-1) + 2 * dSmax) * S2 / 8).floor().clamp(0, nt - 1)
            per_rescale = LN2 * 6 * U * M + E2 + U
            eps_l = LN2 * S2 * (P * dS).sum(-1) + LN2 * 5 * U * M + E2 + R * per_rescale + (33 + nt + R) * U
            b_lse = (1 + 2 ** -10) * (eps_l + LN2 * U * (2 * M + 2 * (math.log2(N) + 8)) + 3 * U * lse.abs())
            eta = LN2 * (S2 * dSmax + 5 * U * M) + E2 + R * per_rescale
            O = P @ v
            b_out = ((1 + 2 ** -7) * ((eta + 2 ** -8 + 2 ** -20 * 8 * nt + R * U)[:, None] * (P @ v.abs())
                                      + (eps_l + 3 * U)[:, None] * O.abs())
                     + 2 ** -8 * O.abs() + N * 2 ** -125 * v.abs().amax(0))
            lse_k = got["lse"][b, h].double()
            dx = S2 * dS + 2 * U * S2a + 3 * U * (lse * LOG2E).abs()[:, None]
            bP = (1 + 2 ** -10) * P * (LN2 * dx + (lse_k - lse).abs()[:, None] + E2) + TINY
            P_ref, lse_ref, O_ref, P_mean = P, lse, O, P
            if perturb == "drop_last_key":
                P_ref = P.clone()
                P_ref[:, N - 1] = 0
                P_ref = P_ref / P_ref.sum(-1, keepdim=True)
                lse_ref = lse + torch.log1p(-P[:, N - 1])
                O_ref, P_mean = P_ref @ v, P_ref
            elif perturb == "drop_head":
                P_mean = torch.zeros_like(P) if h == 0 else P
            elif perturb == "bf16_P":
                P_mean = P.to(torch.bfloat16).double()
            elif perturb == "lse_shift":
                lse_ref = lse + 2.0 ** -12
            w.add("out", got["out"][b, :, h], O_ref, b_out, (b, h))
            w.add("lse", got["lse"][b, h], lse_ref, b_lse, (b, h))
            if got["row0"] is not None:
                w.add("row0", got["row0"][b, h], P_ref[0], bP[0], (b, h))
            A += P_mean
            Ab += bP
            Asum += P + bP
        if got["mean"] is not None:
            w.add("mean", got["mean"][b], A / H, (Ab + (H + 1) * U * 1.01 * Asum) / H + TINY, (b,))
    return w


@pytest.mark.parametrize("B,N,H,sigma,kind", CASES, ids=[_case_id(c) for c in CASES])
def test_forward_vs_fp64_elementwise(dev, B, N, H, sigma, kind):
    qkv = _inputs(dev, B, N, H, sigma, kind, seed=1000 * H + N)
    got = _run(qkv, H)
    w = _compare(qkv, H, got)
    print("\n%s worst err/bound: %s" % (_case_id((B, N, H, sigma, kind)), {k: "%.3f" % v for k, v in w.ratio.items()}))
    assert set(w.ratio) == {"out", "lse", "row0", "mean"}
    assert all(v <= 1.0 for v in w.ratio.values()), w.report()


# ------------------------------------------------------------------ exact permutation probe
def _probe_inputs(dev, B, N, H, seed):
    """Keys: +-1 vectors, rows resampled until |k_j . k_j'| <= 48 for j != j'.  Queries q_i = 16 k_pi(i) with pi a permutation per
    image and group of three heads (so heads share targets and counts of 2 and 3 occur); pi maps the last (partial) query tile
    onto the last key tile.  Values: nonzero bf16 from {+-1/2, +-3/4, +-1, +-2}."""
    g = torch.Generator(device=dev).manual_seed(seed)
    K = torch.randint(0, 2, (B, H, N, D), generator=g, device=dev).float() * 2 - 1
    eye = torch.eye(N, dtype=torch.bool, device=dev)
    for b in range(B):
        for _ in range(50):
            G = (K[b] @ K[b].transpose(-1, -2)).abs().masked_fill(eye, 0)
            bad = (G > 48).any(-1)                                  # [H, N]
            if not bool(bad.any()):
                break
            n = int(bad.sum())
            K[b][bad] = torch.randint(0, 2, (n, D), generator=g, device=dev).float() * 2 - 1
        G = (K[b] @ K[b].transpose(-1, -2)).abs().masked_fill(eye, 0)
        assert float(G.max()) <= 48, "key set with a score gap below 256"
    t0 = (N - 1) // BM * BM
    gc = torch.Generator().manual_seed(seed)
    perms = torch.empty(B, H, N, dtype=torch.long)
    for b in range(B):
        for grp in range(-(-H // 3)):
            pi = torch.cat([torch.randperm(t0, generator=gc), t0 + torch.randperm(N - t0, generator=gc)])
            perms[b, 3 * grp:3 * grp + 3] = pi
    perms = perms.to(dev)
    vals = torch.tensor([0.5, 0.75, 1.0, 2.0, -0.5, -0.75, -1.0, -2.0], device=dev)
    V = vals[torch.randint(0, 8, (B, H, N, D), generator=g, device=dev)]
    Q = 16 * torch.gather(K, 2, perms[..., None].expand(B, H, N, D))
    x = torch.stack([Q, K, V], 1).permute(0, 3, 1, 2, 4)            # [B,N,3,H,D]
    return x.reshape(B, N, 3 * H * D).to(torch.bfloat16).contiguous(), perms, V


def _bad_report(bad, perms, kind):
    """Where the first mismatches are: image, head, query tile, key tile and 32-column slice of the target."""
    idx = bad.nonzero()[:8].tolist()
    rep = []
    for t in idx:
        if kind == "out":                           # [B,N,H,D]
            b, i, h, _ = t
            j = int(perms[b, h, i])
        elif kind == "lse":                         # [B,H,N]
            b, h, i = t
            j = int(perms[b, h, i])
        elif kind == "row0":                        # [B,H,N]
            b, h, j = t
            i = 0
        else:                                       # [B,N,N]
            b, i, j = t
            h = [hh for hh in range(perms.shape[1]) if int(perms[b, hh, i]) == j]
        rep.append(dict(image=b, head=h, query_tile=i // BM, key_tile=j // BM, slice=(j % BM) // MEAN_COLS, query=i, key=j))
    return "%d mismatches, first: %s" % (int(bad.sum()), rep)


@pytest.mark.parametrize("B,N,H", PROBES, ids=[_probe_id(c) for c in PROBES])
def test_permutation_probe_is_exact(dev, B, N, H):
    qkv, perms, V = _probe_inputs(dev, B, N, H, seed=7 * N + H + B)
    got = _run(qkv, H)
    # out: V[pi(i)] bit for bit
    want = torch.gather(V, 2, perms[..., None].expand(B, H, N, D)).permute(0, 2, 1, 3).to(torch.bfloat16)
    bad = got["out"].view(torch.int16) != want.view(torch.int16)
    assert not bool(bad.any()), ("out", _bad_report(bad, perms, "out"))
    # lse = 1024 scale + log(1 + mass < 2^-34): relative error of three fp32 roundings
    bad = ((got["lse"].double() - 1024 * SCALE).abs() > 1024 * SCALE * 2.0 ** -20) | torch.isnan(got["lse"])
    assert not bool(bad.any()), ("lse", _bad_report(bad, perms, "lse"))
    # A-bar: count / H within 2^-13 on the targets, <= 2^-40 elsewhere
    cnt = torch.zeros(B, N, N, device=dev)
    cnt.scatter_add_(2, perms.permute(0, 2, 1), torch.ones(B, N, H, device=dev))
    assert int(cnt.max()) >= min(H, 2)
    A = got["mean"].double()
    tgt = cnt > 0
    exp = cnt.double() / H
    bad = torch.where(tgt, ~((A - exp).abs() <= exp * 2.0 ** -13), ~(A.abs() <= 2.0 ** -40))
    assert not bool(bad.any()), ("mean", _bad_report(bad, perms, "mean"))
    # p_row0: 1 at pi(0), <= 2^-40 elsewhere
    one = torch.zeros(B, H, N, dtype=torch.bool, device=dev)
    one.scatter_(2, perms[:, :, :1], torch.ones_like(perms[:, :, :1], dtype=torch.bool))
    r0 = got["row0"].double()
    bad = torch.where(one, ~((r0 - 1).abs() <= 2.0 ** -13), ~(r0.abs() <= 2.0 ** -40))
    assert not bool(bad.any()), ("row0", _bad_report(bad, perms, "row0"))


# ------------------------------------------------------------------ layout and write footprint
def _same_bits(a, b):
    return a.shape == b.shape and torch.equal(a.contiguous().view(torch.int32 if a.element_size() == 4 else torch.int16),
                                              b.contiguous().view(torch.int32 if b.element_size() == 4 else torch.int16))


def test_mean_into_a_stack_slot_and_write_footprint(dev):
    """A-bar into slot 1 of a sentinel-filled [B,3,N,N] stack: slot 1 matches the reference, slots 0 and 2 keep every sentinel
    bit (the guards after out, lse and p_row0 are checked by _run).  A base offset by 4 bytes gives the same bits; so do calls
    without p_row0 (A-bar, out, lse) and without A-bar (out, lse)."""
    B, N, H = 3, 300, 5
    qkv = _inputs(dev, B, N, H, 1.5, "normal", seed=17)
    stack_f = _sentinel(B * 3 * N * N, dev)
    stack = stack_f[:B * 3 * N * N].view(torch.float32).view(B, 3, N, N)
    got = _run(qkv, H, mean_view=stack[:, 1], mbs=3 * N * N)
    assert bool((stack_f[-GUARD:] == SENT32).all())
    raw = stack_f[:B * 3 * N * N].view(B, 3, N, N)
    assert bool((raw[:, 0] == SENT32).all()) and bool((raw[:, 2] == SENT32).all()), "a write outside slot 1"
    w = _compare(qkv, H, got)
    assert all(v <= 1.0 for v in w.ratio.values()), w.report()
    dense = _run(qkv, H)
    assert _same_bits(dense["mean"], got["mean"]) and _same_bits(dense["out"], got["out"]) and _same_bits(dense["lse"], got["lse"])
    flat = _sentinel(B * N * N + 1, dev)
    shifted = flat[1:1 + B * N * N].view(torch.float32).view(B, N, N)
    assert shifted.data_ptr() % 8 == 4
    off = _run(qkv, H, mean_view=shifted, mbs=N * N)
    assert int(flat[0]) == SENT32 and bool((flat[1 + B * N * N:] == SENT32).all())
    assert _same_bits(off["mean"], dense["mean"]) and _same_bits(off["row0"], dense["row0"])
    no_row0 = _run(qkv, H, row0=False)
    assert _same_bits(no_row0["mean"], dense["mean"]) and _same_bits(no_row0["out"], dense["out"])
    assert _same_bits(no_row0["lse"], dense["lse"])
    no_mean = _run(qkv, H, mean=False, row0=False)
    assert _same_bits(no_mean["out"], dense["out"]) and _same_bits(no_mean["lse"], dense["lse"])


# ------------------------------------------------------------------ determinism and batch independence
def test_bits_do_not_depend_on_the_call_or_the_batch_position(dev):
    """No atomics, no cross-CTA sums: two calls give the same bits, and an image alone gives the same bits as at index 0, 17
    and 47 of a batch of 48 (the CAM inference batch: 16 views x 3 classes, N = 785, H = 12)."""
    B, N, H = 48, 785, 12
    one = _inputs(dev, 1, N, H, 1.5, "normal", seed=5)
    batch = _inputs(dev, B, N, H, 1.5, "normal", seed=6)
    for i in (0, 17, 47):
        batch[i] = one[0]
    a, b = _run(batch, H), _run(batch, H)
    for k in ("out", "lse", "mean", "row0"):
        assert _same_bits(a[k], b[k]), k
    alone = _run(one, H)
    for i in (0, 17, 47):
        for k in ("out", "lse", "mean", "row0"):
            assert _same_bits(a[k][i:i + 1], alone[k]), (k, i)


# ------------------------------------------------------------------ non-finite inputs
def test_nan_inputs_follow_the_reference(dev):
    """B = 2, N = 257, H = 3; a NaN in image 1, head 1.  In q_i (i = 0 and N-1): those rows of out[.., h], lse[h] and A-bar are
    NaN (p_row0[h] too, through row 0), all else bitwise unchanged.  In k_j (j = N-1, the tail column): every row of head h is
    NaN in out, lse and p_row0, and A-bar of the image is NaN.  In v_j: out[.., h] is NaN, lse and A-bar bitwise unchanged.
    Image 0 is bitwise unchanged in every case."""
    B, N, H, hb = 2, 257, 3, 1
    qkv = _inputs(dev, B, N, H, 1.5, "normal", seed=9)
    clean = _run(qkv, H)
    nan = float("nan")

    def hit(s, rows):
        x = qkv.clone().view(B, N, 3, H, D)
        for r in rows:
            x[1, r, s, hb, 3] = nan
        return _run(x.view(B, N, 3 * H * D), H)

    def unchanged(got, keep):
        for k in ("out", "lse", "mean", "row0"):
            m = keep[k]
            assert _same_bits(got[k][m], clean[k][m]), k

    def masks():
        return {k: torch.ones_like(clean[k], dtype=torch.bool) for k in ("out", "lse", "mean", "row0")}

    # NaN in queries 0 and N-1 of head hb
    rows = [0, N - 1]
    got = hit(0, rows)
    keep = masks()
    keep["out"][1, rows, hb] = False
    keep["lse"][1, hb, rows] = False
    keep["mean"][1, rows] = False
    keep["row0"][1, hb] = False
    for k in keep:
        nan_part = got[k][~keep[k]]
        assert bool(torch.isnan(nan_part.float()).all()), ("q", k)
    unchanged(got, keep)
    # NaN in key N-1 of head hb
    got = hit(1, [N - 1])
    keep = masks()
    keep["out"][1, :, hb] = False
    keep["lse"][1, hb] = False
    keep["mean"][1] = False
    keep["row0"][1, hb] = False
    for k in keep:
        assert bool(torch.isnan(got[k][~keep[k]].float()).all()), ("k", k)
    unchanged(got, keep)
    # NaN in value 130 of head hb (dimension 3: the other 63 dimensions of out are unchanged)
    got = hit(2, [130])
    keep = masks()
    keep["out"][1, :, hb, 3] = False
    assert bool(torch.isnan(got["out"][~keep["out"]].float()).all()), "v"
    unchanged(got, keep)


# ------------------------------------------------------------------ the bounds have teeth
def test_negative_controls(dev):
    """The kernels against deliberately wrong references, at B = 2, N = 785, H = 12: each must land >= 10x outside the bounds.
    Printed: whether the scale-normalised errors of test_gpu_parity's forward test (out 1e-2, A-bar and p_row0 2e-3; lse is
    not compared there) would have let the same wrong reference pass."""
    B, N, H = 2, 785, 12
    qkv = _inputs(dev, B, N, H, 1.5, "normal", seed=785)
    got = _run(qkv, H)
    base = _compare(qkv, H, got)
    assert all(v <= 1.0 for v in base.ratio.values()), base.report()
    controls = {"drop_last_key": ("out", "lse", "mean", "row0"), "drop_head": ("mean",), "bf16_P": ("mean",), "lse_shift": ("lse",)}
    lines = []
    for name, outs in controls.items():
        w = _compare(qkv, H, got, perturb=name)
        worst = max(w.ratio[o] for o in outs)
        old = {o: ("passes" if w.rel(o) < EXISTING_TOL[o] else "fails") + " (%.2e)" % w.rel(o) for o in outs if o in EXISTING_TOL}
        lines.append("%-14s worst err/bound %.3g; existing tolerances: %s" % (name, worst, old or "lse not compared"))
        assert worst >= 10, (name, w.report())
    print("\n" + "\n".join(lines))
