"""GPU tier: every form in which the consistency loss's gradient G = dLoss/dA-bar (A-bar: head-mean attention map) reaches the
bf16 attention backward, against fp64 oracles at shapes with several key and query tiles and thin last tiles.

acr_attn_bwd_bf16 takes G as
  - sign codes from acr_consistency_fwd_bwd (one byte per element, rows padded to 128 bytes): the training step;
  - dense fp32 rows whose row and batch strides are multiples of 4 on a 16-byte aligned base: read with 128-bit loads on full
    key tiles (the padded rows of ops.consistency_fwd_bwd, i.e. the non-code fallback);
  - dense fp32 in any other layout: read element by element (autograd's dense gradient).
Each of them has its own code path in the tile body and in the delta pre-pass.  The tests call the C ABI directly, so they
control every stride and every pre-filled buffer.  N = 129, 257 and 1025 leave one live key column and one live query row in
the last tile; N = 785 is the 448x448 training shape (seven tiles, 17 keys in the last one).
"""
import ctypes

import pytest
import torch

pytestmark = pytest.mark.gpu

BF16_TOL = 1e-2
TOL = {"q": 2 * BF16_TOL, "k": 2 * BF16_TOL, "v": 2 * BF16_TOL, "q_row0": 2 * BF16_TOL, "q_rows": 2 * BF16_TOL, "g_row0": BF16_TOL}
D = 64
SCALE = D ** -0.5
PLUS, MINUS, PAD = 0x3F, 0xBF, 0x7F      # code bytes (top byte of +-0.5f); 0x7F decodes to ~1.7e38


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def _lib():
    from acr_wsss_b200 import _lib
    return _lib


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ok(rc, what):
    assert rc == 0, f"{what} failed (rc={rc}): {_lib().last_error()}"


def _rup(n, m):
    return (n + m - 1) // m * m


def _orc():
    from oracle import acr_oracle as orc
    return orc


def _rel(a, b):
    """max |a-b| / max |b| in fp64 (the scale-normalised max error of tests/helpers.py, computed where the tensors live)."""
    a, b = a.double(), b.double()
    return float((a - b).abs().max() / (b.abs().max() + 1e-300))


# ------------------------------------------------------------------ C-ABI calls
def _inputs(dev, B, N, H, seed):
    g = torch.Generator().manual_seed(seed)
    qkv = (torch.randn(B, N, 3 * H * D, generator=g) * 1.5).to(torch.bfloat16).to(dev)
    d_out = torch.randn(B, N, H * D, generator=g).to(torch.bfloat16).to(dev)
    return qkv, d_out, g


def _forward(qkv, H):
    B, N, _ = qkv.shape
    out = torch.empty(B, N, H * D, device=qkv.device, dtype=torch.bfloat16)
    lse = torch.empty(B, H, N, device=qkv.device)
    _ok(_lib().lib().acr_attn_fwd_bf16(_p(qkv), B, N, H, D, SCALE, _p(out), _p(lse), None, 0, None, _stream()), "acr_attn_fwd_bf16")
    return out, lse


def _backward(qkv, out, lse, d_out, H, g=None, code=None, w=(0.0, 0.0), g_scale=None):
    """g: [B,N,N] fp32 with unit column stride (any row / batch stride, any base); code: [B,N,ld] uint8 with unit column stride.
    Returns (d_qkv, g_row0); both are pre-filled with NaN, so an element the kernels do not write fails every comparison."""
    B, N, _ = qkv.shape
    L = _lib().lib()
    d_qkv = torch.full_like(qkv, float("nan"))
    g_row0 = torch.full((B, H, N), float("nan"), device=qkv.device)
    wsb = L.acr_attn_bwd_bf16_workspace(B, N, H, D)
    ws = torch.empty(wsb, device=qkv.device, dtype=torch.uint8)
    gs, cs = (0, 0), (0, 0)
    if g is not None:
        assert g.dtype == torch.float32 and g.stride(2) == 1
        gs = (g.stride(0), g.stride(1))
    if code is not None:
        assert code.dtype == torch.uint8 and code.stride(2) == 1
        cs = (code.stride(0), code.stride(1))
    _ok(L.acr_attn_bwd_bf16(_p(qkv), _p(out), _p(lse), _p(d_out), B, N, H, D, SCALE, _p(g), gs[0], gs[1], _p(code), cs[0], cs[1],
                            float(w[0]), float(w[1]), _p(g_scale), _p(d_qkv), _p(g_row0), _p(ws), wsb, _stream()), "acr_attn_bwd_bf16")
    return d_qkv, g_row0


def _consistency(a1, a2, p, c1=None, c2=None, c_ld=0, g1=None, g2=None, g_ld=0, alpha=(100.0, 100.0)):
    B, L_, N, _ = a1.shape
    L = _lib().lib()
    loss2 = torch.full((2,), float("nan"), device=a1.device)
    wsb = L.acr_consistency_workspace(B, L_, N)
    ws = torch.empty(wsb, device=a1.device, dtype=torch.uint8)
    _ok(L.acr_consistency_fwd_bwd(_p(a1), _p(a2), B, L_, N, p, alpha[0], alpha[1], _p(loss2), _p(g1), _p(g2), g_ld,
                                  _p(c1), _p(c2), c_ld, _p(ws), wsb, _stream()), "acr_consistency_fwd_bwd")
    return loss2


# ------------------------------------------------------------------ sign codes: the test's own decoder and generator
def _decode(code, N, w_cls, w_aff, scale=1.0):
    """[B,N,ld] sign codes -> the fp64 [B,N,N] gradient they stand for: 0x3F -> +1, 0xBF -> -1, 0x00 -> 0; row 0 times w_cls,
    the other rows times w_aff; everything times scale.  Any other byte in [0, N) is an error."""
    c = code[..., :N]
    assert bool(((c == 0) | (c == PLUS) | (c == MINUS)).all())
    s = (c == PLUS).double() - (c == MINUS).double()
    w = torch.full((N, 1), float(w_aff), dtype=torch.float64, device=code.device)
    w[0, 0] = float(w_cls)
    return s * w * scale


def _random_codes(gen, B, N, dev, L=3, l=1, extra_ld=0):
    """Slot l of a [B,L,N,ld] code stack (ld = N padded to 128, plus extra_ld) with random bytes from {0x00, 0x3F, 0xBF} in
    every column, column 0 included, and zero padding.  The slot's batch stride is L*N*ld bytes."""
    ld = _rup(N, 128) + extra_ld
    stack = torch.zeros(B, L, N, ld, dtype=torch.uint8)
    stack[..., :N] = torch.tensor([0, PLUS, MINUS], dtype=torch.uint8)[torch.randint(0, 3, (B, L, N, N), generator=gen)]
    return stack.to(dev)[:, l]


def _sign_bytes(d):
    return torch.where(d > 0, PLUS, torch.where(d < 0, MINUS, 0)).to(torch.uint8)


def _negate(c):
    return torch.where(c == PLUS, MINUS, torch.where(c == MINUS, PLUS, 0)).to(torch.uint8)


def _oracle(qkv, d_out, H, G):
    """fp64 on the device: (d_qkv [B,N,3E], row 0 of dP [B,H,N])."""
    dqkv, dP = _orc().attention_core_backward(qkv.double(), H, SCALE, d_out.double(), None if G is None else G.double())
    return dqkv, dP[:, :, 0, :]


def _errors(d_qkv, g_row0, ref, ref_row0, H):
    """Scale-normalised errors of dQ, dK, dV, of dQ's query row 0 and of its other rows each on their own scale (with the
    training weights w_cls = (N-1) w_aff, row 0 sets the max over all rows: a wrong w_cls, or lost precision in the other rows,
    hides under it), and of g_row0."""
    B, N, _ = d_qkv.shape
    got, exp = d_qkv.reshape(B, N, 3, H * D), ref.reshape(B, N, 3, H * D)
    e = {name: _rel(got[:, :, s], exp[:, :, s]) for s, name in enumerate("qkv")}
    e["q_row0"] = _rel(got[:, 0, 0], exp[:, 0, 0])
    e["q_rows"] = _rel(got[:, 1:, 0], exp[:, 1:, 0]) if N > 1 else 0.0
    e["g_row0"] = _rel(g_row0, ref_row0)
    return e


def _assert_close(e, what):
    assert all(e[k] < TOL[k] for k in TOL), (what, e)


# ------------------------------------------------------------------ (a) the sign codes themselves
CONS_CASES = [(1, 1, 1), (2, 3, 5), (1, 2, 16), (2, 2, 28), (8, 12, 28), (1, 1, 32)]


@pytest.mark.parametrize("layout", ["separate", "one_buffer", "swapped"])
@pytest.mark.parametrize("B,L,p", CONS_CASES)
def test_consistency_sign_codes_are_exact(dev, B, L, p, layout):
    """The code bytes are sign(a1 - a2[pi][:, pi]) exactly (the sign of an fp32 difference is exact), view 2's are the permuted
    negation, column 0 and the row padding are 0x00, and every byte of every row is written: in separate buffers (with a row
    stride beyond N's 128-byte padding), as the two halves of one [2B,L,N,ld] buffer, and with the halves swapped."""
    orc = _orc()
    N = p * p + 1
    g = torch.Generator(device=dev).manual_seed(1000 * B + 10 * L + p)
    a1 = torch.softmax(torch.randn(B, L, N, N, device=dev, generator=g) * 2, -1)
    a2 = torch.softmax(torch.randn(B, L, N, N, device=dev, generator=g) * 2, -1)
    pi = orc.flip_perm(p).to(dev)
    a2[0, 0, 0, 1:] = a1[0, 0, 0, pi[1:]]                  # exact ties on a cls row ...
    a2[-1, -1, int(pi[N - 1])] = a1[-1, -1, N - 1, pi]     # ... and on an affinity row: sign(0) = 0 must survive
    ld = _rup(N, 128) + (128 if layout == "separate" else 0)
    if layout == "separate":
        c1 = torch.full((B, L, N, ld), PAD, dtype=torch.uint8, device=dev)
        c2 = torch.full((B, L, N, ld), PAD, dtype=torch.uint8, device=dev)
        bufs = (c1, c2)
    else:
        c = torch.full((2 * B, L, N, ld), PAD, dtype=torch.uint8, device=dev)
        c1, c2 = (c[B:], c[:B]) if layout == "swapped" else (c[:B], c[B:])
        bufs = (c,)
    loss_codes = _consistency(a1, a2, p, c1=c1, c2=c2, c_ld=ld)
    for buf in bufs:
        assert not bool((buf == PAD).any()), "a byte of [0, ld) was not written"
    d = a1 - a2[:, :, pi][:, :, :, pi]
    e1 = _sign_bytes(d)
    e1[..., 0] = 0
    assert bool((e1[0, 0, 0, 1:] == 0).all()) and bool((e1[-1, -1, N - 1, 1:] == 0).all())      # the ties are there
    e2 = _negate(e1)[:, :, pi][:, :, :, pi]
    assert torch.equal(c1[..., :N], e1)
    assert torch.equal(c2[..., :N], e2)
    for c_ in (c1, c2):
        assert not bool(c_[..., 0].any()) and not bool(c_[..., N:].any())        # column 0 and the padding: no gradient
    # loss2 against the closed form (fp64 means); the small cases also through the oracle's own gradient signs
    if B * L * N * N <= 1 << 22:
        cls, aff, g1, _ = orc.consistency_loss_closed_form(a1.double().cpu(), a2.double().cpu(), p, 1.0, 1.0)
        assert torch.equal(torch.sign(g1), torch.sign(_decode(c1.cpu(), N, 1.0, 1.0)))
        cls, aff = float(cls), float(aff)
    else:
        cls, aff = float(d[:, :, 0, 1:].double().abs().mean()), float(d[:, :, 1:, 1:].double().abs().mean())
    assert abs(float(loss_codes[0]) - cls) <= 1e-5 * cls + 1e-12
    assert abs(float(loss_codes[1]) - aff) <= 1e-5 * aff + 1e-12
    # the per-CTA partials are summed in the same order whatever the kernel writes: the loss is bitwise the same
    loss_only = _consistency(a1, a2, p)
    g1 = torch.empty(B, L, N, N, device=dev)
    g2 = torch.empty(B, L, N, N, device=dev)
    loss_dense = _consistency(a1, a2, p, g1=g1, g2=g2, g_ld=N)
    assert torch.equal(loss_only, loss_codes) and torch.equal(loss_dense, loss_codes)


# ------------------------------------------------------------------ (b) one G, five layouts
LAYOUT_SHAPES = [(1, 26, 3), (1, 128, 1), (2, 129, 3), (1, 257, 16), (2, 785, 12), (3, 1025, 12)]


@pytest.mark.parametrize("B,N,H", LAYOUT_SHAPES)
def test_one_gradient_in_five_layouts_is_bitwise_identical(dev, B, N, H):
    """G = +-w (w_cls = 2^-10 on row 0, w_aff = 2^-20 elsewhere) times a device scale of 0.5, handed over as contiguous rows,
    as slot l of a [B,L,N,Np] stack (Np = N padded to 4: 128-bit loads), at a base offset by 4 bytes, with a row stride of
    N + 64, and as sign codes with ld = N padded to 128 and with a larger ld.  With power-of-two weights and scale, the dense
    value g times 1/H and the code's 0.5 times 2*w*scale/H are the same exact product, fed into the same fma in the delta
    pre-pass and in the tile body: d_qkv and g_row0 must be bitwise identical."""
    from acr_wsss_b200 import ops
    qkv, d_out, gen = _inputs(dev, B, N, H, seed=11 * N + H)
    out, lse = _forward(qkv, H)
    w_cls, w_aff, sc = 2.0 ** -10, 2.0 ** -20, 0.5
    g_scale = torch.full((1,), sc, device=dev)
    L, l = 3, 1
    codes = _random_codes(gen, B, N, dev, L=L, l=l)
    G = _decode(codes, N, w_cls, w_aff, sc).float()                                 # exact in fp32
    assert torch.equal(ops.decode_sign_codes(codes, N, w_cls, w_aff, g_scale), G)
    Np = _rup(N, 4)
    stack = torch.zeros(B, L, N, Np, device=dev)
    stack[:, l, :, :N] = G
    flat = torch.zeros(B * N * Np + 4, device=dev)
    shifted = flat[1:1 + B * N * Np].view(B, N, Np)[..., :N]
    shifted.copy_(G)
    assert shifted.data_ptr() % 16 == 4
    wide = torch.zeros(B, N, N + 64, device=dev)
    wide[..., :N] = G
    codes_wide = torch.zeros(B, L, N, _rup(N, 128) + 256, dtype=torch.uint8, device=dev)
    codes_wide[:, l, :, :N] = codes[..., :N]
    ref = _backward(qkv, out, lse, d_out, H, g=G.contiguous())
    forms = {
        "padded stack slot": dict(g=stack[:, l, :, :N]),
        "base + 4 bytes": dict(g=shifted),
        "row stride N + 64": dict(g=wide[..., :N]),
        "codes, ld = roundup(N, 128)": dict(code=codes, w=(w_cls, w_aff), g_scale=g_scale),
        "codes, ld = roundup(N, 128) + 256": dict(code=codes_wide[:, l], w=(w_cls, w_aff), g_scale=g_scale),
    }
    assert bool(torch.isfinite(ref[0].float()).all()) and bool(torch.isfinite(ref[1]).all())
    for name, kw in forms.items():
        got = _backward(qkv, out, lse, d_out, H, **kw)
        assert torch.equal(got[0], ref[0]), name
        assert torch.equal(got[1], ref[1]), name


# ------------------------------------------------------------------ (c) against the fp64 oracle
ORACLE_SHAPES = [(1, 1, 1), (2, 26, 3), (1, 128, 16), (3, 129, 3), (2, 257, 12), (2, 785, 12), (1, 1025, 16)]
MIXES = [("dO", None), ("G", "dense"), ("G", "codes"), ("dO+G", "dense"), ("dO+G", "codes")]


def _g_case(dev, gen, B, N, H, form):
    """G of the size of the dO term (dP = dO V^T is ~12 here): dense G ~ 8 H N(0,1) as slot 1 of a padded [B,3,N,Np] stack (what
    ops.consistency_fwd_bwd hands over); codes with w_cls = 32 H, w_aff = 8 H.  Returns (backward kwargs, fp64 G)."""
    if form == "dense":
        Np = _rup(N, 4)
        stack = torch.zeros(B, 3, N, Np)
        stack[:, 1, :, :N] = torch.randn(B, N, N, generator=gen) * (8.0 * H)
        g = stack.to(dev)[:, 1, :, :N]
        return dict(g=g), g.double()
    codes = _random_codes(gen, B, N, dev)
    w = (32.0 * H, 8.0 * H)
    return dict(code=codes, w=w), _decode(codes, N, *w)


@pytest.mark.parametrize("mix,form", MIXES)
@pytest.mark.parametrize("B,N,H", ORACLE_SHAPES)
def test_backward_vs_fp64_oracle(dev, B, N, H, mix, form):
    """dO only, G only (d_out = 0, so an error in G is not hidden under the dO term; dV must then be exactly zero) and both,
    with G dense or as random sign codes (which also put nonzero bytes in column 0: the kernel must treat them as a general G)."""
    qkv, d_out, gen = _inputs(dev, B, N, H, seed=7 * N + 3 * H + B)
    if mix == "G":
        d_out = torch.zeros_like(d_out)
    out, lse = _forward(qkv, H)
    kw, G = _g_case(dev, gen, B, N, H, form) if form is not None else ({}, None)
    d_qkv, g_row0 = _backward(qkv, out, lse, d_out, H, **kw)
    ref, ref_row0 = _oracle(qkv, d_out, H, G)
    e = _errors(d_qkv, g_row0, ref, ref_row0, H)
    if N == 1:
        # one key: P = 1, so dS = P (dP - delta) = 0 and dQ, dK are the rounding residue of dP - delta, which the fp64 oracle
        # does not have.  Measure them against the size dS K * scale would have without that cancellation.
        size = float(ref_row0.abs().max()) * float(qkv.float().abs().max()) * SCALE
        got = d_qkv.reshape(B, N, 3, H * D).float()
        e["q"] = e["q_row0"] = float(got[:, :, 0].abs().max()) / size
        e["k"] = float(got[:, :, 1].abs().max()) / size
    _assert_close(e, (mix, form))
    if mix == "G":
        assert not bool(d_qkv.reshape(B, N, 3, H * D)[:, :, 2].any()), "dV = P^T dO must be exactly zero without dO"


# ------------------------------------------------------------------ (d) the row padding of the codes is never read
@pytest.mark.parametrize("B,N,H", [(2, 785, 12), (1, 257, 3)])
def test_code_row_padding_is_not_read(dev, B, N, H):
    """Every padding byte [N, ld) set to 0x7F (which decodes to ~1.7e38) must not change a bit of the result, in the delta
    pre-pass or in the tile body.  (Query rows past N read the clamped row N-1, which is a valid row.)"""
    qkv, d_out, gen = _inputs(dev, B, N, H, seed=N + 5)
    out, lse = _forward(qkv, H)
    codes = _random_codes(gen, B, N, dev, extra_ld=128)
    w = (0.75, 0.125)
    clean = _backward(qkv, out, lse, d_out, H, code=codes, w=w)
    dirty_codes = codes.clone()
    dirty_codes[..., N:] = PAD
    dirty = _backward(qkv, out, lse, d_out, H, code=dirty_codes, w=w)
    assert bool(torch.isfinite(clean[0].float()).all())
    assert torch.equal(clean[0], dirty[0]) and torch.equal(clean[1], dirty[1])


# ------------------------------------------------------------------ (e) magnitude: dQ's 64-bit fixed point (resolution 2^-40)
def test_code_gradient_at_production_weights(dev):
    """The training step's affinity gradient alone: B = 8, L = 12, N = 785, alpha = 100, so w_aff = alpha / (B L (N-1)^2) ~ 1.7e-6
    and dQ is ~1e-9.  dQ is summed over key tiles in fixed point with resolution 2^-40 (~9e-13): the result must still match
    the fp64 oracle at the bf16 tolerance."""
    B, L, N, H, alpha = 8, 12, 785, 12, 100.0
    qkv, d_out, gen = _inputs(dev, B, N, H, seed=785)
    d_out = torch.zeros_like(d_out)
    out, lse = _forward(qkv, H)
    codes = _random_codes(gen, B, N, dev, L=L, l=5)
    w = (alpha / (B * L * (N - 1)), alpha / (B * L * float(N - 1) ** 2))
    one = torch.ones(1, device=dev)
    d_qkv, g_row0 = _backward(qkv, out, lse, d_out, H, code=codes, w=w, g_scale=one)
    ref, ref_row0 = _oracle(qkv, d_out, H, _decode(codes, N, *w))
    e = _errors(d_qkv, g_row0, ref, ref_row0, H)
    dq = d_qkv.reshape(B, N, 3, H, D)[:, :, 0].double()
    dq_ref = ref.reshape(B, N, 3, H, D)[:, :, 0]
    row_max = dq_ref.abs().amax(-1)
    row_err = (dq - dq_ref).abs().amax(-1) / row_max
    print(f"production weights w_cls={w[0]:.3e} w_aff={w[1]:.3e}: row-max |dQ| of query row 0 {float(row_max[:, 0].min()):.3e} .. "
          f"{float(row_max[:, 0].max()):.3e}, of the other rows {float(row_max[:, 1:].min()):.3e} .. {float(row_max[:, 1:].max()):.3e}; "
          f"worst error of a row on its own scale {float(row_err.max()):.3e}; errors {e}")
    _assert_close(e, "production weights")


def test_fixed_point_dq_scale_sweep(dev):
    """dO and G both scaled by s in {1, 2^-8, 2^-16} (O(1) inputs at s = 1): dQ(s) / s stays within tolerance of dQ(1) and of
    the oracle, so the fixed-point resolution does not eat small gradients."""
    B, N, H = 2, 785, 12
    qkv, d_out, gen = _inputs(dev, B, N, H, seed=31)
    out, lse = _forward(qkv, H)
    codes = _random_codes(gen, B, N, dev)
    w = (32.0 * H, 8.0 * H)
    ref, ref_row0 = _oracle(qkv, d_out, H, _decode(codes, N, *w))
    base = None
    for s in (1.0, 2.0 ** -8, 2.0 ** -16):
        d_qkv, g_row0 = _backward(qkv, out, lse, d_out * s, H, code=codes, w=(w[0] * s, w[1] * s))
        dqkv_s = d_qkv.double() / s
        _assert_close(_errors(dqkv_s, g_row0.double() / s, ref, ref_row0, H), s)
        dq = dqkv_s.reshape(B, N, 3, H * D)[:, :, 0]
        if base is None:
            base = dq
        assert _rel(dq, base) < BF16_TOL, s


# ------------------------------------------------------------------ (f) the checks have teeth
def test_tolerances_separate_wrong_gradients_from_rounding(dev):
    """G only, N = 785, codes: the kernel matches the oracle, and is at least 10x the tolerance away from the oracle evaluated
    with a deliberately wrong G -- the codes of key tile 3 zeroed, w_cls and w_aff swapped, the 17 tail columns dropped.  So
    these bug classes cannot pass as rounding."""
    B, N, H = 2, 785, 12
    qkv, d_out, gen = _inputs(dev, B, N, H, seed=3)
    d_out = torch.zeros_like(d_out)
    out, lse = _forward(qkv, H)
    codes = _random_codes(gen, B, N, dev)
    w = (32.0 * H, 8.0 * H)
    d_qkv, g_row0 = _backward(qkv, out, lse, d_out, H, code=codes, w=w)
    G = _decode(codes, N, *w)
    _assert_close(_errors(d_qkv, g_row0, *_oracle(qkv, d_out, H, G), H), "right G")
    tile3 = G.clone()
    tile3[..., 384:512] = 0
    no_tail = G.clone()
    no_tail[..., 768:] = 0
    wrong = {"key tile 3 zeroed": tile3, "w_cls and w_aff swapped": _decode(codes, N, w[1], w[0]), "tail columns dropped": no_tail}
    for name, Gw in wrong.items():
        e = _errors(d_qkv, g_row0, *_oracle(qkv, d_out, H, Gw), H)
        assert max(e[k] / TOL[k] for k in TOL) >= 10, (name, e)
        assert max(e[k] / TOL[k] for k in ("q", "k", "q_row0", "q_rows")) >= 10, (name, e)      # not only through g_row0 = G[0] / H


# ------------------------------------------------------------------ (g) end to end at the training shape
@pytest.mark.parametrize("swapped", [False, True])
def test_consistency_to_attention_backward_end_to_end(dev, swapped):
    """ops.attention_core (bf16) -> stack_views_split (both views as one batch of 2B) -> ops.consistency_loss at p = 28, B = 2,
    L = 2, H = 12: the leaves' qkv gradients against the fp64 chain (G of each view and block from the closed form on the
    kernels' own stacks -- signs at near-ties must come from the same maps -- times the upstream scalar, through
    attention_core_backward), and the sign-code path against the dense fallback (stacks without per-block states)."""
    from acr_wsss_b200 import ops
    orc = _orc()
    B, L, p, H, alpha, upstream = 2, 2, 28, 12, 100.0, 0.5
    N = p * p + 1
    gen = torch.Generator().manual_seed(28)
    qkvs = [(torch.randn(2 * B, N, 3 * H * D, generator=gen) * 1.5).to(torch.bfloat16).to(dev) for _ in range(L)]

    def run(compact):
        leaves = [q.clone().requires_grad_(True) for q in qkvs]
        stack = torch.empty(2 * B, L, N, N, device=dev)
        maps, states = [], []
        for l in range(L):
            st = {"capture_grad": False}
            _, m = ops.attention_core(leaves[l], H, SCALE, stack[:, l], st, "bf16")
            maps.append(m)
            states.append(st)
        a1, a2 = ops.stack_views_split(stack, maps, states if compact else None)
        total, loss2 = ops.consistency_loss(a2, a1, p, alpha) if swapped else ops.consistency_loss(a1, a2, p, alpha)
        (upstream * total).backward()
        return a1.detach(), a2.detach(), loss2, [q.grad for q in leaves]

    a1, a2, loss2, grads = run(True)
    first, second = (a2, a1) if swapped else (a1, a2)
    cls, aff, g_first, g_second = orc.consistency_loss_closed_form(first.cpu(), second.cpu(), p, alpha, alpha)
    assert abs(float(loss2[0]) - float(cls)) <= 1e-5 * float(cls) and abs(float(loss2[1]) - float(aff)) <= 1e-5 * float(aff)
    g_a1, g_a2 = (g_second, g_first) if swapped else (g_first, g_second)
    G = torch.cat([g_a1, g_a2], 0).to(dev).double() * upstream        # [2B,L,N,N]: the batch holds view 1, then view 2
    zeros = torch.zeros(2 * B, N, H * D, device=dev)
    for l in range(L):
        ref, _ = _orc().attention_core_backward(qkvs[l].double(), H, SCALE, zeros.double(), G[:, l])
        got = grads[l].reshape(2 * B, N, 3, H * D)
        exp = ref.reshape(2 * B, N, 3, H * D)
        e = {"q": _rel(got[:, :, 0], exp[:, :, 0]), "k": _rel(got[:, :, 1], exp[:, :, 1]), "q_row0": _rel(got[:, 0, 0], exp[:, 0, 0]),
             "q_rows": _rel(got[:, 1:, 0], exp[:, 1:, 0])}
        assert all(e[k] < TOL[k] for k in e), (l, e)
        assert not bool(got[:, :, 2].any())
    _, _, loss2_dense, grads_dense = run(False)
    assert torch.equal(loss2, loss2_dense)
    for x, y in zip(grads, grads_dense):
        assert _rel(x, y) < 2e-3


# ------------------------------------------------------------------ (h) determinism in code mode
def test_code_mode_backward_is_identical_run_to_run(dev):
    B, N, H = 2, 785, 12
    qkv, d_out, gen = _inputs(dev, B, N, H, seed=8)
    out, lse = _forward(qkv, H)
    codes = _random_codes(gen, B, N, dev)
    g_scale = torch.full((1,), 0.37, device=dev)
    runs = [_backward(qkv, out, lse, d_out, H, code=codes, w=(3.0, 0.7), g_scale=g_scale) for _ in range(3)]
    for d_qkv, g_row0 in runs[1:]:
        assert torch.equal(d_qkv, runs[0][0]) and torch.equal(g_row0, runs[0][1])
