"""CPU tier: acr_attn_fwd_bf16 (csrc/attn_tc.cu) and acr_attn_fwd_f32 (csrc/attn_f32.cu) reject invalid arguments before any
device work.  The addresses are fake and never dereferenced.  A valid bf16 call must stop at the sm_100 check on a machine
without such a device; where one is present the valid calls are not made, because they would launch on the fake addresses."""
import ctypes

from acr_wsss_b200 import _lib

B, N, H, D = 2, 785, 12, 64


def _fake():
    buf = ctypes.create_string_buffer(4096)
    return buf, (ctypes.addressof(buf) + 255) & ~255


def _no_sm100():
    return not _lib.lib().acr_device_is_sm100()


def _fwd(**over):
    keep, a = _fake()
    lib = _lib.lib()
    x = dict(qkv=a, B=B, N=N, H=H, D=D, out=a, lse=a, mean=a, mbs=3 * N * N, row0=a)
    x.update(over)
    rc = lib.acr_attn_fwd_bf16(x["qkv"], x["B"], x["N"], x["H"], x["D"], 0.125, x["out"], x["lse"], x["mean"], x["mbs"], x["row0"], None)
    del keep
    return rc, lib.acr_last_error_string().decode()


def test_attn_fwd_bf16_rejects_invalid_arguments_before_any_launch():
    _, a = _fake()
    bad = {
        "null qkv": (dict(qkv=None), -1), "null out": (dict(out=None), -1), "null lse": (dict(lse=None), -1),
        "B 0": (dict(B=0), -1), "B -1": (dict(B=-1), -1), "N 0": (dict(N=0), -1), "H 0": (dict(H=0), -1),
        "D 32": (dict(D=32), -1), "D 128": (dict(D=128), -1), "H 33": (dict(H=33), -1), "B 65536": (dict(B=65536), -1),
        "qkv misaligned by 2": (dict(qkv=a + 2), -2), "qkv misaligned by 8": (dict(qkv=a + 8), -2),
        "out misaligned by 8": (dict(out=a + 8), -2),
        "p_row0 without attn_mean": (dict(mean=None, mbs=0), -1),
        "mean stride N*N - 1": (dict(mbs=N * N - 1), -1), "mean stride 0": (dict(mbs=0), -1),
        "mean stride N": (dict(mbs=N), -1), "mean stride -N*N": (dict(mbs=-N * N), -1),
        "mean stride -1 at B 1": (dict(B=1, mbs=-1), -1),
    }
    for what, (over, code) in bad.items():
        rc, err = _fwd(**over)
        assert rc == code, (what, rc, err)
        assert err.startswith("acr_attn_fwd_bf16"), (what, err)
    rc, err = _fwd(mbs=N * N - 1)
    assert "mean_batch_stride" in err, err


def test_attn_fwd_bf16_valid_calls_reach_the_device_check():
    """Every stride rule's boundary on the accepting side: N*N (dense [B,N,N]), L*N*N (slot of a [B,L,N,N] stack), any stride
    for one image, any stride without a map; H = 32 and B = 65535 are the largest accepted."""
    if not _no_sm100():
        return
    for over in (dict(), dict(mbs=N * N), dict(B=1, mbs=0), dict(B=1, mbs=5), dict(mean=None, row0=None, mbs=-7),
                 dict(mean=None, row0=None, mbs=0), dict(row0=None), dict(H=32), dict(B=65535), dict(N=1, H=1, mbs=1)):
        rc, err = _fwd(**over)
        assert rc == -3, (over, rc, err)
        assert err.startswith("acr_attn_fwd_bf16"), (over, err)


def test_attn_fwd_f32_rejects_overlapping_mean_maps():
    """The exact path writes the same head-mean layout and follows the same stride rule (checked before its first launch)."""
    keep, a = _fake()
    lib = _lib.lib()
    for mbs in (N * N - 1, 0, -N * N):
        rc = lib.acr_attn_fwd_f32(a, B, N, H, D, 0.125, a, a, a, mbs, None)
        assert rc == -1, (mbs, rc)
        err = lib.acr_last_error_string().decode()
        assert err.startswith("acr_attn_fwd_f32") and "mean_batch_stride" in err, (mbs, err)
    rc = lib.acr_attn_fwd_f32(a, 1, N, H, D, 0.125, a, a, a, -1, None)
    assert rc == -1
    del keep
