"""CPU tier: acr_attn_bwd_bf16 and acr_consistency_fwd_bwd reject an inconsistent form of the affinity gradient (dense and
sign codes at once, half a pair of code buffers, short or misaligned rows) before any device work.  The addresses are fake
and never dereferenced: every call below is invalid, so none of them gets as far as a launch."""
import ctypes

from acr_wsss_b200 import _lib

B, N, H, D = 2, 785, 12, 64
LD = 896                    # N padded to 128


def _fake():
    buf = ctypes.create_string_buffer(4096)
    return buf, (ctypes.addressof(buf) + 255) & ~255


def _attn_bwd(**over):
    keep, a = _fake()
    L = _lib.lib()
    x = dict(g=None, g_bs=0, g_ld=0, code=a, c_bs=3 * N * LD, c_ld=LD)
    x.update(over)
    rc = L.acr_attn_bwd_bf16(a, a, a, a, B, N, H, D, 0.125, x["g"], x["g_bs"], x["g_ld"], x["code"], x["c_bs"], x["c_ld"],
                             1.0, 1.0, None, a, None, a, L.acr_attn_bwd_bf16_workspace(B, N, H, D), None)
    del keep
    return rc, L.acr_last_error_string().decode()


def _consistency(**over):
    keep, a = _fake()
    L = _lib.lib()
    x = dict(N=26, p=5, g1=None, g2=None, g_ld=0, c1=a, c2=a, c_ld=128)
    x.update(over)
    rc = L.acr_consistency_fwd_bwd(a, a, 2, 3, x["N"], x["p"], 1.0, 1.0, a, x["g1"], x["g2"], x["g_ld"], x["c1"], x["c2"], x["c_ld"],
                                   a, L.acr_consistency_workspace(2, 3, 26), None)
    del keep
    return rc, L.acr_last_error_string().decode()


def test_attn_bwd_rejects_inconsistent_gradient_forms():
    _, a = _fake()
    bad = {
        "dense and codes": (dict(g=a, g_bs=N * N, g_ld=N), -1, "g_mean OR g_code"),
        "dense row stride < N": (dict(g=a, g_bs=N * N, g_ld=N - 1, code=None), -1, "g_row_stride < N"),
        "code row stride 100": (dict(c_ld=100), -2, "g_code rows"),
        "code row stride 768 < 896": (dict(c_ld=768, c_bs=3 * N * 768), -2, "g_code rows"),
        "code base misaligned by 4": (dict(code=a + 4), -2, "g_code rows"),
        "code batch stride 8 mod 16": (dict(c_bs=3 * N * LD + 8), -2, "g_code rows"),
    }
    for what, (over, code, msg) in bad.items():
        rc, err = _attn_bwd(**over)
        assert rc == code, (what, rc, err)
        assert err.startswith("acr_attn_bwd_bf16") and msg in err, (what, err)


def test_consistency_rejects_inconsistent_gradient_forms():
    _, a = _fake()
    bad = {
        "dense and codes": (dict(g1=a, g2=a, g_ld=26), "dense gradients OR sign codes"),
        "code1 only": (dict(c2=None), "code1/code2"),
        "code2 only": (dict(c1=None), "code1/code2"),
        "code row stride < N": (dict(c_ld=25), "code_row_stride < N"),
        "N != p*p + 1": (dict(N=27), "is not p*p+1"),
    }
    for what, (over, msg) in bad.items():
        rc, err = _consistency(**over)
        assert rc == -1, (what, rc, err)
        assert err.startswith("acr_consistency_fwd_bwd") and msg in err, (what, err)
