"""CPU tier: acr_dense_crf (csrc/densecrf.cu) rejects every invalid argument before it touches the device."""
import ctypes
import math

from acr_wsss_b200 import _lib

N, C, H, W = 2, 21, 375, 500


def _args(**over):
    """A valid call on fake device addresses that are never dereferenced, with `over` replaced."""
    buf = ctypes.create_string_buffer(4096)
    dev = ctypes.c_void_p((ctypes.addressof(buf) + 255) & ~255)
    a = dict(images=dev, probs=dev, q=dev, N=N, C=C, H=H, W=W, n_iter=10, sxy_g=3.0, compat_g=3.0, sxy_b=80.0, srgb=13.0,
             compat_b=10.0, clip=1e-5, ws=dev, ws_bytes=None)
    a.update(over)
    if a["ws_bytes"] is None:
        a["ws_bytes"] = _lib.lib().acr_dense_crf_workspace(N, C, H, W)
    a["_keep"] = buf
    return a


def _call(a):
    return _lib.lib().acr_dense_crf(a["images"], a["probs"], a["q"], a["N"], a["C"], a["H"], a["W"], a["n_iter"], a["sxy_g"],
                                    a["compat_g"], a["sxy_b"], a["srgb"], a["compat_b"], a["clip"], a["ws"], a["ws_bytes"], None)


def test_dense_crf_rejects_invalid_arguments_before_any_launch():
    nan, inf = math.nan, math.inf
    bad = {
        "null images": dict(images=None), "null probs": dict(probs=None), "null q": dict(q=None), "null workspace": dict(ws=None),
        "N 0": dict(N=0), "C 0": dict(C=0), "H 0": dict(H=0), "W < 0": dict(W=-3), "C 97": dict(C=97),
        "n_iter < 0": dict(n_iter=-1),
        "sxy_g 0": dict(sxy_g=0.0), "sxy_b < 0": dict(sxy_b=-80.0), "srgb 0": dict(srgb=0.0),
        "sxy_g nan": dict(sxy_g=nan), "sxy_b inf": dict(sxy_b=inf), "srgb nan": dict(srgb=nan),
        "compat_g nan": dict(compat_g=nan), "compat_b inf": dict(compat_b=-inf),
        "clip 0": dict(clip=0.0), "clip > 1": dict(clip=1.5), "clip < 0": dict(clip=-1e-5), "clip nan": dict(clip=nan),
        "6HW >= 2^28": dict(H=1 << 13, W=(1 << 28) // 6 // (1 << 13) + 1, sxy_g=1e4, sxy_b=1e4),
        "int16 keys overflow": dict(sxy_g=0.01),
    }
    for what, over in bad.items():
        assert _call(_args(**over)) == -1, what
        assert _lib.lib().acr_last_error_string().startswith(b"acr_dense_crf"), what
    assert _call(_args(ws_bytes=_lib.lib().acr_dense_crf_workspace(N, C, H, W) - 1)) == -4
    a = _args()
    assert _call(_args(ws=ctypes.c_void_p(a["ws"].value + 16))) == -2


def test_dense_crf_workspace():
    L = _lib.lib()
    one = L.acr_dense_crf_workspace(1, 21, 375, 500)
    assert one > 0 and one % 256 == 0
    assert L.acr_dense_crf_workspace(8, 21, 375, 500) == 8 * one
    assert L.acr_dense_crf_workspace(20, 21, 375, 500) == 8 * one          # images go through in batches of 8
    assert L.acr_dense_crf_workspace(1, 97, 375, 500) == 0
    assert L.acr_dense_crf_workspace(0, 21, 375, 500) == 0
