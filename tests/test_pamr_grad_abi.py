"""CPU tier: acr_pamr_fwd_save and acr_pamr_bwd (csrc/pamr.cu) reject every invalid argument before they touch the device."""
import ctypes

from acr_wsss_b200 import _lib

B, K, C, H, W, MH, MW, T = 2, 3, 21, 448, 448, 28, 28, 10
DIL = [1, 2, 4, 8, 12, 24]
BIG = 1 << 62                                                      # a buffer size that passes every size check


def _dev():
    buf = ctypes.create_string_buffer(4096)
    return buf, ctypes.c_void_p((ctypes.addressof(buf) + 255) & ~255)


def _dil(d):
    return (ctypes.c_int * max(len(d), 1))(*d) if d is not None else None


def _save_call(**over):
    """acr_pamr_fwd_save on fake device addresses that are never dereferenced, with `over` replaced."""
    keep, dev = _dev()
    a = dict(x=dev, mask=dev, B=B, K=K, C=C, H=H, W=W, mh=MH, mw=MW, dil=DIL, nd=None, num_iter=T, out=dev, saved=dev,
             saved_bytes=None)
    a.update(over)
    nd = len(a["dil"]) if a["nd"] is None else a["nd"]
    if a["saved_bytes"] is None:
        a["saved_bytes"] = _lib.lib().acr_pamr_save_workspace(B, K, C, H, W, len(DIL), T)
    return _lib.lib().acr_pamr_fwd_save(a["x"], a["mask"], a["B"], a["K"], a["C"], a["H"], a["W"], a["mh"], a["mw"],
                                        _dil(a["dil"]), nd, a["num_iter"], a["out"], a["saved"], a["saved_bytes"], None)


def _bwd_call(**over):
    keep, dev = _dev()
    a = dict(x=dev, saved=dev, saved_bytes=None, g=dev, B=B, K=K, C=C, H=H, W=W, mh=MH, mw=MW, dil=DIL, nd=None, num_iter=T,
             d_x=dev, d_mask=dev, ws=dev, ws_bytes=None)
    a.update(over)
    nd = len(a["dil"]) if a["nd"] is None else a["nd"]
    if a["saved_bytes"] is None:
        a["saved_bytes"] = _lib.lib().acr_pamr_save_workspace(B, K, C, H, W, len(DIL), T)
    if a["ws_bytes"] is None:
        a["ws_bytes"] = _lib.lib().acr_pamr_bwd_workspace(B, K, C, H, W, len(DIL))
    return _lib.lib().acr_pamr_bwd(a["x"], a["saved"], a["saved_bytes"], a["g"], a["B"], a["K"], a["C"], a["H"], a["W"],
                                   a["mh"], a["mw"], _dil(a["dil"]), nd, a["num_iter"], a["d_x"], a["d_mask"], a["ws"],
                                   a["ws_bytes"], None)


COMMON_BAD = {
    "B 0": dict(B=0), "K 0": dict(K=0), "C < 0": dict(C=-1), "H 0": dict(H=0), "W 0": dict(W=0), "mh 0": dict(mh=0),
    "mw < 0": dict(mw=-2),
    "nd 0": dict(dil=[], nd=0), "nd 9": dict(dil=[1] * 9), "dilation 0": dict(dil=[1, 0, 2]), "dilation < 0": dict(dil=[-1]),
    "num_iter < 0": dict(num_iter=-1),
    "null dilations": dict(dil=None, nd=1),
}
GRID_BAD = {"H > 65535": dict(H=65536, W=4), "B*C > 65535": dict(B=3, C=21846)}


def test_pamr_fwd_save_rejects_invalid_arguments_before_any_launch():
    L = _lib.lib()
    bad = dict(COMMON_BAD)
    bad.update({"null x": dict(x=None), "null mask": dict(mask=None), "null out": dict(out=None), "null saved": dict(saved=None)})
    bad.update({k: dict(v, saved_bytes=BIG) for k, v in GRID_BAD.items()})
    for what, over in bad.items():
        assert _save_call(**over) == -1, what
        assert L.acr_last_error_string().startswith(b"acr_pamr_fwd_save"), what
    need = L.acr_pamr_save_workspace(B, K, C, H, W, len(DIL), T)
    assert _save_call(saved_bytes=need - 1) == -4


def test_pamr_bwd_rejects_invalid_arguments_before_any_launch():
    L = _lib.lib()
    bad = dict(COMMON_BAD)
    bad.update({"null x": dict(x=None), "null saved": dict(saved=None), "null g_out": dict(g=None),
                "null workspace": dict(ws=None), "neither gradient": dict(d_x=None, d_mask=None)})
    bad.update({k: dict(v, saved_bytes=BIG, ws_bytes=BIG) for k, v in GRID_BAD.items()})
    bad["B*C*mh*mw >= 2^31"] = dict(mh=32768, mw=32768, saved_bytes=BIG, ws_bytes=BIG)
    for what, over in bad.items():
        assert _bwd_call(**over) == -1, what
        assert L.acr_last_error_string().startswith(b"acr_pamr_bwd"), what
    assert _bwd_call(ws_bytes=L.acr_pamr_bwd_workspace(B, K, C, H, W, len(DIL)) - 1) == -4
    assert _bwd_call(saved_bytes=L.acr_pamr_save_workspace(B, K, C, H, W, len(DIL), T) - 1) == -4
    # the saved state of a longer forward is fine, of a shorter one is not
    assert _bwd_call(num_iter=T + 1) == -4


def test_pamr_grad_workspaces():
    L = _lib.lib()
    # the weights, then one padded iterate per iteration (the forward's workspace holds the weights and two of them)
    wgt = L.acr_pamr_save_workspace(1, 3, 21, 448, 448, 6, 0)
    slot = L.acr_pamr_save_workspace(1, 3, 21, 448, 448, 6, 1) - wgt
    assert wgt > 0 and slot > 0 and slot % 256 == 0
    assert L.acr_pamr_save_workspace(1, 3, 21, 448, 448, 6, 10) == wgt + 10 * slot
    assert L.acr_pamr_workspace(1, 3, 21, 448, 448, 6) == wgt + 2 * slot
    assert L.acr_pamr_save_workspace(1, 3, 21, 448, 448, 6, -1) == 0
    assert L.acr_pamr_save_workspace(0, 3, 21, 448, 448, 6, 10) == 0
    bwd = L.acr_pamr_bwd_workspace(1, 3, 21, 448, 448, 6)
    assert bwd > 0 and bwd % 256 == 0
    assert L.acr_pamr_bwd_workspace(1, 3, 21, 448, 0, 6) == 0
