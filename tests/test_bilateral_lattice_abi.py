"""CPU tier: acr_bilateral_batch (csrc/bilateral.cu) rejects invalid arguments before it touches the device, its workspace
covers one batch chunk of 8 images whatever N is, and the oracle's vertex-count door agrees with a hand count."""
import ctypes

import numpy as np

from acr_wsss_b200 import _lib
from oracle import bilateral_oracle as bo

N, K, H, W = 9, 21, 33, 31


def _call(**over):
    """A valid call on fake device addresses that are never dereferenced, with `over` replaced."""
    buf = ctypes.create_string_buffer(4096)
    dev = ctypes.c_void_p((ctypes.addressof(buf) + 255) & ~255)
    a = dict(images=dev, ins=dev, outs=dev, N=N, K=K, H=H, W=W, srgb=15.0, sxy=50.0, ws=dev, ws_bytes=None)
    a.update(over)
    if a["ws_bytes"] is None:
        a["ws_bytes"] = _lib.lib().acr_bilateral_workspace(a["N"], a["K"], a["H"], a["W"])
    return _lib.lib().acr_bilateral_batch(a["images"], a["ins"], a["outs"], a["N"], a["K"], a["H"], a["W"], a["srgb"], a["sxy"],
                                          a["ws"], a["ws_bytes"], None, None)


def test_bilateral_rejects_97_planes_before_any_launch():
    """K <= 96: the slice's output tile of 128 pixels x K planes must fit 48 KB of shared memory."""
    assert _call(K=97) == -1
    err = _lib.lib().acr_last_error_string()
    assert err.startswith(b"acr_bilateral_batch") and b"K=97" in err, err


def test_bilateral_rejects_bad_buffers():
    for what, over in {"null images": dict(images=None), "null ins": dict(ins=None), "null outs": dict(outs=None),
                       "null workspace": dict(ws=None), "N 0": dict(N=0), "K 0": dict(K=0), "sxy 0": dict(sxy=0.0)}.items():
        assert _call(**over) == -1, what
    buf = ctypes.create_string_buffer(4096)
    base = (ctypes.addressof(buf) + 255) & ~255
    for off in (4, 16, 128):
        assert _call(ws=ctypes.c_void_p(base + off)) == -2, off
    assert _call(ws_bytes=_lib.lib().acr_bilateral_workspace(N, K, H, W) - 1) == -4


def test_bilateral_workspace_is_one_chunk_of_8_images():
    L = _lib.lib()
    one = L.acr_bilateral_workspace(1, K, H, W)
    assert one > 0 and one % 256 == 0
    assert L.acr_bilateral_workspace(8, K, H, W) == 8 * one
    for n in (9, 16, 17, 100):
        assert L.acr_bilateral_workspace(n, K, H, W) == L.acr_bilateral_workspace(8, K, H, W), n
    # value rows are K rounded up to 4 planes
    assert L.acr_bilateral_workspace(1, 81, H, W) == L.acr_bilateral_workspace(1, 84, H, W)
    assert L.acr_bilateral_workspace(0, K, H, W) == 0 and L.acr_bilateral_workspace(1, 0, H, W) == 0


def test_oracle_lattice_size_by_hand():
    """A 1 x 1 image is embedded with its three phantom pad pixels (all-zero features).  A black pixel is at the origin as
    well: one simplex, its d + 1 = 6 vertices.  A bright pixel at sigma_rgb = 1 lies far from the origin: a second,
    disjoint simplex, 12 vertices."""
    black = np.zeros((1, 3, 1, 1), np.float32)
    assert bo.oracle_lattice_sizes(black, 1.0, 1.0) == [6]
    bright = np.full((2, 3, 1, 1), 77.0, np.float32)
    assert bo.oracle_lattice_sizes(np.concatenate([black, bright]), 1.0, 1.0) == [6, 12, 12]
    # the filter is linear and the planes are independent: equal planes of a single pixel come out equal and positive
    out = bo.oracle_bilateral(black, np.full((1, 2, 1, 1), 3.0, np.float32), 1.0, 1.0)
    assert out.shape == (1, 2, 1, 1) and out[0, 0, 0, 0] == out[0, 1, 0, 0] > 0
