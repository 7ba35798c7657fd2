"""CPU tier: acr_cam_finish (batched CAM finish, csrc/cam_finish.cu) rejects every invalid argument before it touches the device."""
import ctypes

from acr_wsss_b200 import _lib

M, N_COPIES, C = 2, 3, 20


def _args(**over):
    """A valid call (2 images, 2 scales, 4 planes) on fake device addresses that are never dereferenced, with `over` replaced."""
    buf = ctypes.create_string_buffer(4096)
    dev = ctypes.c_void_p((ctypes.addressof(buf) + 255) & ~255)
    a = dict(cams=[dev, dev], patch=[dev, dev], grid=[7, 7, 14, 14], ns=2, M=M, n=N_COPIES, C=C, labels=dev,
             planes=[[0, 0, 2, 0, 375, 500], [187500, 0, 14, 1, 375, 500], [375000, 1, 0, 0, 1, 7], [375007, 1, 5, 1, 17, 1]],
             num_planes=None, out=dev, out_elems=375024, ws=dev, ws_bytes=4 * 48)
    a.update(over)
    a["_keep"] = buf
    return a


def _call(a):
    L = _lib.lib()
    ptrs = lambda v: None if v is None else (ctypes.c_void_p * max(1, len(v)))(*v)
    grid = None if a["grid"] is None else (ctypes.c_int * len(a["grid"]))(*a["grid"])
    flat = None if a["planes"] is None else [x for p in a["planes"] for x in p]
    table = None if flat is None else (ctypes.c_longlong * max(1, len(flat)))(*flat)
    npl = a["num_planes"] if a["num_planes"] is not None else (len(a["planes"]) if a["planes"] is not None else 1)
    return L.acr_cam_finish(ptrs(a["cams"]), ptrs(a["patch"]), grid, a["ns"], a["M"], a["n"], a["C"], a["labels"], table, npl,
                            a["out"], a["out_elems"], a["ws"], a["ws_bytes"], None)


def _plane(i, **kw):
    p = list(_args()["planes"])
    row = list(p[i])
    for k, v in kw.items():
        row[["offset", "image", "channel", "kind", "rows", "cols"].index(k)] = v
    p[i] = row
    return p


def test_cam_finish_rejects_invalid_arguments_before_any_launch():
    bad = {
        "null cams": dict(cams=None), "null patch": dict(patch=None), "null grid": dict(grid=None), "null labels": dict(labels=None),
        "null map of a scale": dict(cams=[_args()["labels"], None]),
        "no scale": dict(ns=0), "9 scales": dict(ns=9),
        "M < 1": dict(M=0), "n < 1": dict(n=0), "C < 1": dict(C=0),
        "grid rows 0": dict(grid=[7, 7, 0, 14]), "grid cols < 0": dict(grid=[7, -1, 14, 14]),
        "negative plane count": dict(num_planes=-1),
        "null table": dict(planes=None, num_planes=4), "null out": dict(out=None), "null workspace": dict(ws=None),
        "rows 0": dict(planes=_plane(0, rows=0)), "cols < 0": dict(planes=_plane(2, cols=-7)),
        "negative offset": dict(planes=_plane(1, offset=-1)),
        "plane past the end": dict(planes=_plane(3, offset=375008)),
        "offset past the end": dict(planes=_plane(3, offset=1 << 40)),
        "rows*cols overflows": dict(planes=_plane(0, rows=1 << 31, cols=1 << 31)),
        "image out of range": dict(planes=_plane(1, image=M)), "unknown kind": dict(planes=_plane(1, kind=2)),
        "GETAM copy >= n": dict(planes=_plane(0, channel=N_COPIES)), "patch class >= C": dict(planes=_plane(1, channel=C)),
        "negative channel": dict(planes=_plane(2, channel=-1)),
    }
    L = _lib.lib()
    for what, over in bad.items():
        assert _call(_args(**over)) == -1, what
        assert L.acr_last_error_string().startswith(b"acr_cam_finish"), what
    assert _call(_args(ws_bytes=4 * 48 - 1)) == -4                       # workspace holds the table copy
    a = _args()
    assert _call(_args(ws=ctypes.c_void_p(a["ws"].value + 4))) == -2       # 8-byte aligned table copy


def test_cam_finish_zero_planes_launches_nothing():
    assert _call(_args(planes=[], out=None, ws=None, ws_bytes=0, out_elems=0)) == 0
