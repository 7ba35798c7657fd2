"""CPU tier: acr_cam_label_counts / acr_label_map_counts (pseudo-label evaluation, csrc/label_eval.cu) reject every invalid
argument with ACR_E_INVAL and a message before they touch the device.  Only invalid calls are made: the device addresses
below are fake."""
import ctypes

from acr_wsss_b200 import _lib

K = 21


def _fake():
    buf = ctypes.create_string_buffer(4096)
    return buf, ctypes.c_void_p((ctypes.addressof(buf) + 255) & ~255)


def _cam_args(**over):
    """A valid call: 2 images (375x500, 1x7), 3 planes, 100 thresholds i/100, with `over` replaced."""
    buf, dev = _fake()
    a = dict(cams=dev, cam_elems=2 * 187500 + 7, planes=[[0, 0, 14], [187500, 0, 2], [375000, 1, 19]], gt=dev,
             gt_elems=187507, images=[[0, 375, 500], [187500, 1, 7]], thresholds=[i / 100 for i in range(100)], num_cls=K,
             counts=dev, ws=dev, ws_bytes=None, num_planes=None, num_images=None, num_thresholds=None)
    a.update(over)
    a["_keep"] = buf
    return a


def _arr(ctype, rows):
    if rows is None:
        return None
    flat = [x for r in rows for x in (r if isinstance(r, (list, tuple)) else [r])]
    return (ctype * max(1, len(flat)))(*flat)


def _call_cam(a):
    L = _lib.lib()
    npl = a["num_planes"] if a["num_planes"] is not None else (len(a["planes"]) if a["planes"] is not None else 1)
    nim = a["num_images"] if a["num_images"] is not None else (len(a["images"]) if a["images"] is not None else 1)
    nth = a["num_thresholds"] if a["num_thresholds"] is not None else (len(a["thresholds"]) if a["thresholds"] is not None else 1)
    wsb = a["ws_bytes"] if a["ws_bytes"] is not None else L.acr_label_counts_workspace(max(nim, 0), max(npl, 0), max(nth, 0))
    return L.acr_cam_label_counts(a["cams"], a["cam_elems"], _arr(ctypes.c_longlong, a["planes"]), npl, a["gt"], a["gt_elems"],
                                  _arr(ctypes.c_longlong, a["images"]), nim, _arr(ctypes.c_double, a["thresholds"]), nth,
                                  a["num_cls"], a["counts"], a["ws"], wsb, None)


def _plane(i, **kw):
    p = [list(r) for r in _cam_args()["planes"]]
    for k, v in kw.items():
        p[i][["offset", "image", "cls"].index(k)] = v
    return p


def _image(i, **kw):
    p = [list(r) for r in _cam_args()["images"]]
    for k, v in kw.items():
        p[i][["offset", "rows", "cols"].index(k)] = v
    return p


def test_cam_label_counts_rejects_invalid_arguments_before_any_launch():
    thr = [i / 100 for i in range(100)]
    bad = {
        "null cams": dict(cams=None), "null planes": dict(planes=None, num_planes=3), "null gt": dict(gt=None),
        "null images": dict(images=None, num_images=2), "null thresholds": dict(thresholds=None, num_thresholds=100),
        "null counts": dict(counts=None), "null workspace": dict(ws=None),
        "num_cls 0": dict(num_cls=0), "num_cls 256": dict(num_cls=256), "num_cls -1": dict(num_cls=-1),
        "negative plane count": dict(num_planes=-1), "negative image count": dict(num_images=-1),
        "no threshold": dict(thresholds=[], num_thresholds=0), "4097 thresholds": dict(thresholds=[0.5] * 4097),
        "plane class = num_cls - 1": dict(planes=_plane(1, cls=K - 1)), "negative plane class": dict(planes=_plane(0, cls=-1)),
        "plane class >= num_cls - 1 at num_cls 1": dict(num_cls=1, planes=[[0, 0, 0]]),
        "two planes of one class": dict(planes=_plane(1, cls=14)),
        "plane image out of range": dict(planes=_plane(2, image=2)), "negative plane image": dict(planes=_plane(0, image=-1)),
        "plane past the CAM buffer": dict(planes=_plane(2, offset=375001)), "negative plane offset": dict(planes=_plane(0, offset=-1)),
        "plane offset past the end": dict(planes=_plane(0, offset=1 << 40)),
        "ground truth past its buffer": dict(images=_image(1, offset=187501)),
        "negative ground-truth offset": dict(images=_image(0, offset=-1)),
        "rows 0": dict(images=_image(0, rows=0)), "cols < 0": dict(images=_image(1, cols=-7)),
        "rows*cols = 2^31": dict(images=_image(0, rows=1 << 16, cols=1 << 15), gt_elems=1 << 40, cam_elems=1 << 40),
        "NaN threshold": dict(thresholds=thr[:5] + [float("nan")] + thr[6:]),
        "inf threshold": dict(thresholds=thr[:99] + [float("inf")]), "-inf threshold": dict(thresholds=[float("-inf")] + thr[1:]),
        "threshold infinite in float32": dict(thresholds=thr[:99] + [1e300]),
        "descending thresholds": dict(thresholds=[0.1, 0.3, 0.2]),
        "histograms over 200 KB (K 21, T 1248)": dict(thresholds=[0.5] * 1248),
        "histograms over 200 KB (K 81, T 317)": dict(num_cls=81, thresholds=[0.5] * 317),
    }
    L = _lib.lib()
    for what, over in bad.items():
        assert _call_cam(_cam_args(**over)) == -1, what
        msg = L.acr_last_error_string()
        assert msg.startswith(b"acr_cam_label_counts:") and len(msg) > len(b"acr_cam_label_counts: "), what
    a = _cam_args()
    need = L.acr_label_counts_workspace(2, 3, 100)
    assert need == 2 * 64 + 3 * 16 + 100 * 4
    assert _call_cam(_cam_args(ws_bytes=need - 1)) == -4                       # the workspace holds the tables
    assert _call_cam(_cam_args(ws=ctypes.c_void_p(a["ws"].value + 4))) == -2
    assert _call_cam(_cam_args(counts=ctypes.c_void_p(a["counts"].value + 4))) == -2


def test_cam_label_counts_with_no_image_launches_nothing():
    assert _call_cam(_cam_args(planes=[], images=[], cams=None, gt_elems=0, cam_elems=0)) == 0


def _call_map(pred, gt, elems, images, num_cls, counts, ws, ws_bytes, num_images=None):
    L = _lib.lib()
    n = num_images if num_images is not None else (len(images) if images is not None else 1)
    return L.acr_label_map_counts(pred, gt, elems, _arr(ctypes.c_longlong, images), n, num_cls, counts, ws, ws_bytes, None)


def test_label_map_counts_rejects_invalid_arguments_before_any_launch():
    buf, dev = _fake()
    L = _lib.lib()
    images = [[0, 375, 500], [187500, 1, 7]]
    ok = dict(pred=dev, gt=dev, elems=187507, images=images, num_cls=K, counts=dev, ws=dev, ws_bytes=L.acr_label_counts_workspace(2, 0, 0))
    bad = {
        "null pred": dict(pred=None), "null gt": dict(gt=None), "null images": dict(images=None, num_images=2),
        "null counts": dict(counts=None), "null workspace": dict(ws=None),
        "num_cls 0": dict(num_cls=0), "num_cls 256": dict(num_cls=256), "negative image count": dict(num_images=-1),
        "image past the buffers": dict(elems=187506), "negative offset": dict(images=[[-1, 375, 500]]),
        "rows 0": dict(images=[[0, 0, 500]]), "cols < 0": dict(images=[[0, 375, -500]]),
    }
    for what, over in bad.items():
        assert _call_map(**{**ok, **over}) == -1, what
        assert L.acr_last_error_string().startswith(b"acr_label_map_counts:"), what
    assert _call_map(**{**ok, "ws_bytes": 2 * 64 - 1}) == -4
    assert _call_map(**{**ok, "ws": ctypes.c_void_p(dev.value + 4)}) == -2
    assert _call_map(**{**ok, "images": [], "pred": dev, "elems": 0}) == 0            # nothing to count: no launch
    del buf
