"""CPU tier: the CAM contraction entry points (acr_affinity_refine_tc, acr_patch_cam_tc in csrc/refine_tc.cu), the batched
GETAM row-0 kernel (acr_getam_row0_batch, csrc/cam.cu) and the low-res size limit of acr_cam_finish reject invalid arguments
before any launch.  The addresses are fake and never dereferenced.  A valid call must stop at the sm_100 check on a machine
without such a device; where one is present the valid calls are not made, because they would launch on the fake addresses."""
import ctypes

from acr_wsss_b200 import _lib

B, L, N = 2, 12, 785


def _fake():
    buf = ctypes.create_string_buffer(4096)
    return buf, (ctypes.addressof(buf) + 255) & ~255


def _no_sm100():
    return not _lib.lib().acr_device_is_sm100()


def _align256(n):
    return (n + 255) // 256 * 256


def _refine(**over):
    keep, a = _fake()
    lib = _lib.lib()
    x = dict(attn=a, B=B, L=L, N=N, cam=a, C=20, t=1, normalize=0, out=a, ws=None, ws_bytes=0)
    x.update(over)
    rc = lib.acr_affinity_refine_tc(x["attn"], x["B"], x["L"], x["N"], x["cam"], x["C"], x["t"], x["normalize"], x["out"],
                                    x["ws"], x["ws_bytes"], None)
    del keep
    return rc, lib.acr_last_error_string().decode()


def _patch_cam(**over):
    keep, a = _fake()
    lib = _lib.lib()
    x = dict(tok=a, bs=785 * 768, rs=768, B=2, M=784, E=768, w=a, bias=a, C=20, out=a)
    x.update(over)
    rc = lib.acr_patch_cam_tc(x["tok"], x["bs"], x["rs"], x["B"], x["M"], x["E"], x["w"], x["bias"], x["C"], 1, x["out"], None)
    del keep
    return rc, lib.acr_last_error_string().decode()


def test_refine_tc_workspace():
    lib = _lib.lib()
    Np = N - 1
    two = _align256(B * Np * Np * 4) + _align256(B * Np * 20 * 4)
    assert lib.acr_affinity_refine_tc_workspace(B, N, 20, 2) == two
    assert lib.acr_affinity_refine_tc_workspace(B, N, 20, 3) == two           # one A and one ping-pong buffer for any t > 1
    assert lib.acr_affinity_refine_tc_workspace(1, 2, 1, 2) == 512            # each part padded to 256 bytes
    assert lib.acr_affinity_refine_tc_workspace(3, 401, 33, 2) == _align256(3 * 400 * 400 * 4) + _align256(3 * 400 * 33 * 4)
    for args in ((B, N, 20, 1), (B, N, 20, 0), (0, N, 20, 2), (B, 1, 20, 2), (B, N, 0, 2)):
        assert lib.acr_affinity_refine_tc_workspace(*args) == 0, args


def test_refine_tc_rejects_invalid_arguments_before_any_launch():
    lib = _lib.lib()
    bad = {
        "null attn": dict(attn=None), "null cam": dict(cam=None), "null out": dict(out=None),
        "B 0": dict(B=0), "B 65536": dict(B=65536), "L 0": dict(L=0), "N 1": dict(N=1), "C 0": dict(C=0), "t 0": dict(t=0),
        "C 128 with normalize": dict(C=128, normalize=1), "C 200": dict(C=200),
    }
    for what, over in bad.items():
        rc, err = _refine(**over)
        assert rc == -1, (what, rc, err)
        assert err.startswith("acr_affinity_refine_tc"), (what, err)
    rc, err = _refine(C=128, normalize=1)
    assert "C + normalize must be <= 128" in err, err
    need = lib.acr_affinity_refine_tc_workspace(B, N, 20, 2)
    _, ws = _fake()
    short = {
        "no workspace": dict(t=2, ws=None, ws_bytes=need),
        "short workspace": dict(t=2, ws=ws, ws_bytes=need - 1),
        "misaligned workspace": dict(t=2, ws=ws + 16, ws_bytes=need),
        "t 3, no workspace": dict(t=3, normalize=1),
    }
    for what, over in short.items():
        rc, err = _refine(**over)
        assert rc == -4, (what, rc, err)
        assert err.startswith("acr_affinity_refine_tc"), (what, err)
    if _no_sm100():
        for over in (dict(), dict(C=127, normalize=1), dict(C=128, normalize=0), dict(t=2, ws=ws, ws_bytes=need)):
            rc, err = _refine(**over)
            assert rc == -3, (over, rc, err)


def test_patch_cam_tc_rejects_invalid_arguments_before_any_launch():
    bad = {
        "null tokens": dict(tok=None), "null weight": dict(w=None), "null out": dict(out=None),
        "B 0": dict(B=0), "B 65536": dict(B=65536), "M 0": dict(M=0), "E 0": dict(E=0), "C 0": dict(C=0), "C 129": dict(C=129),
        "row stride < E": dict(rs=767),
    }
    for what, over in bad.items():
        rc, err = _patch_cam(**over)
        assert rc == -1, (what, rc, err)
        assert err.startswith("acr_patch_cam_tc"), (what, err)
    if _no_sm100():
        for over in (dict(), dict(C=128), dict(bias=None), dict(rs=773)):
            rc, err = _patch_cam(**over)
            assert rc == -3, (over, rc, err)


def test_getam_row0_batch_rejects_invalid_arguments():
    keep, a = _fake()
    lib = _lib.lib()
    x0 = dict(p=a, g=a, S=48, L=12, H=12, N=785, start=0, func=0, skip=1, out=a)
    bad = {
        "null p": dict(p=None), "null g": dict(g=None), "null out": dict(out=None),
        "S 0": dict(S=0), "S 65536": dict(S=65536), "L 0": dict(L=0), "H 0": dict(H=0), "N 1": dict(N=1),
        "start_layer < 0": dict(start=-1), "start_layer = L": dict(start=12),
        "func -1": dict(func=-1), "func 4": dict(func=4), "skip 0": dict(skip=0), "skip = N": dict(skip=785),
    }
    for what, over in bad.items():
        x = dict(x0, **over)
        rc = lib.acr_getam_row0_batch(x["p"], x["g"], x["S"], x["L"], x["H"], x["N"], x["start"], x["func"], x["skip"], x["out"], None)
        assert rc == -1, (what, rc)
        assert lib.acr_last_error_string().startswith(b"acr_getam_row0_batch"), what
    del keep


def test_cam_finish_rejects_low_res_maps_over_200_kb():
    """2 * sum_s ph*pw floats of low-res maps must fit 200 KB of shared memory: 204,800 bytes pass the check, 204,808 do not."""
    keep, a = _fake()
    lib = _lib.lib()
    dev = ctypes.c_void_p(a)

    def call(grid):
        ns = len(grid) // 2
        maps = (ctypes.c_void_p * ns)(*([dev] * ns))
        table = (ctypes.c_longlong * 6)(0, 0, 0, 0, 4, 4)
        return lib.acr_cam_finish(maps, maps, (ctypes.c_int * len(grid))(*grid), ns, 1, 1, 1, dev, table, 1, dev, 16, dev, 48, None)

    over = [80, 160, 80, 160, 1, 1]
    assert call(over) == -1
    err = lib.acr_last_error_string().decode()
    assert err.startswith("acr_cam_finish") and "204808 bytes exceed 204800" in err, err
    if _no_sm100():
        assert call([80, 160, 80, 160]) == -3                                # exactly 200 KB
    del keep
