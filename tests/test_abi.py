"""CPU tier: the C-ABI library builds, loads and exports every symbol include/acr_b200.h declares.
No compute calls here (no GPU in the build container)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "acr_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b((?:acr_|bilateralfilter_)\w+)\s*\(", src)))


def test_header_symbols_are_exported_and_bound():
    from acr_wsss_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__ as g
        g.build()
    names = _declared_symbols()
    assert len(names) >= 18
    handle = ctypes.CDLL(_lib.LIB_PATH)
    for n in names:
        assert hasattr(handle, n), f"{n} declared in acr_b200.h but not exported"
        assert n in _lib.SIGNATURES, f"{n} has no ctypes signature in acr_wsss_b200/_lib.py"
    assert sorted(_lib.SIGNATURES) == names
    assert _lib.lib().acr_abi_version() == 1


def test_product_fails_loudly_without_cuda():
    import torch
    from acr_wsss_b200 import ops
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError):
        ops.consistency_fwd_bwd(torch.zeros(1, 1, 5, 5), torch.zeros(1, 1, 5, 5), 2)


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "acr_wsss_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            txt = open(os.path.join(pkg, fn)).read()
            assert "oracle" not in re.sub(r'""".*?"""', "", txt, flags=re.S).replace("# ", ""), fn


def test_invalid_arguments_are_rejected_before_any_launch():
    from acr_wsss_b200 import _lib
    L = _lib.lib()
    assert L.acr_consistency_fwd_bwd(None, None, 1, 1, 5, 2, 1.0, 1.0, None, None, None, 0, None, None, 0, None, 0, None) == -1
    assert b"null" in L.acr_last_error_string()
    assert L.acr_consistency_workspace(8, 12, 785) >= 8 * 12 * 785 * 4
    assert L.acr_bilateral_workspace(1, 21, 224, 224) > 0
    assert L.acr_pamr_workspace(1, 3, 21, 448, 448, 6) > 0
    # the trunk-glue / optimiser / data-path entry points validate before touching the device too
    import ctypes
    buf = ctypes.create_string_buffer(4096)
    al = ctypes.c_void_p((ctypes.addressof(buf) + 255) & ~255)          # a 256-byte aligned host address: never dereferenced
    mis = ctypes.c_void_p(al.value + 2)
    assert L.acr_gelu_fwd_bf16(None, None, 8, None) == -1
    assert L.acr_gelu_fwd_bf16(mis, al, 8, None) == -2
    assert L.acr_gelu_bwd_bf16(al, al, al, 4, 12, None, 0, None, 0, None) == -1            # F not a multiple of 8
    assert L.acr_gelu_bwd_bf16(al, al, al, 4, 16, al, 1, al, 8, None) == -4                # workspace too small
    assert L.acr_gelu_bwd_workspace(3072) == 64 * 3072 * 4
    assert L.acr_layernorm_fwd(al, 1, al, None, al, al, 4, 768, 1e-6, al, 1, al, al, None) == -1   # residual without sum_out
    assert L.acr_layernorm_fwd(al, 1, None, None, al, al, 4, 100, 1e-6, al, 1, al, al, None) == -1  # E not a multiple of 128
    assert L.acr_layernorm_bwd(al, 1, None, al, 1, al, al, al, 4, 768, al, al, al, None, 0, al, 16, None) == -4
    assert L.acr_layernorm_bwd_workspace(768) == 3 * 296 * 768 * 4
    assert L.acr_sgd_momentum_step(al, al, al, None, 6, 0.5, al, None) == -1               # n not a multiple of 4
    assert L.acr_sgd_momentum_step(mis, al, al, None, 8, 0.5, al, None) == -2
    assert L.acr_augment_batch(None, None, None, 1, 64, None, None, None) == -1
    assert L.acr_augment_batch(al, al, al, 0, 64, al, None, None) == -1
    assert L.acr_colsum_bf16(al, 4, 7, al, 0, al, 1 << 20, None) == -1                    # F odd
    tot, cnt = ctypes.c_double(), ctypes.c_longlong()
    assert L.acr_profile_read(None, ctypes.byref(tot), ctypes.byref(cnt)) == -1
    # GETAM row 0, one image and a batch of S samples: L = 12, H = 12, N = 785
    ok = dict(p=al, g=al, start=0, func=0, skip=1, out=al)
    for over in (dict(p=None), dict(g=None), dict(out=None), dict(start=-1), dict(start=12), dict(func=4), dict(skip=0),
                 dict(skip=785)):
        x = dict(ok, **over)
        assert L.acr_getam_row0(x["p"], x["g"], 12, 12, 785, x["start"], x["func"], x["skip"], x["out"], None, None) == -1, over
        assert L.acr_getam_row0_batch(x["p"], x["g"], 48, 12, 12, 785, x["start"], x["func"], x["skip"], x["out"], None) == -1, over
    for S in (0, 65536):
        assert L.acr_getam_row0_batch(al, al, S, 12, 12, 785, 0, 0, 1, al, None) == -1, S


def test_pseudo_label_writer_roundtrip(tmp_path):
    """The .npy dict format of infer_cam.py:227-228 as evaluation.py:28-36 reads it, and the IoU bookkeeping of :33-67."""
    import numpy as np
    from acr_wsss_b200 import save_cam_dict, load_cam_dict, pseudo_label, label_iou
    rng = np.random.default_rng(0)
    cam = {3: rng.random((5, 7), dtype=np.float32), 14: rng.random((5, 7), dtype=np.float32)}
    f = tmp_path / "img.npy"
    save_cam_dict(str(f), cam)
    back = np.load(str(f), allow_pickle=True).item()          # exactly evaluation.py:29
    assert sorted(back) == [3, 14] and back[3].dtype == np.float32 and np.array_equal(back[14], cam[14])
    assert sorted(load_cam_dict(str(f))) == [3, 14]
    lab = pseudo_label(back, 20, 0.4)
    tensor = np.zeros((21, 5, 7), np.float32)                # evaluation.py:30-36 restated
    for k in back:
        tensor[k + 1] = back[k]
    tensor[0] = 0.4
    assert np.array_equal(lab, np.argmax(tensor, 0).astype(np.uint8))
    gt = lab.copy()
    gt[0, 0] = 255
    gt[1, 1] = (gt[1, 1] + 1) % 21
    iou, miou = label_iou([lab], [gt])
    assert iou.shape == (21,) and 0.0 < miou < 1.0


def test_bench_reference_arm_prints_one_json_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside ours): exactly one JSON line on stdout with the
    contract's keys; and our arm refuses to run without a GPU instead of falling back."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-500:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["cpu_baseline"]["kind"] == "port" and d["value"] > 0
    import torch
    if not torch.cuda.is_available():
        r2 = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=600)
        assert r2.returncode != 0 and "no CUDA device" in (r2.stderr + r2.stdout)
