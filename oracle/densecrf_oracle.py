"""ctypes door onto oracle/densecrf_oracle.c, the CPU restatement of densecrf 2.x mean-field inference.  TEST INFRASTRUCTURE ONLY.

Parity with pydensecrf itself is not pinned (see DESIGN.md section 2); the lattice is tied to the pinned bilateral oracle by
`bilateral` (bit-exact with permuto_oracle.c at H*W % 4 == 0).
"""
import ctypes
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "densecrf_oracle.c")
_lib = None

def _build():
    """Compile densecrf_oracle.c (scalar, -ffp-contract=off: separate multiply and add roundings, as the GPU code) into
    oracle/_build, or into the temporary directory when the tree is read-only; rebuilt when the source is newer."""
    for d in (os.path.join(_HERE, "_build"), os.path.join(tempfile.gettempdir(), f"acr_densecrf_oracle_{os.getuid()}")):
        so = os.path.join(d, "libdensecrf_oracle.so")
        if os.path.exists(so) and os.path.getmtime(so) >= os.path.getmtime(_SRC):
            return so
        try:
            os.makedirs(d, exist_ok=True)
            if not os.access(d, os.W_OK):
                continue
            tmp = f"{so}.{os.getpid()}.tmp"
            subprocess.run([os.environ.get("CC", "gcc"), "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-o", tmp, _SRC, "-lm"],
                           check=True, stdout=subprocess.DEVNULL)
            os.replace(tmp, so)             # atomic: a concurrent loader never sees a half-written library
            return so
        except OSError:
            continue
    raise RuntimeError("cannot build oracle/densecrf_oracle.c: no writable build directory")


def _load():
    global _lib
    if _lib is None:
        lib = ctypes.CDLL(_build())
        f, i, p = ctypes.c_float, ctypes.c_int, ctypes.c_void_p
        lib.densecrf_oracle.argtypes = [p, p, p, i, i, i, i, f, f, f, f, f, f, p]
        lib.densecrf_oracle.restype = None
        lib.densecrf_oracle_bilateral.argtypes = [p, p, p, i, i, i, f, f]
        lib.densecrf_oracle_bilateral.restype = i
        _lib = lib
    return _lib


def dense_crf(image, probs, n_iter=10, sxy_g=3.0, compat_g=3.0, sxy_b=80.0, srgb=13.0, compat_b=10.0, clip=1e-5,
              return_lattice_sizes=False):
    """One image: image [3,H,W] (0..255), probs [C,H,W] -> Q [C,H,W] float32 (and (M_gauss, M_bilateral) on request)."""
    image = np.ascontiguousarray(image, dtype=np.float32)
    probs = np.ascontiguousarray(probs, dtype=np.float32)
    C, H, W = probs.shape
    assert image.shape == (3, H, W)
    q = np.empty_like(probs)
    m = (ctypes.c_int * 2)()
    _load().densecrf_oracle(image.ctypes.data, probs.ctypes.data, q.ctypes.data, C, H, W, int(n_iter), sxy_g, compat_g,
                            sxy_b, srgb, compat_b, clip, ctypes.cast(m, ctypes.c_void_p))
    return (q, (m[0], m[1])) if return_lattice_sizes else q


def bilateral(image, ins, sigmargb, sigmaxy):
    """The d = 5 lattice filter alone: image [3,H,W], ins [K,H,W] -> outs [K,H,W] (no normalisation)."""
    image = np.ascontiguousarray(image, dtype=np.float32)
    ins = np.ascontiguousarray(ins, dtype=np.float32)
    K, H, W = ins.shape
    out = np.empty_like(ins)
    _load().densecrf_oracle_bilateral(image.ctypes.data, ins.ctypes.data, out.ctypes.data, K, H, W, sigmargb, sigmaxy)
    return out
