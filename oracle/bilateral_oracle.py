"""ctypes doors onto the two CPU checkers of the bilateral filter.  TEST INFRASTRUCTURE ONLY.

  oracle_bilateral : oracle/permuto_oracle.c (this repo's C restatement; always available after
                     `make -C oracle`); oracle_lattice_sizes returns its vertex count per image
  ref_bilateral    : oracle/_ref/libbilateral_ref.so = the reference's own C++
                     (wrapper/bilateralfilter/{bilateralfilter,permutohedral}.cpp) compiled in the build
                     container; travels to the GPU box as a prebuilt file, absent in a fresh clone.
"""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ORACLE_SO = os.path.join(_HERE, "_build", "libpermuto_oracle.so")
_REF_SO = os.path.join(_HERE, "_ref", "libbilateral_ref.so")
_ARGS = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int,
         ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_float]


def build():
    subprocess.run(["make", "-C", _HERE], check=True, stdout=subprocess.DEVNULL)


def _call(fn, images, ins, sigmargb, sigmaxy):
    images = np.ascontiguousarray(images, dtype=np.float32)
    ins = np.ascontiguousarray(ins, dtype=np.float32)
    N, K, H, W = ins.shape
    assert images.shape == (N, 3, H, W)
    outs = np.zeros_like(ins)
    fn(images.ctypes.data, images.size, ins.ctypes.data, ins.size, outs.ctypes.data, outs.size,
       N, K, H, W, float(sigmargb), float(sigmaxy))
    return outs


def _oracle_lib():
    if not os.path.exists(_ORACLE_SO):
        build()
    lib = ctypes.CDLL(_ORACLE_SO)
    lib.permuto_oracle_batch.argtypes = _ARGS
    lib.permuto_oracle_batch.restype = None
    lib.permuto_oracle_image_variant.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
                                                 ctypes.c_int, ctypes.c_float, ctypes.c_float, ctypes.c_int]
    lib.permuto_oracle_image_variant.restype = ctypes.c_int
    return lib


def oracle_bilateral(images, ins, sigmargb, sigmaxy, skip_blur_axis=None):
    """The filter, or with skip_blur_axis = j (0..5) the filter without its j-th blur pass (a known-wrong variant)."""
    lib = _oracle_lib()
    if skip_blur_axis is None:
        return _call(lib.permuto_oracle_batch, images, ins, sigmargb, sigmaxy)
    assert 0 <= skip_blur_axis <= 5
    images = np.ascontiguousarray(images, dtype=np.float32)
    ins = np.ascontiguousarray(ins, dtype=np.float32)
    N, K, H, W = ins.shape
    outs = np.zeros_like(ins)
    for n in range(N):
        lib.permuto_oracle_image_variant(images[n].ctypes.data, ins[n].ctypes.data, outs[n].ctypes.data, K, H, W,
                                         float(sigmargb), float(sigmaxy), int(skip_blur_axis))
    return outs


def oracle_lattice_sizes(images, sigmargb, sigmaxy):
    """Number of lattice vertices M of every image of images [N,3,H,W] (the reference's phantom pad pixels included)."""
    lib = _oracle_lib()
    images = np.ascontiguousarray(images, dtype=np.float32)
    N, three, H, W = images.shape
    assert three == 3
    return [int(lib.permuto_oracle_image_variant(images[n].ctypes.data, None, None, 0, H, W, float(sigmargb), float(sigmaxy), -1))
            for n in range(N)]


def have_ref():
    return os.path.exists(_REF_SO)


def ref_bilateral(images, ins, sigmargb, sigmaxy):
    lib = ctypes.CDLL(_REF_SO)
    lib.ref_bilateralfilter_batch.argtypes = _ARGS
    lib.ref_bilateralfilter_batch.restype = None
    return _call(lib.ref_bilateralfilter_batch, images, ins, sigmargb, sigmaxy)
