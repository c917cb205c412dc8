"""TEST INFRASTRUCTURE ONLY — ctypes binding of oracle/_ref/libdso_ref_select.so: the REFERENCE's own PixelSelector::makeMaps behind the
C harness oracle/ref_select.cpp (built by oracle/ref_select_build.sh from the reference's sources where they lie).  Only
tests/golden/make_select_golden.py uses it: it records the reference's results into tests/golden/ref_select.npz."""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_ref", "libdso_ref_select.so")
_LIB = None

f32p = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")
f64p = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")


def lib():
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            subprocess.check_call(["bash", os.path.join(_HERE, "ref_select_build.sh")])
        L = C.CDLL(LIB_PATH)
        L.ref_make_maps.argtypes = [C.c_int, C.c_int, f64p, f32p, C.c_void_p, C.c_void_p, C.c_float, C.c_int, C.c_float, C.POINTER(C.c_int32), f32p,
                                    C.c_void_p]
        _LIB = L
    return _LIB


def make_maps(img, K, density, recursionsLeft=1, thFactor=1.0, potential=3, B=None, settings=None):
    """PixelSelector::makeMaps on the frame FrameHessian::makeImages builds from img (CalibHessian::B = B, identity when None).
    settings = (minGradHistCut, minGradHistAdd, gradDownweightPerLevel, selectDirectionDistribution) or None.
    Returns (map as uint8 h x w, numHaveSub, potential after the call, [dIp of levels 0..2])."""
    h, w = img.shape
    m = np.zeros(w * h, np.float32)
    pot = C.c_int32(potential)
    dIp = np.zeros(sum((w >> l) * (h >> l) * 3 for l in range(3)), np.float32)
    Bc = None if B is None else np.ascontiguousarray(B, np.float32)
    Sc = None if settings is None else np.ascontiguousarray(settings, np.float32)
    r = lib().ref_make_maps(w, h, np.ascontiguousarray(K, np.float64), np.ascontiguousarray(img, np.float32).reshape(-1),
                            None if Bc is None else Bc.ctypes.data, None if Sc is None else Sc.ctypes.data, float(density), int(recursionsLeft),
                            float(thFactor), C.byref(pot), m, dIp.ctypes.data)
    lv, off = [], 0
    for l in range(3):
        sz = (w >> l) * (h >> l) * 3
        lv.append(dIp[off:off + sz].reshape(h >> l, w >> l, 3))
        off += sz
    return m.reshape(h, w).astype(np.uint8), r, pot.value, lv
