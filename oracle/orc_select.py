"""TEST INFRASTRUCTURE ONLY — ctypes binding of oracle/liborc_select.so, the CPU oracle of pixel selection for new keyframes
(PixelSelector::makeMaps and FullSystem::makeNewTraces, oracle/orc_select.cpp).  Frames are built with oracle.orc.make_images.

Only tests/ and tools/bench_select.py may import this."""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "liborc_select.so")
_LIB = None

f32p = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")
i32p = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
u8p = np.ctypeslib.ndpointer(dtype=np.uint8, flags="C_CONTIGUOUS")


def build():
    subprocess.check_call(["make", "-s", "-C", _HERE, "-f", "Makefile.select"])


def lib():
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            build()
        L = C.CDLL(LIB_PATH)
        vp = C.c_void_p
        L.orc_random_pattern.argtypes = [C.c_int, u8p]
        L.orc_random_pattern.restype = None
        L.orc_make_maps.argtypes = [C.c_int, C.c_int, f32p, f32p, f32p, vp, vp, C.c_float, C.c_int, C.c_float, C.POINTER(C.c_int32), f32p]
        L.orc_make_new_traces.argtypes = [C.c_int, C.c_int, f32p, f32p, f32p, vp, vp, C.c_float, C.c_int, C.c_float, C.POINTER(C.c_int32),
                                          C.POINTER(C.c_int32), C.c_int, i32p, i32p, f32p, f32p, f32p, f32p, f32p]
        _LIB = L
    return _LIB


def random_pattern(n):
    """PixelSelector::randomPattern: glibc srand(3141592), then rand() & 0xFF, n times"""
    out = np.zeros(n, np.uint8)
    lib().orc_random_pattern(n, out)
    return out


def _select_args(dIp, B, settings):
    c = lambda a: np.ascontiguousarray(a, np.float32)
    lv = [c(dIp[l]).reshape(-1) for l in range(3)]
    Bc = None if B is None else c(B)
    Sc = None if settings is None else c(settings)
    return lv, Bc, Sc, (None if Bc is None else Bc.ctypes.data), (None if Sc is None else Sc.ctypes.data)


def make_maps(dIp, density, recursionsLeft=1, thFactor=1.0, potential=3, B=None, settings=None):
    """PixelSelector::makeMaps on the frame whose levels 0..2 are dIp[l] (h_l x w_l x 3) -> (map uint8 h x w, numHaveSub, potential after).
    B = CalibHessian::B (256 floats) or None; settings = (minGradHistCut, minGradHistAdd, gradDownweightPerLevel, selectDirectionDistribution)."""
    h, w = dIp[0].shape[:2]
    lv, Bc, Sc, Bp, Sp = _select_args(dIp, B, settings)
    m = np.zeros(w * h, np.float32)
    pot = C.c_int32(potential)
    r = lib().orc_make_maps(w, h, lv[0], lv[1], lv[2], Bp, Sp, float(density), int(recursionsLeft), float(thFactor), C.byref(pot), m)
    return m.reshape(h, w).astype(np.uint8), r, pot.value


def make_new_traces(dIp, density, recursionsLeft=1, thFactor=1.0, potential=3, B=None, settings=None):
    """FullSystem::makeNewTraces: the kept immature points (dict of arrays, raster order), numHaveSub and the potential after the call."""
    h, w = dIp[0].shape[:2]
    lv, Bc, Sc, Bp, Sp = _select_args(dIp, B, settings)
    cap = w * h
    P = dict(u=np.zeros(cap, np.int32), v=np.zeros(cap, np.int32), type=np.zeros(cap, np.float32), color=np.zeros((cap, 8), np.float32),
             weights=np.zeros((cap, 8), np.float32), gradH=np.zeros((cap, 4), np.float32), energyTH=np.zeros(cap, np.float32))
    pot, sub = C.c_int32(potential), C.c_int32(0)
    n = lib().orc_make_new_traces(w, h, lv[0], lv[1], lv[2], Bp, Sp, float(density), int(recursionsLeft), float(thFactor), C.byref(pot), C.byref(sub),
                                  cap, P["u"], P["v"], P["type"], P["color"].reshape(-1), P["weights"].reshape(-1), P["gradH"].reshape(-1),
                                  P["energyTH"])
    return {k: a[:n] for k, a in P.items()}, sub.value, pot.value
