"""TEST INFRASTRUCTURE ONLY — ctypes binding of oracle/_ref/libdso_ref.so: the REFERENCE's own hot-path translation units
compiled from /root/reference by oracle/ref_build.sh behind the C harness oracle/ref_harness.cpp.

It exposes the same Window interface as oracle/orc.py (the CPU restatement), so tests/test_ref_pin.py can run both on the
same seeded inputs: that comparison is what pins the oracle to the reference.  Only tests/ may import this."""
import ctypes as C
import os
import subprocess

import numpy as np

from . import orc

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DMV_REF_LIB", os.path.join(_HERE, "_ref", "libdso_ref.so"))  # DMV_REF_LIB: tools/eigen_order_sensitivity.py
_LIB = None


def available():
    return os.path.exists(LIB_PATH) or os.path.isdir("/root/reference/src/dso")


def build():
    subprocess.check_call(["bash", os.path.join(_HERE, "ref_build.sh")])


class _Adapter:
    """presents ref_* entry points under the orc_* names orc.Window calls"""

    def __init__(self, L):
        self._L = L

    def __getattr__(self, name):
        if name.startswith("orc_"):
            return getattr(self._L, "ref_" + name[4:])
        raise AttributeError(name)


def lib():
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            build()
        L = C.CDLL(LIB_PATH)
        vp = C.c_void_p
        f32p, f64p, i32p, u8p = orc.f32p, orc.f64p, orc.i32p, orc.u8p
        L.ref_win_create.restype = vp
        L.ref_win_create.argtypes = [C.c_int, C.c_int, C.c_int, f64p, C.c_int]
        L.ref_win_destroy.argtypes = [vp]
        L.ref_win_set_setting.argtypes = [vp, C.c_char_p, C.c_double]
        L.ref_win_set_frame.argtypes = [vp, C.c_int, f64p, f64p, f64p, f64p, C.c_float, C.c_float, C.c_int, f32p]
        L.ref_win_set_points.argtypes = [vp, C.c_int, i32p, f32p, f32p, f32p, f32p, f32p, f32p, u8p]
        L.ref_win_set_residuals.argtypes = [vp, C.c_int, i32p, i32p, vp, vp, vp]
        L.ref_win_prepare.argtypes = [vp]
        for n in ("ref_win_nres", "ref_win_npts", "ref_win_nf"):
            getattr(L, n).argtypes = [vp]
        L.ref_win_get_precalc.argtypes = [vp, f32p]
        L.ref_win_get_RT.argtypes = [vp, f32p]
        L.ref_win_activate.argtypes = [vp, C.c_int, i32p, f32p, f32p, f32p, f32p, f32p, f32p, f32p, C.c_int, i32p, f32p, i32p]
        L.ref_win_marginalize.argtypes = [vp, C.c_int, i32p, C.c_int, f64p, f64p, f64p, f64p, f64p, f64p, C.POINTER(C.c_int), i32p, f32p, u8p]
        L.ref_win_marginalize_frame.argtypes = [vp, C.c_int, f64p, f64p, f64p, f64p]
        L.ref_win_get_nullspaces.argtypes = [vp, f64p]
        L.ref_win_orthogonalize.argtypes = [vp, f64p]
        L.ref_win_get_adjoints.argtypes = [vp, f64p, f64p]
        L.ref_win_get_adHTdeltaF.argtypes = [vp, f32p]
        L.ref_win_get_frame_tables.argtypes = [vp, f64p, f64p, f64p, f32p]
        L.ref_win_get_calib.argtypes = [vp, f32p, f32p, f64p]
        L.ref_win_linearize_all.restype = C.c_double
        L.ref_win_linearize_all.argtypes = [vp, C.c_int, C.c_int]
        L.ref_win_apply_res.argtypes = [vp]
        L.ref_win_get_res_outputs.argtypes = [vp, i32p, f32p, f32p, f32p, vp, i32p, u8p, f32p]
        L.ref_win_accumulate.argtypes = [vp, C.c_int, f64p, f64p, f64p, f64p, f64p, f64p, C.POINTER(C.c_int)]
        L.ref_win_get_point_outputs.argtypes = [vp, f32p, f32p, f32p, f32p, f32p, f32p, f32p, f32p]
        L.ref_win_solve.argtypes = [vp, C.c_int, C.c_double, C.c_int, f64p, f64p, f64p]
        L.ref_win_hot_iteration.restype = C.c_double
        L.ref_win_hot_iteration.argtypes = [vp, f64p, C.c_int]
        L.ref_win_calc_LEnergy.restype = C.c_double
        L.ref_win_calc_LEnergy.argtypes = [vp]
        L.ref_win_calc_MEnergy.restype = C.c_double
        L.ref_win_calc_MEnergy.argtypes = [vp]
        L.ref_pyr_levels.argtypes = [C.c_int, C.c_int, f64p]
        L.ref_make_images.restype = C.c_int64
        L.ref_make_images.argtypes = [C.c_int, C.c_int, f64p, f32p, f32p, vp]
        L.ref_init_point.argtypes = [f32p, C.c_int, C.c_int, f64p, C.c_float, C.c_float, f32p, f32p]
        L.ref_ip_init.argtypes = [C.c_int, f32p, C.c_int, C.c_int, f64p, i32p, i32p, f32p, f32p, f32p, f32p, u8p]
        L.ref_ip_trace.argtypes = [C.c_int, f32p, C.c_int, C.c_int, f64p, f32p, f32p, f32p, f32p, f32p, f32p, f32p, f32p, f32p, f32p, f32p, f32p, i32p, f32p,
                                   f32p]
        L.ref_ct_create.restype = vp
        L.ref_ct_create.argtypes = [C.c_int, C.c_int, f64p]
        L.ref_ct_destroy.argtypes = [vp]
        L.ref_ct_levels.argtypes = [vp]
        L.ref_ct_make_coarse_depth.argtypes = [vp, C.c_int, f32p, f32p, f32p, f32p, f32p]
        L.ref_ct_get_ref_points.argtypes = [vp, C.c_int, vp, vp, vp, vp]
        L.ref_ct_set_new_frame.argtypes = [vp, f32p, C.c_float, C.c_float, C.c_double, C.c_double]
        L.ref_ct_get_K.argtypes = [vp, C.c_int, f32p, i32p]
        L.ref_ct_calc_res.argtypes = [vp, C.c_int, f64p, f64p, C.c_double, C.c_double, C.c_float, f64p]
        L.ref_ct_get_warped.argtypes = [vp, vp]
        L.ref_ct_calc_gs.argtypes = [vp, C.c_int, C.c_double, C.c_double, C.c_int, f64p, f64p]
        L.ref_ct_track.argtypes = [vp, f64p, f64p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_int, f64p, C.c_int, f64p, f64p, C.POINTER(C.c_int)]
        _LIB = L
    return _LIB


class Window(orc.Window):
    """The reference's EnergyFunctional / PointFrameResidual objects built from a synth.make_window() dict.
    Process-global state (wG, hG, settings) belongs to the reference: keep ONE RefWindow alive at a time."""

    def __init__(self, W, nthreads=1, settings=None):
        W = dict(W)
        W.pop("HM", None); W.pop("bM", None)
        self._ref = lib()
        super().__init__(W, nthreads=nthreads, settings=settings, _lib=_Adapter(self._ref))

    def activate(self, host, P, minObs=1):
        """the reference's ImmaturePoint::linearizeResidual under the optimizeImmaturePoint driver, on this window's frames"""
        n = len(P["u"])
        c = lambda a, t: np.ascontiguousarray(a, t)
        status = np.zeros(n, np.int32); idepth = np.zeros(n, np.float32); rs = np.zeros((n, self.nf), np.int32)
        self._ref.ref_win_activate(self.h, n, c(host, np.int32), P["u"], P["v"], P["color"], P["weights"], P["energyTH"], c(P["idepth_min"], np.float32),
                                   c(P["idepth_max"], np.float32), int(minObs), status, idepth, rs.reshape(-1))
        return status, idepth, rs

    def __del__(self):
        try:
            self._ref.ref_win_destroy(self.h)
        except Exception:
            pass


def make_images(img, K):
    L = lib()
    h, w = img.shape
    K = np.ascontiguousarray(K, np.float64)
    lv = L.ref_pyr_levels(w, h, K)
    tot = sum((w >> l) * (h >> l) * 3 for l in range(lv))
    out = np.zeros(tot, np.float32)
    n = L.ref_make_images(w, h, K, np.ascontiguousarray(img, np.float32).reshape(-1), out, None)
    assert n == tot
    res, off = [], 0
    for l in range(lv):
        sz = (w >> l) * (h >> l) * 3
        res.append(out[off:off + sz].reshape(h >> l, w >> l, 3))
        res[-1][[0, -1], :, 1:] = 0   # gradients of the first and last row: left uninitialised by FrameHessian::makeImages (HessianBlocks.cpp:L169-179)
        off += sz
    return res


def init_point(dI, w, h, K, u, v):
    c = np.zeros(8, np.float32); wt = np.zeros(8, np.float32)
    ok = lib().ref_init_point(np.ascontiguousarray(dI, np.float32).reshape(-1), w, h, np.ascontiguousarray(K, np.float64), float(u), float(v), c, wt)
    return bool(ok), c, wt


class CoarseTracker(orc.CoarseTracker):
    """The reference's CoarseTracker (levels as setGlobalCalib yields them; forcing a level count is not possible there)."""

    def __init__(self, w, h, K):
        self._ref = lib()
        self.L = _Adapter(self._ref)
        self.w, self.h = w, h
        self.hd = self._ref.ref_ct_create(w, h, np.ascontiguousarray(K, np.float64))
        self.levels = self._ref.ref_ct_levels(self.hd)
        self._keep = []

    def __del__(self):
        try:
            self._ref.ref_ct_destroy(self.hd)
        except Exception:
            pass


def ip_init(dI_host, w, h, K, u, v):
    K = np.ascontiguousarray(K, np.float64)
    return orc.ip_init(dI_host, w, h, u, v, _fn=lambda n, dI, w_, h_, *rest: lib().ref_ip_init(n, dI, w_, h_, K, *rest))


def ip_trace(P, dI, w, h, K, KRKi, Kt, aff):
    K = np.ascontiguousarray(K, np.float64)
    return orc.ip_trace(P, dI, w, h, KRKi, Kt, aff, _fn=lambda n, dI_, w_, h_, *rest: lib().ref_ip_trace(n, dI_, w_, h_, K, *rest))


class CoarseInit(orc.CoarseInit):
    """the reference's compiled CoarseInitializer behind the same interface (oracle/ref_harness.cpp ref_ci_*).  Process-global calibration
    state belongs to the reference: keep one alive at a time."""

    _PREFIX = "ref_ci_"

    def __init__(self, w, h, K):
        super().__init__(w, h, K, _lib=lib())
