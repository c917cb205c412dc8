"""ctypes binding of the C ABI in include/dmvio_b200.h (libdmvio_b200.so).

This is the only way Python (tests, bench.py, __graft_entry__) reaches the product: there is no Python/torch
re-implementation of the path and no CPU fallback — loading fails loudly if the CUDA library is missing.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DMVIO_B200_LIB") or os.path.join(_HERE, "libdmvio_b200.so")   # override: A/B runs of differently built libraries
_LIB = None

f32p = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")
f64p = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
i32p = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
vp = C.c_void_p

MAX_FRAMES = 8
PRECALC_FLOATS = 32


class DmvError(RuntimeError):
    pass


class BAConfig(C.Structure):
    _fields_ = [("w", C.c_int), ("h", C.c_int), ("max_frames", C.c_int), ("max_points", C.c_int), ("device", C.c_int), ("chunk_points", C.c_int)]


class BAParams(C.Structure):
    _fields_ = [("huberTH", C.c_float), ("outlierTHSumComponent", C.c_float), ("affineOptModeA", C.c_float), ("affineOptModeB", C.c_float)]


class BAState(C.Structure):
    _fields_ = [("calib", C.c_float * 8), ("precalc", vp), ("frameEnergyTH", vp), ("idepth", vp), ("idepth_zero", vp)]


class BALinResult(C.Structure):
    _fields_ = [("energy", C.c_double), ("n_in", C.c_int), ("n_oob", C.c_int), ("n_outlier", C.c_int)]


class BAActivateArgs(C.Structure):
    _fields_ = [("n", C.c_int)] + [(k, C.c_void_p) for k in ("host", "u", "v", "color8", "weights8", "energyTH", "idepth_min", "idepth_max", "RT")] + \
               [("minObs", C.c_int)] + [(k, C.c_void_p) for k in ("status", "idepth", "res_state")]


class BAMargArgs(C.Structure):
    _fields_ = [("n", C.c_int32), ("point", C.c_void_p), ("adHTdeltaF", C.c_void_p), ("cDeltaF", C.c_float * 4), ("idepthFixPriorMargFac", C.c_float)] + \
               [(k, C.c_void_p) for k in ("M", "Mb", "Msc", "Mbsc", "resInM", "ngoodRes", "res_toZeroF", "isLinearized")]


class IPPoints(C.Structure):
    _fields_ = [("n", C.c_int)] + [(k, C.c_void_p) for k in ("u", "v", "color8", "weights8", "gradH4", "energyTH", "idepth_min", "idepth_max", "quality",
                                                              "lastTraceStatus", "lastTraceUV2", "lastTracePixelInterval")]


class BABatch:
    """dmv_ba_batch: B independent windows (BA handles on one device) linearised by ONE launch (include/dmvio_b200.h)."""

    def __init__(self, bas):
        self.L = lib()
        self.bas = list(bas)
        n = len(self.bas)
        self._harr = (C.c_void_p * n)(*[b.h for b in self.bas])
        h = C.c_void_p()
        check(self.L.dmv_ba_batch_create(self._harr, n, C.byref(h)))
        self.h = h

    def _args(self, xs, states):
        n = len(self.bas)
        self._xs = [None if x is None else _c(x, np.float64) for x in (xs or [None] * n)]
        self._sts = [b._state(*st) for b, st in zip(self.bas, states)]
        xarr = (C.c_void_p * n)(*[None if x is None else x.ctypes.data for x in self._xs])
        sarr = (C.c_void_p * n)(*[C.addressof(st) for st in self._sts])
        return xarr, sarr

    def gn_step(self, xs, states):
        """states[i] = (calib8, precalc, TH); xs[i] = x or None.  Returns one result dict per window."""
        n = len(self.bas)
        xarr, sarr = self._args(xs, states)
        res = (BALinResult * n)()
        sums = np.zeros(3 * n)
        check(self.L.dmv_ba_batch_gn_step(self.h, xarr, sarr, res, sums.ctypes.data))
        return [dict(energy=r.energy, n_in=r.n_in, n_oob=r.n_oob, n_outlier=r.n_outlier, sums=sums[3 * i:3 * i + 3]) for i, r in enumerate(res)]

    def bench(self, xs, states, iters=100, warmup=5):
        """returns (kernel ms per launch [CUDA events], e2e ms per batched call [wall clock, issued from C], None)"""
        n = len(self.bas)
        xarr, sarr = self._args(xs, states)
        e2e, ker = C.c_double(0), C.c_double(0)
        check(self.L.dmv_ba_batch_bench(self.h, self._harr, n, xarr, sarr, max(1, warmup), C.byref(e2e), C.byref(ker)))
        check(self.L.dmv_ba_batch_bench(self.h, self._harr, n, xarr, sarr, iters, C.byref(e2e), C.byref(ker)))
        return ker.value, e2e.value, None

    def close(self):
        if self.h:
            self.L.dmv_ba_batch_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class CTConfig(C.Structure):
    _fields_ = [("w", C.c_int), ("h", C.c_int), ("levels", C.c_int), ("max_points", C.c_int), ("device", C.c_int)]


class CTTrackArgs(C.Structure):
    _fields_ = [("R", C.c_double * 9), ("t", C.c_double * 3), ("a", C.c_double), ("b", C.c_double), ("ref_a", C.c_double), ("ref_b", C.c_double),
                ("ref_exposure", C.c_float), ("new_exposure", C.c_float), ("coarseCutoffTH", C.c_float), ("affineOptModeA", C.c_float),
                ("affineOptModeB", C.c_float), ("coarsestLvl", C.c_int), ("minResForAbort", C.c_double * 5)]


class CTTrackResult(C.Structure):
    _fields_ = [("R", C.c_double * 9), ("t", C.c_double * 3), ("a", C.c_double), ("b", C.c_double), ("lastResiduals", C.c_double * 5),
                ("flowIndicators", C.c_double * 3), ("trackingGood", C.c_int), ("iterations", C.c_int), ("evaluations", C.c_int), ("status", C.c_int)]


class CIEvalArgs(C.Structure):
    _fields_ = [("level", C.c_int), ("RKi", C.c_float * 9), ("t_d", C.c_double * 3), ("t_log", C.c_double * 3), ("r2new_aff", C.c_float * 2),
                ("huberTH", C.c_float), ("alphaK", C.c_float), ("alphaW", C.c_float), ("couplingWeight", C.c_float),
                ("weightZeroPriorX", C.c_double), ("weightZeroPriorY", C.c_double),
                ("idepth_new", C.c_void_p), ("isGood", C.c_void_p), ("energy2", C.c_void_p), ("iR", C.c_void_p),
                ("isGood_new", C.c_void_p), ("energy_new2", C.c_void_p), ("maxstep", C.c_void_p), ("lastHessian_new", C.c_void_p),
                ("JbBuffer_new10", C.c_void_p)]


class CIEvalResult(C.Structure):
    _fields_ = [("H", C.c_float * 64), ("b", C.c_float * 8), ("Hsc", C.c_float * 64), ("bsc", C.c_float * 8), ("res3", C.c_float * 3),
                ("alphaOpt", C.c_float), ("n_good_new", C.c_int)]


class PSSettings(C.Structure):
    _fields_ = [("minGradHistCut", C.c_float), ("minGradHistAdd", C.c_float), ("gradDownweightPerLevel", C.c_float), ("selectDirectionDistribution", C.c_int)]


class PSArgs(C.Structure):
    _fields_ = [("density", C.c_float), ("recursionsLeft", C.c_int), ("thFactor", C.c_float), ("currentPotential", C.c_int), ("B256", C.c_void_p),
                ("settings", C.POINTER(PSSettings))]


class PSResult(C.Structure):
    _fields_ = [("numHaveSub", C.c_int), ("currentPotential", C.c_int)]


# every symbol declared in include/dmvio_b200.h (checked by tests/test_capi_symbols.py)
SYMBOLS = [
    "dmv_last_error", "dmv_version", "dmv_device_count",
    "dmv_ba_create", "dmv_ba_destroy", "dmv_ba_set_params", "dmv_ba_default_params", "dmv_ba_upload_frame", "dmv_ba_upload_image", "dmv_ba_adopt_frame",
    "dmv_ba_set_window", "dmv_ba_set_points", "dmv_ba_set_residuals", "dmv_ba_set_adjoints", "dmv_ba_set_state", "dmv_ba_linearize",
    "dmv_ba_get_residual_outputs", "dmv_ba_get_target_energies", "dmv_ba_apply_res", "dmv_ba_accumulate", "dmv_ba_get_point_outputs", "dmv_ba_get_solve_HdiF",
    "dmv_ba_resubstitute", "dmv_ba_backup_points", "dmv_ba_restore_points", "dmv_ba_get_idepth", "dmv_ba_gn_step", "dmv_nccl_unique_id",
    "dmv_ba_comm_init", "dmv_ba_activate_points", "dmv_ba_marginalize_points", "dmv_ba_drop_residuals", "dmv_ba_reset_oob", "dmv_ba_p2p_export", "dmv_ba_p2p_import", "dmv_ba_last_timing", "dmv_ba_bench_device", "dmv_ba_kernel_launch_count", "dmv_ba_io_bytes", "dmv_ba_set_timing", "dmv_ba_bench_e2e",
    "dmv_ba_batch_create", "dmv_ba_batch_destroy", "dmv_ba_batch_gn_step", "dmv_ba_batch_set_timing", "dmv_ba_batch_last_kernel_ms", "dmv_ba_batch_bench",
    "dmv_ct_create", "dmv_ct_destroy", "dmv_ct_set_K", "dmv_ct_set_ref", "dmv_ct_make_coarse_depth", "dmv_ct_get_ref", "dmv_ct_upload_new", "dmv_ct_upload_new_image", "dmv_ct_set_huber",
    "dmv_ci_create", "dmv_ci_destroy", "dmv_ci_set_K", "dmv_ci_upload_first", "dmv_ci_upload_new", "dmv_ci_set_points", "dmv_ci_calc_res_and_gs", "dmv_ci_kernel_launch_count",
    "dmv_ct_calc_res_gs", "dmv_ct_track", "dmv_ip_default_settings", "dmv_ct_init_points", "dmv_ct_trace_points", "dmv_ct_trace_points_multi", "dmv_ct_set_timing", "dmv_ct_last_timing", "dmv_ct_kernel_launch_count", "dmv_ct_last_point_evaluations",
    "dmv_ps_default_settings", "dmv_ct_select_pixels", "dmv_ct_make_new_traces",
]


def lib():
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise DmvError(f"{LIB_PATH} is missing: build it with `make -C dm-vio_b200` (python -c 'import __graft_entry__ as g; g.build()')")
        L = C.CDLL(LIB_PATH)
        L.dmv_last_error.restype = C.c_char_p
        L.dmv_version.restype = C.c_char_p
        L.dmv_ba_create.argtypes = [C.POINTER(BAConfig), C.POINTER(vp)]
        L.dmv_ba_destroy.argtypes = [vp]
        L.dmv_ba_set_params.argtypes = [vp, C.POINTER(BAParams)]
        L.dmv_ba_default_params.argtypes = [C.POINTER(BAParams)]
        L.dmv_ba_upload_frame.argtypes = [vp, C.c_int, f32p]
        L.dmv_ba_upload_image.argtypes = [vp, C.c_int, f32p]
        L.dmv_ba_set_window.argtypes = [vp, C.c_int, vp]
        L.dmv_ba_set_points.argtypes = [vp, C.c_int, i32p, f32p, f32p, f32p, vp, f32p, f32p, vp]
        L.dmv_ba_set_residuals.argtypes = [vp, C.c_int, i32p, i32p, vp, vp]
        L.dmv_ba_set_adjoints.argtypes = [vp, f64p, f64p]
        L.dmv_ba_set_state.argtypes = [vp, C.POINTER(BAState)]
        L.dmv_ba_linearize.argtypes = [vp, C.POINTER(BALinResult)]
        L.dmv_ba_get_residual_outputs.argtypes = [vp, vp, vp, vp, vp, vp]
        L.dmv_ba_get_target_energies.argtypes = [vp, C.c_int, f32p, C.c_int, C.POINTER(C.c_int)]
        L.dmv_ba_apply_res.argtypes = [vp]
        L.dmv_ba_accumulate.argtypes = [vp, f64p, f64p, f64p, f64p, C.POINTER(C.c_int)]
        L.dmv_ba_get_point_outputs.argtypes = [vp, vp, vp, vp, vp, vp]
        L.dmv_ba_resubstitute.argtypes = [vp, f64p, vp, C.c_int, f64p]
        L.dmv_ba_backup_points.argtypes = [vp]
        L.dmv_ba_restore_points.argtypes = [vp]
        L.dmv_ba_get_idepth.argtypes = [vp, vp, vp]
        L.dmv_ba_gn_step.argtypes = [vp, vp, C.POINTER(BAState), C.POINTER(BALinResult), f64p]
        L.dmv_nccl_unique_id.argtypes = [vp]
        L.dmv_ba_comm_init.argtypes = [vp, C.c_int, C.c_int, vp]
        L.dmv_ba_activate_points.argtypes = [vp, C.POINTER(BAActivateArgs)]
        L.dmv_ba_marginalize_points.argtypes = [vp, C.POINTER(BAMargArgs)]
        L.dmv_ba_drop_residuals.argtypes = [vp, C.c_int, i32p]
        L.dmv_ba_reset_oob.argtypes = [vp]
        L.dmv_ba_p2p_export.argtypes = [vp, vp]
        L.dmv_ba_p2p_import.argtypes = [vp, C.c_int, C.c_int, vp]
        L.dmv_ba_last_timing.argtypes = [vp, f32p]
        L.dmv_ba_bench_device.argtypes = [vp, vp, C.c_int, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_float)]
        L.dmv_ba_kernel_launch_count.argtypes = [vp, C.POINTER(C.c_longlong)]
        L.dmv_ba_set_timing.argtypes = [vp, C.c_int]
        L.dmv_ba_bench_e2e.argtypes = [vp, vp, C.POINTER(BAState), C.c_int, C.POINTER(C.c_double)]
        L.dmv_ba_io_bytes.argtypes = [vp, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]
        L.dmv_ba_get_solve_HdiF.argtypes = [vp, f32p]
        L.dmv_ba_adopt_frame.argtypes = [vp, C.c_int, vp]
        L.dmv_ba_batch_create.argtypes = [vp, C.c_int, C.POINTER(vp)]
        L.dmv_ba_batch_destroy.argtypes = [vp]
        L.dmv_ba_batch_gn_step.argtypes = [vp, vp, vp, vp, vp]
        L.dmv_ba_batch_set_timing.argtypes = [vp, C.c_int]
        L.dmv_ba_batch_last_kernel_ms.argtypes = [vp, C.POINTER(C.c_float)]
        L.dmv_ba_batch_bench.argtypes = [vp, vp, C.c_int, vp, vp, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]
        L.dmv_ct_create.argtypes = [C.POINTER(CTConfig), C.POINTER(vp)]
        L.dmv_ct_destroy.argtypes = [vp]
        L.dmv_ct_set_K.argtypes = [vp, C.c_int, C.c_float, C.c_float, C.c_float, C.c_float]
        L.dmv_ct_set_ref.argtypes = [vp, C.c_int, C.c_int, f32p, f32p, f32p, f32p]
        L.dmv_ct_make_coarse_depth.argtypes = [vp, C.c_int, f32p, f32p, f32p, f32p, i32p]
        L.dmv_ct_get_ref.argtypes = [vp, C.c_int, C.POINTER(C.c_int), vp, vp, vp, vp]
        L.dmv_ct_upload_new.argtypes = [vp, C.c_int, f32p]
        L.dmv_ct_upload_new_image.argtypes = [vp, f32p]
        L.dmv_ct_set_huber.argtypes = [vp, C.c_float]
        L.dmv_ct_calc_res_gs.argtypes = [vp, C.c_int, f32p, f32p, f32p, C.c_float, C.c_float, C.c_int, f64p, f64p, f64p, C.POINTER(C.c_int)]
        L.dmv_ct_track.argtypes = [vp, C.POINTER(CTTrackArgs), C.POINTER(CTTrackResult)]
        L.dmv_ct_init_points.argtypes = [vp, C.c_int, i32p, i32p, f32p, f32p, f32p, f32p, i32p]
        L.dmv_ps_default_settings.argtypes = [C.POINTER(PSSettings)]
        L.dmv_ps_default_settings.restype = None
        L.dmv_ct_select_pixels.argtypes = [vp, C.POINTER(PSArgs), vp, C.POINTER(PSResult)]
        L.dmv_ct_make_new_traces.argtypes = [vp, C.POINTER(PSArgs), C.c_int, C.POINTER(C.c_int), vp, vp, vp, vp, vp, vp, vp, C.POINTER(PSResult)]
        L.dmv_ct_trace_points.argtypes = [vp, C.POINTER(IPPoints), f32p, f32p, f32p, vp]
        L.dmv_ct_trace_points_multi.argtypes = [vp, C.c_int, vp, f32p, vp]
        L.dmv_ct_set_timing.argtypes = [vp, C.c_int]
        L.dmv_ct_last_timing.argtypes = [vp, f32p]
        L.dmv_ct_kernel_launch_count.argtypes = [vp, C.POINTER(C.c_longlong)]
        L.dmv_ct_last_point_evaluations.argtypes = [vp, C.POINTER(C.c_double)]
        L.dmv_ci_create.argtypes = [C.POINTER(CTConfig), C.POINTER(vp)]
        L.dmv_ci_destroy.argtypes = [vp]
        L.dmv_ci_set_K.argtypes = [vp, C.c_int, C.c_float, C.c_float, C.c_float, C.c_float]
        L.dmv_ci_upload_first.argtypes = [vp, C.c_int, vp]
        L.dmv_ci_upload_new.argtypes = [vp, C.c_int, vp]
        L.dmv_ci_set_points.argtypes = [vp, C.c_int, C.c_int, vp, vp, vp]
        L.dmv_ci_calc_res_and_gs.argtypes = [vp, C.POINTER(CIEvalArgs), C.POINTER(CIEvalResult)]
        L.dmv_ci_kernel_launch_count.argtypes = [vp, C.POINTER(C.c_longlong)]
        _LIB = L
    return _LIB


def check(rc):
    if rc != 0:
        raise DmvError(f"dmvio_b200 error {rc}: {lib().dmv_last_error().decode()}")


def _p(a):
    return None if a is None else a.ctypes.data_as(vp)


def _c(a, t):
    return None if a is None else np.ascontiguousarray(a, t)


class BA:
    """Thin RAII wrapper over a dmv_ba handle; argument names follow include/dmvio_b200.h."""

    def __init__(self, w, h, max_frames=8, max_points=8192, device=0, chunk_points=0):
        self.L = lib()
        cfg = BAConfig(w, h, max_frames, max_points, device, chunk_points)
        self.h = vp()
        check(self.L.dmv_ba_create(C.byref(cfg), C.byref(self.h)))
        self.w, self.hh = w, h
        self.nf = self.npts = self.nres = 0
        self._keep = {}

    def close(self):
        if self.h:
            self.L.dmv_ba_destroy(self.h)
            self.h = vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_params(self, huberTH=9.0, outlierTHSumComponent=2500.0, affineOptModeA=1e12, affineOptModeB=1e8):
        p = BAParams(huberTH, outlierTHSumComponent, affineOptModeA, affineOptModeB)
        check(self.L.dmv_ba_set_params(self.h, C.byref(p)))

    def upload_frame(self, slot, dI):
        check(self.L.dmv_ba_upload_frame(self.h, slot, _c(dI, np.float32).reshape(-1)))

    def upload_image(self, slot, img):
        check(self.L.dmv_ba_upload_image(self.h, slot, _c(img, np.float32).reshape(-1)))

    def adopt_frame(self, slot, ct):
        """level-0 plane of the frame resident in the coarse-tracker handle `ct` (capi.CT), device to device"""
        check(self.L.dmv_ba_adopt_frame(self.h, slot, ct.h))

    def set_window(self, nf, slots=None):
        s = _c(slots, np.int32)
        check(self.L.dmv_ba_set_window(self.h, nf, _p(s)))
        self.nf = nf
        self.N = 8 * nf + 4

    def set_points(self, host, u, v, idepth, idepth_zero, color, weights, priorF=None):
        self.npts = len(host)
        iz, pf = _c(idepth_zero, np.float32), _c(priorF, np.float32)
        check(self.L.dmv_ba_set_points(self.h, self.npts, _c(host, np.int32), _c(u, np.float32), _c(v, np.float32), _c(idepth, np.float32),
                                       _p(iz), _c(color, np.float32).reshape(-1), _c(weights, np.float32).reshape(-1), _p(pf)))

    def set_residuals(self, point, target, state=None, energy=None):
        self.nres = len(point)
        s, e = _c(state, np.int32), _c(energy, np.float32)
        check(self.L.dmv_ba_set_residuals(self.h, self.nres, _c(point, np.int32), _c(target, np.int32), _p(s), _p(e)))

    def set_adjoints(self, adHost, adTarget):
        check(self.L.dmv_ba_set_adjoints(self.h, _c(adHost, np.float64).reshape(-1), _c(adTarget, np.float64).reshape(-1)))

    def _state(self, calib8, precalc, TH, idepth=None, idepth_zero=None):
        st = BAState()
        k = _c(calib8, np.float32)
        for i in range(8):
            st.calib[i] = float(k[i])
        pc, th, idd, idz = _c(precalc, np.float32), _c(TH, np.float32), _c(idepth, np.float32), _c(idepth_zero, np.float32)
        self._keep = dict(pc=pc, th=th, idd=idd, idz=idz)
        st.precalc, st.frameEnergyTH, st.idepth, st.idepth_zero = _p(pc), _p(th), _p(idd), _p(idz)
        return st

    def set_state(self, calib8, precalc, TH, idepth=None, idepth_zero=None):
        st = self._state(calib8, precalc, TH, idepth, idepth_zero)
        check(self.L.dmv_ba_set_state(self.h, C.byref(st)))

    def linearize(self):
        r = BALinResult()
        check(self.L.dmv_ba_linearize(self.h, C.byref(r)))
        return dict(energy=r.energy, n_in=r.n_in, n_oob=r.n_oob, n_outlier=r.n_outlier)

    def gn_step(self, x, calib8, precalc, TH, idepth=None, idepth_zero=None):
        st = self._state(calib8, precalc, TH, idepth, idepth_zero)
        r = BALinResult()
        sums = np.zeros(3)
        xx = _c(x, np.float64)
        check(self.L.dmv_ba_gn_step(self.h, _p(xx), C.byref(st), C.byref(r), sums))
        return dict(energy=r.energy, n_in=r.n_in, n_oob=r.n_oob, n_outlier=r.n_outlier, sums=sums)

    def residual_outputs(self):
        n = self.nres
        o = dict(newState=np.zeros(n, np.int32), newEnergy=np.zeros(n, np.float32), newEnergyWithOutlier=np.zeros(n, np.float32),
                 centerProjectedTo=np.zeros((n, 3), np.float32), JpJdF=np.zeros((n, 8), np.float32))
        check(self.L.dmv_ba_get_residual_outputs(self.h, _p(o["newState"]), _p(o["newEnergy"]), _p(o["newEnergyWithOutlier"]),
                                                 _p(o["centerProjectedTo"]), _p(o["JpJdF"])))
        return o

    def target_energies(self, target):
        out = np.zeros(max(self.npts, 1), np.float32)
        n = C.c_int(0)
        check(self.L.dmv_ba_get_target_energies(self.h, target, out, len(out), C.byref(n)))
        return out[:n.value]

    def apply_res(self):
        check(self.L.dmv_ba_apply_res(self.h))

    def accumulate(self):
        N = self.N
        o = dict(HA=np.zeros((N, N)), bA=np.zeros(N), Hsc=np.zeros((N, N)), bsc=np.zeros(N))
        n = C.c_int(0)
        check(self.L.dmv_ba_accumulate(self.h, o["HA"].reshape(-1), o["bA"], o["Hsc"].reshape(-1), o["bsc"], C.byref(n)))
        o["resInA"] = n.value
        return o

    def point_outputs(self):
        n = self.npts
        o = dict(Hdd=np.zeros(n, np.float32), bd=np.zeros(n, np.float32), Hcd=np.zeros((n, 4), np.float32), HdiF=np.zeros(n, np.float32),
                 bdSumF=np.zeros(n, np.float32))
        check(self.L.dmv_ba_get_point_outputs(self.h, _p(o["Hdd"]), _p(o["bd"]), _p(o["Hcd"]), _p(o["HdiF"]), _p(o["bdSumF"])))
        return o

    def resubstitute(self, x, apply=False):
        step = np.zeros(self.npts, np.float32)
        sums = np.zeros(3)
        check(self.L.dmv_ba_resubstitute(self.h, _c(x, np.float64), _p(step), int(apply), sums))
        return step, sums

    def backup_points(self):
        check(self.L.dmv_ba_backup_points(self.h))

    def restore_points(self):
        check(self.L.dmv_ba_restore_points(self.h))

    def get_idepth(self):
        a, b = np.zeros(self.npts, np.float32), np.zeros(self.npts, np.float32)
        check(self.L.dmv_ba_get_idepth(self.h, _p(a), _p(b)))
        return a, b

    def last_timing(self):
        ms = np.zeros(4, np.float32)
        check(self.L.dmv_ba_last_timing(self.h, ms))
        return ms

    def bench_device(self, x=None, iters=100, flush_l2=True):
        a, b = C.c_float(0), C.c_float(0)
        xx = _c(x, np.float64)
        check(self.L.dmv_ba_bench_device(self.h, _p(xx), iters, int(flush_l2), C.byref(a), C.byref(b)))
        return a.value, b.value

    def launch_count(self):
        n = C.c_longlong(0)
        check(self.L.dmv_ba_kernel_launch_count(self.h, C.byref(n)))
        return n.value

    def set_timing(self, enable=True):
        check(self.L.dmv_ba_set_timing(self.h, int(enable)))

    def bench_e2e(self, x, calib8, precalc, TH, iters=100):
        st = self._state(calib8, precalc, TH)
        ms = C.c_double(0)
        xx = _c(x, np.float64)
        check(self.L.dmv_ba_bench_e2e(self.h, _p(xx), C.byref(st), iters, C.byref(ms)))
        return ms.value

    def io_bytes(self):
        a, b = C.c_longlong(0), C.c_longlong(0)
        check(self.L.dmv_ba_io_bytes(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def comm_init(self, nranks, rank, uid_bytes):
        buf = C.create_string_buffer(bytes(uid_bytes), 128)
        check(self.L.dmv_ba_comm_init(self.h, nranks, rank, C.cast(buf, vp)))


    def activate_points(self, host, P, RT, minObs=1):
        """FullSystem::optimizeImmaturePoint for the immature points P (dict as oracle.orc.ip_init) hosted in window frames `host`;
        returns status (1 activate / 0 keep / -1 delete), idepth, res_state (n, nf)."""
        n = len(P["u"])
        keep = [_c(host, np.int32)] + [_c(P[k], np.float32) for k in ("u", "v", "color", "weights", "energyTH", "idepth_min", "idepth_max")] + [_c(RT, np.float32)]
        status = np.zeros(n, np.int32); idepth = np.zeros(n, np.float32); rs = np.zeros((n, self.nf), np.int32)
        args = BAActivateArgs(n, *[a.ctypes.data for a in keep], int(minObs), status.ctypes.data, idepth.ctypes.data, rs.ctypes.data)
        check(self.L.dmv_ba_activate_points(self.h, C.byref(args)))
        return status, idepth, rs

    def reset_oob(self):
        check(self.L.dmv_ba_reset_oob(self.h))

    def drop_residuals(self, idx):
        """residuals leave the window (FullSystemOptimize.cpp:L196-214); the remaining ones keep their order"""
        idx = _c(idx, np.int32)
        check(self.L.dmv_ba_drop_residuals(self.h, len(idx), idx))
        self.nres -= len(np.unique(idx))

    def marginalize_points(self, pts, adHTdeltaF, cDeltaF, prior_fac=600.0 * 600.0):
        """flagPointsForRemoval's linearize / fixLinearizationF loop + marginalizePointsF for the listed points (dmv_ba_marginalize_points).
        Returns dict: M, Mb, Msc, Mbsc, H = M - Msc, b = Mb - Mbsc, resInM, ngood [n], rtz [nres, 8], isLinearized [nres]."""
        N = 8 * self.nf + 4
        pts = _c(pts, np.int32)
        ad = _c(adHTdeltaF, np.float32)
        assert ad.size == self.nf * self.nf * 8
        o = dict(M=np.zeros((N, N)), Mb=np.zeros(N), Msc=np.zeros((N, N)), Mbsc=np.zeros(N), ngood=np.zeros(len(pts), np.int32),
                 rtz=np.zeros((self.nres, 8), np.float32), isLinearized=np.zeros(self.nres, np.uint8))
        n = C.c_int32(0)
        args = BAMargArgs(len(pts), pts.ctypes.data, ad.ctypes.data, (C.c_float * 4)(*[float(x) for x in cDeltaF]), float(prior_fac),
                          o["M"].ctypes.data, o["Mb"].ctypes.data, o["Msc"].ctypes.data, o["Mbsc"].ctypes.data, C.addressof(n),
                          o["ngood"].ctypes.data, o["rtz"].ctypes.data, o["isLinearized"].ctypes.data)
        check(self.L.dmv_ba_marginalize_points(self.h, C.byref(args)))
        o["resInM"] = n.value
        o["H"], o["b"] = o["M"] - o["Msc"], o["Mb"] - o["Mbsc"]
        return o

    def p2p_export(self):
        """64-byte CUDA IPC handle of this rank's exchange inbox (all-gather it, then p2p_import)."""
        buf = C.create_string_buffer(64)
        check(self.L.dmv_ba_p2p_export(self.h, C.cast(buf, vp)))
        return bytes(buf.raw)

    def p2p_import(self, nranks, rank, handles):
        blob = b"".join(bytes(h) for h in handles)
        assert len(blob) == 64 * nranks
        buf = C.create_string_buffer(blob, len(blob))
        check(self.L.dmv_ba_p2p_import(self.h, nranks, rank, C.cast(buf, vp)))


def nccl_unique_id():
    buf = C.create_string_buffer(128)
    check(lib().dmv_nccl_unique_id(C.cast(buf, vp)))
    return bytes(buf.raw)


class CT:
    def __init__(self, w, h, levels, max_points=65536, device=0):
        self.L = lib()
        cfg = CTConfig(w, h, levels, max_points, device)
        self.h = vp()
        check(self.L.dmv_ct_create(C.byref(cfg), C.byref(self.h)))
        self.levels = levels
        self._wh = (w, h)

    def close(self):
        if self.h:
            self.L.dmv_ct_destroy(self.h)
            self.h = vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_K(self, lvl, fx, fy, cx, cy):
        check(self.L.dmv_ct_set_K(self.h, lvl, fx, fy, cx, cy))

    def set_ref(self, lvl, u, v, idepth, color):
        check(self.L.dmv_ct_set_ref(self.h, lvl, len(u), _c(u, np.float32), _c(v, np.float32), _c(idepth, np.float32), _c(color, np.float32)))

    def upload_new(self, lvl, dIp):
        check(self.L.dmv_ct_upload_new(self.h, lvl, _c(dIp, np.float32).reshape(-1)))

    def upload_new_image(self, img):
        check(self.L.dmv_ct_upload_new_image(self.h, _c(img, np.float32).reshape(-1)))

    def set_huber(self, th):
        check(self.L.dmv_ct_set_huber(self.h, th))

    def calc_res_gs(self, lvl, RKi, t, affLL, b0, cutoff, want_gs=True):
        res6 = np.zeros(6); H = np.zeros(64); b = np.zeros(8); n = C.c_int(0)
        check(self.L.dmv_ct_calc_res_gs(self.h, lvl, _c(RKi, np.float32).reshape(-1), _c(t, np.float32), _c(affLL, np.float32), b0, cutoff,
                                        int(want_gs), res6, H, b, C.byref(n)))
        return res6, H.reshape(8, 8), b, n.value

    def track(self, R, t, a, b, coarsest=None, minRes=None, ref_a=0.0, ref_b=0.0, ref_exposure=1.0, new_exposure=1.0, cutoff=20.0,
              affModeA=1e12, affModeB=1e8):
        """trackNewestCoarse in one launch (dmv_ct_track) from refToNew (R, t) and aff_g2l (a, b); minRes = minResForAbort (NaN = never abort).
        Returns the dmv_ct_track_result fields as a dict."""
        args = CTTrackArgs()
        args.R[:] = [float(x) for x in np.asarray(R, np.float64).reshape(-1)]
        args.t[:] = [float(x) for x in np.asarray(t, np.float64).reshape(-1)]
        args.a, args.b, args.ref_a, args.ref_b = a, b, ref_a, ref_b
        args.ref_exposure, args.new_exposure, args.coarseCutoffTH, args.affineOptModeA, args.affineOptModeB = ref_exposure, new_exposure, cutoff, affModeA, affModeB
        args.coarsestLvl = self.levels - 1 if coarsest is None else coarsest
        args.minResForAbort[:] = [float(x) for x in (np.full(5, np.nan) if minRes is None else np.asarray(minRes, np.float64))]
        r = CTTrackResult()
        check(self.L.dmv_ct_track(self.h, C.byref(args), C.byref(r)))
        return dict(R=np.array(r.R).reshape(3, 3), t=np.array(r.t), a=r.a, b=r.b, lastResiduals=np.array(r.lastResiduals), flow=np.array(r.flowIndicators),
                    good=r.trackingGood, iterations=r.iterations, evaluations=r.evaluations, status=r.status)

    def make_coarse_depth(self, Ku, Kv, new_idepth, HdiF):
        """makeCoarseDepthL0 on the device with the resident frame as the reference; returns pc_n per level"""
        pc_n = np.zeros(8, np.int32)
        check(self.L.dmv_ct_make_coarse_depth(self.h, len(Ku), _c(Ku, np.float32), _c(Kv, np.float32), _c(new_idepth, np.float32), _c(HdiF, np.float32), pc_n))
        return pc_n

    def get_ref(self, lvl):
        n = C.c_int(0)
        check(self.L.dmv_ct_get_ref(self.h, lvl, C.byref(n), None, None, None, None))
        a = [np.zeros(n.value, np.float32) for _ in range(4)]
        check(self.L.dmv_ct_get_ref(self.h, lvl, C.byref(n), *[x.ctypes.data for x in a]))
        return dict(u=a[0], v=a[1], idepth=a[2], color=a[3])

    @staticmethod
    def _ps_args(density, recursionsLeft, thFactor, potential, B, settings):
        keep = []
        a = PSArgs(float(density), int(recursionsLeft), float(thFactor), int(potential), None, None)
        if B is not None:
            Bc = _c(B, np.float32)
            assert Bc.size == 256
            keep.append(Bc)
            a.B256 = Bc.ctypes.data
        if settings is not None:
            st = PSSettings(float(settings[0]), float(settings[1]), float(settings[2]), int(settings[3]))
            keep.append(st)
            a.settings = C.pointer(st)
        return a, keep

    def select_pixels(self, density, recursionsLeft=1, thFactor=1.0, potential=3, B=None, settings=None, want_map=True):
        """PixelSelector::makeMaps on the resident frame -> (map as uint8 h x w or None, numHaveSub, potential after the call).
        B = CalibHessian::B (256 floats) or None; settings = (minGradHistCut, minGradHistAdd, gradDownweightPerLevel, selectDirectionDistribution)."""
        a, keep = self._ps_args(density, recursionsLeft, thFactor, potential, B, settings)
        r = PSResult()
        w, h = self._wh
        m = np.zeros((h, w), np.float32) if want_map else None
        check(self.L.dmv_ct_select_pixels(self.h, C.byref(a), None if m is None else m.ctypes.data, C.byref(r)))
        return (None if m is None else m.astype(np.uint8)), r.numHaveSub, r.currentPotential

    def make_new_traces(self, density, recursionsLeft=1, thFactor=1.0, potential=3, B=None, settings=None, cap=None):
        """FullSystem::makeNewTraces on the resident frame -> (dict u, v, type, color, weights, gradH, energyTH; numHaveSub; potential after)"""
        a, keep = self._ps_args(density, recursionsLeft, thFactor, potential, B, settings)
        w, h = self._wh
        cap = w * h if cap is None else cap
        P = dict(u=np.zeros(cap, np.int32), v=np.zeros(cap, np.int32), type=np.zeros(cap, np.float32), color=np.zeros((cap, 8), np.float32),
                 weights=np.zeros((cap, 8), np.float32), gradH=np.zeros((cap, 4), np.float32), energyTH=np.zeros(cap, np.float32))
        n = C.c_int(0)
        r = PSResult()
        check(self.L.dmv_ct_make_new_traces(self.h, C.byref(a), cap, C.byref(n), *[P[k].ctypes.data for k in ("u", "v", "type", "color", "weights",
                                                                                                               "gradH", "energyTH")], C.byref(r)))
        return {k: x[:n.value] for k, x in P.items()}, r.numHaveSub, r.currentPotential

    def init_points(self, u, v):
        """ImmaturePoint constructor on the resident frame; same dict layout as oracle.orc.ip_init."""
        n = len(u)
        P = dict(u=_c(u, np.float32), v=_c(v, np.float32), color=np.zeros((n, 8), np.float32), weights=np.zeros((n, 8), np.float32),
                 gradH=np.zeros((n, 4), np.float32), energyTH=np.zeros(n, np.float32))
        ok = np.zeros(n, np.int32)
        check(self.L.dmv_ct_init_points(self.h, n, _c(u, np.int32), _c(v, np.int32), P["color"].reshape(-1), P["weights"].reshape(-1), P["gradH"].reshape(-1),
                                        P["energyTH"], ok))
        P["ok"] = ok.astype(np.uint8)
        P.update(idepth_min=np.zeros(n, np.float32), idepth_max=np.full(n, np.nan, np.float32), quality=np.full(n, 10000, np.float32),
                 status=np.full(n, 5, np.int32), lastTraceUV=np.zeros((n, 2), np.float32), lastTracePixelInterval=np.zeros(n, np.float32))
        return P

    def trace_points(self, P, KRKi, Kt, aff):
        """ImmaturePoint::traceOn for the points of one host frame (dict of arrays as oracle.orc.ip_init returns) against the resident newest
        frame; returns a dict with the updated in/out fields (P itself is not modified)."""
        n = len(P["u"])
        keep = {k: _c(P[k], np.float32) for k in ("u", "v", "color", "weights", "gradH", "energyTH")}
        out = {"idepth_min": np.array(P["idepth_min"], np.float32, copy=True), "idepth_max": np.array(P["idepth_max"], np.float32, copy=True),
               "quality": np.array(P["quality"], np.float32, copy=True), "status": np.array(P["status"], np.int32, copy=True),
               "lastTraceUV": np.array(P["lastTraceUV"], np.float32, copy=True), "lastTracePixelInterval": np.array(P["lastTracePixelInterval"], np.float32, copy=True)}
        pts = IPPoints(n, *[a.ctypes.data for a in (keep["u"], keep["v"], keep["color"], keep["weights"], keep["gradH"], keep["energyTH"], out["idepth_min"],
                                                     out["idepth_max"], out["quality"], out["status"], out["lastTraceUV"], out["lastTracePixelInterval"])])
        check(self.L.dmv_ct_trace_points(self.h, C.byref(pts), _c(KRKi, np.float32).reshape(-1), _c(Kt, np.float32), _c(aff, np.float32), None))
        Q = dict(P)
        Q.update(out)
        return Q

    def trace_points_multi(self, sets):
        """sets = [(P, KRKi, Kt, aff), ...]: the immature points of several host keyframes in ONE launch (dmv_ct_trace_points_multi);
        returns the list of updated dicts."""
        ns = len(sets)
        arr = (IPPoints * ns)()
        keeps, outs = [], []
        tab = np.zeros((ns, 14), np.float32)
        for k, (P, KRKi, Kt, aff) in enumerate(sets):
            keep = {q: _c(P[q], np.float32) for q in ("u", "v", "color", "weights", "gradH", "energyTH")}
            out = {"idepth_min": np.array(P["idepth_min"], np.float32, copy=True), "idepth_max": np.array(P["idepth_max"], np.float32, copy=True),
                   "quality": np.array(P["quality"], np.float32, copy=True), "status": np.array(P["status"], np.int32, copy=True),
                   "lastTraceUV": np.array(P["lastTraceUV"], np.float32, copy=True), "lastTracePixelInterval": np.array(P["lastTracePixelInterval"], np.float32, copy=True)}
            arr[k] = IPPoints(len(P["u"]), *[a.ctypes.data for a in (keep["u"], keep["v"], keep["color"], keep["weights"], keep["gradH"], keep["energyTH"], out["idepth_min"],
                                                                      out["idepth_max"], out["quality"], out["status"], out["lastTraceUV"], out["lastTracePixelInterval"])])
            tab[k, :9] = np.asarray(KRKi, np.float32).reshape(-1); tab[k, 9:12] = Kt; tab[k, 12:14] = aff
            keeps.append(keep); outs.append(out)
        check(self.L.dmv_ct_trace_points_multi(self.h, ns, C.addressof(arr), tab.reshape(-1), None))
        res = []
        for (P, _, _, _), out in zip(sets, outs):
            Q = dict(P); Q.update(out); res.append(Q)
        return res

    def set_timing(self, enable=True):
        check(self.L.dmv_ct_set_timing(self.h, int(enable)))

    def last_timing(self):
        ms = np.zeros(4, np.float32)
        check(self.L.dmv_ct_last_timing(self.h, ms))
        return ms

    def launch_count(self):
        n = C.c_longlong(0)
        check(self.L.dmv_ct_kernel_launch_count(self.h, C.byref(n)))
        return n.value


class CI:
    """CoarseInitializer::calcResAndGS on the device (include/dmvio_b200.h, dmv_ci_*)"""

    def __init__(self, w, h, levels, max_points=16384, device=0):
        self.L = lib()
        cfg = CTConfig(w, h, levels, max_points, device)   # dmv_ci_config has the same layout
        self.h = vp()
        check(self.L.dmv_ci_create(C.byref(cfg), C.byref(self.h)))
        self.levels = levels

    def close(self):
        if self.h:
            self.L.dmv_ci_destroy(self.h)
            self.h = vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_K(self, lvl, fx, fy, cx, cy):
        check(self.L.dmv_ci_set_K(self.h, lvl, C.c_float(fx), C.c_float(fy), C.c_float(cx), C.c_float(cy)))

    def upload_first(self, lvl, dIp):
        check(self.L.dmv_ci_upload_first(self.h, lvl, _p(_c(dIp, np.float32).reshape(-1))))

    def upload_new(self, lvl, dIp):
        check(self.L.dmv_ci_upload_new(self.h, lvl, _p(_c(dIp, np.float32).reshape(-1))))

    def set_points(self, lvl, u, v, outlierTH):
        check(self.L.dmv_ci_set_points(self.h, lvl, len(u), _p(_c(u, np.float32)), _p(_c(v, np.float32)), _p(_c(outlierTH, np.float32))))
        self._n = getattr(self, "_n", {})
        self._n[lvl] = len(u)

    def calc_res_and_gs(self, lvl, RKi, t, t_log, r2new_aff, idepth_new, isGood, energy2, iR, huberTH=9.0, alphaK=2.5 * 2.5, alphaW=150.0 * 150.0,
                        couplingWeight=1.0, wzpx=0.0, wzpy=0.0):
        n = self._n[lvl]
        a = CIEvalArgs()
        a.level = lvl
        a.RKi[:] = [float(x) for x in np.asarray(RKi, np.float32).reshape(-1)]
        a.t_d[:] = [float(x) for x in t]
        a.t_log[:] = [float(x) for x in t_log]
        a.r2new_aff[:] = [float(np.float32(x)) for x in r2new_aff]
        a.huberTH, a.alphaK, a.alphaW, a.couplingWeight, a.weightZeroPriorX, a.weightZeroPriorY = huberTH, alphaK, alphaW, couplingWeight, wzpx, wzpy
        ins = [_c(idepth_new, np.float32), _c(isGood, np.uint8), _c(energy2, np.float32).reshape(-1), _c(iR, np.float32)]
        a.idepth_new, a.isGood, a.energy2, a.iR = [x.ctypes.data for x in ins]
        o = dict(isGood_new=np.zeros(n, np.uint8), energy_new=np.zeros((n, 2), np.float32), maxstep=np.zeros(n, np.float32),
                 lastHessian_new=np.zeros(n, np.float32), Jb=np.zeros((n, 10), np.float32))
        a.isGood_new, a.energy_new2, a.maxstep, a.lastHessian_new, a.JbBuffer_new10 = [o[k].ctypes.data for k in ("isGood_new", "energy_new", "maxstep", "lastHessian_new", "Jb")]
        r = CIEvalResult()
        check(self.L.dmv_ci_calc_res_and_gs(self.h, C.byref(a), C.byref(r)))
        o.update(H=np.array(r.H, np.float32).reshape(8, 8), b=np.array(r.b, np.float32), Hsc=np.array(r.Hsc, np.float32).reshape(8, 8),
                 bsc=np.array(r.bsc, np.float32), res=np.array(r.res3, np.float32), alphaOpt=float(r.alphaOpt), n_good_new=int(r.n_good_new))
        return o
