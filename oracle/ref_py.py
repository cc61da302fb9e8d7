"""ctypes binding of oracle/_ref/libphovo_ref.so: the reference's OWN
CPhotoconsistencyOdometryAnalytic<unsigned char,double>, compiled unmodified from
$REF/phovo/include against the OpenCV/Eigen stand-ins in oracle/shim (oracle/Makefile).

TEST INFRASTRUCTURE.  Used to pin the C oracle (and through it the CUDA path) against the reference
source itself, and to mint tests/golden/ref_*.npz.  The library is built where REF names a checkout
of the original project; it is git-ignored, and the tests that need it skip without it.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(_HERE, "_ref", "libphovo_ref.so")


def available():
    ref = os.environ.get("REF")
    if not os.path.exists(LIB) and ref and os.path.isdir(os.path.join(ref, "phovo", "include")):
        subprocess.call(["make", "-s", "-C", _HERE, "ref"], stdout=subprocess.DEVNULL)
    return os.path.exists(LIB)


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not available():
            raise RuntimeError("oracle/_ref/libphovo_ref.so is not built (set REF to a checkout of the original project)")
        L = C.CDLL(LIB)
        vp, dp = C.c_void_p, C.POINTER(C.c_double)
        L.ref_create.restype = vp
        L.ref_destroy.argtypes = [vp]
        L.ref_read_config.argtypes = [vp, C.c_char_p]
        L.ref_set_depth_range.argtypes = [vp, C.c_double, C.c_double]
        L.ref_set_intrinsics.argtypes = [vp, dp]
        L.ref_set_source.argtypes = [vp, vp, vp, C.c_int, C.c_int]
        L.ref_set_target.argtypes = [vp, vp, C.c_int, C.c_int]
        L.ref_set_initial_state.argtypes = [vp, dp]
        L.ref_optimize.argtypes = [vp]
        L.ref_get_state.argtypes = [vp, dp]
        L.ref_get_rt.argtypes = [vp, dp]
        L.ref_num_iterations.argtypes = [vp]
        L.ref_get_iteration.argtypes = [vp, C.c_int, C.POINTER(C.c_int), dp, dp]
        L.ref_warp_image.argtypes = [vp, vp, C.c_int, C.c_int, dp, dp, vp]
        L.refbi_create.restype = vp
        L.refbi_destroy.argtypes = [vp]
        L.refbi_read_config.argtypes = [vp, C.c_char_p]
        L.refbi_set_intrinsics.argtypes = [vp, dp]
        L.refbi_set_source.argtypes = [vp, vp, vp, C.c_int, C.c_int]
        L.refbi_set_target.argtypes = [vp, vp, vp, C.c_int, C.c_int]
        L.refbi_set_initial_state.argtypes = [vp, dp]
        L.refbi_optimize.argtypes = [vp]
        L.refbi_get_state.argtypes = [vp, dp]
        L.refbi_num_iterations.argtypes = [vp]
        L.refbi_get_iteration.argtypes = [vp, C.c_int, C.POINTER(C.c_int), dp, dp]
        L.refce_create.restype = vp
        L.refce_destroy.argtypes = [vp]
        L.refce_read_config.argtypes = [vp, C.c_char_p]
        L.refce_set_intrinsics.argtypes = [vp, dp]
        L.refce_set_source.argtypes = [vp, vp, vp, C.c_int, C.c_int]
        L.refce_set_target.argtypes = [vp, vp, C.c_int, C.c_int]
        L.refce_set_initial_state.argtypes = [vp, dp]
        L.refce_get_state.argtypes = [vp, dp]
        L.refce_evaluate.argtypes = [vp, C.c_int, dp, dp, dp]
        L.refce_evaluate.restype = C.c_int
        L.refce_optimize.argtypes = [vp]
        L.refce_num_iter_stats.argtypes = [vp]
        L.refce_get_iter_stats.argtypes = [vp, C.c_int, vp]
        _lib = L
    return _lib


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


class Reference:
    """The reference solver object, driven with the call sequence of the reference apps
    (PhotoconsistencyFrameAlignment.cpp:90-105)."""

    def __init__(self, config_yaml, K):
        self.L = lib()
        self.h = self.L.ref_create()
        self.L.ref_read_config(self.h, os.fsencode(config_yaml))
        self.K = np.ascontiguousarray(K, dtype=np.float64).reshape(9)
        self.L.ref_set_intrinsics(self.h, _dp(self.K))

    def __del__(self):
        if getattr(self, "h", None):
            self.L.ref_destroy(self.h)
            self.h = None

    def align(self, gray0, depth0, gray1, state0=None):
        g0 = np.ascontiguousarray(gray0, dtype=np.uint8)
        d0 = np.ascontiguousarray(depth0, dtype=np.float64)
        g1 = np.ascontiguousarray(gray1, dtype=np.uint8)
        r, c = g0.shape
        self.L.ref_set_source(self.h, g0.ctypes.data, d0.ctypes.data, r, c)
        self.L.ref_set_target(self.h, g1.ctypes.data, r, c)
        s0 = np.zeros(6) if state0 is None else np.ascontiguousarray(state0, dtype=np.float64)
        self.L.ref_set_initial_state(self.h, _dp(s0))
        self.L.ref_optimize(self.h)
        s = np.zeros(6)
        self.L.ref_get_state(self.h, _dp(s))
        rt = np.zeros(16)
        self.L.ref_get_rt(self.h, _dp(rt))
        iters = []
        for i in range(self.L.ref_num_iterations(self.h)):
            n = C.c_int()
            H, g = np.zeros(36), np.zeros(6)
            self.L.ref_get_iteration(self.h, i, C.byref(n), _dp(H), _dp(g))
            iters.append(dict(n=n.value, H=H.reshape(6, 6), g=g))
        return s, rt.reshape(4, 4), iters


class ReferenceBiObjective:
    """The reference's photometric + depth solver (CPhotoconsistencyOdometryBiObjective.h), driven like
    the apps drive it; the target frame's depth IS used here."""

    def __init__(self, config_yaml, K):
        self.L = lib()
        self.h = self.L.refbi_create()
        self.L.refbi_read_config(self.h, os.fsencode(config_yaml))
        self.K = np.ascontiguousarray(K, dtype=np.float64).reshape(9)
        self.L.refbi_set_intrinsics(self.h, _dp(self.K))

    def __del__(self):
        if getattr(self, "h", None):
            self.L.refbi_destroy(self.h)
            self.h = None

    def align(self, gray0, depth0, gray1, depth1, state0=None):
        g0 = np.ascontiguousarray(gray0, dtype=np.uint8)
        d0 = np.ascontiguousarray(depth0, dtype=np.float64)
        g1 = np.ascontiguousarray(gray1, dtype=np.uint8)
        d1 = np.ascontiguousarray(depth1, dtype=np.float64)
        r, c = g0.shape
        self.L.refbi_set_source(self.h, g0.ctypes.data, d0.ctypes.data, r, c)
        self.L.refbi_set_target(self.h, g1.ctypes.data, d1.ctypes.data, r, c)
        s0 = np.zeros(6) if state0 is None else np.ascontiguousarray(state0, dtype=np.float64)
        self.L.refbi_set_initial_state(self.h, _dp(s0))
        self.L.refbi_optimize(self.h)
        s = np.zeros(6)
        self.L.refbi_get_state(self.h, _dp(s))
        iters = []
        for i in range(self.L.refbi_num_iterations(self.h)):
            n = C.c_int()
            H, g = np.zeros(36), np.zeros(6)
            self.L.refbi_get_iteration(self.h, i, C.byref(n), _dp(H), _dp(g))
            iters.append(dict(n=n.value, H=H.reshape(6, 6), g=g))
        return s, iters


class ReferenceCeres:
    """The reference's Ceres-based solver class (CPhotoconsistencyOdometryCeres.h) with ITS residual
    functor and sampler (third_party/sample.h, jet_extras.h), compiled unmodified against the
    ceres::Jet / ceres::Problem stand-ins of oracle/shim/ceres.  Ceres' minimiser is absent:
    evaluate() pins residuals + Jacobians; optimize() runs the oracle's restated LM on that functor."""

    def __init__(self, config_yaml, K):
        self.L = lib()
        self.h = self.L.refce_create()
        self.L.refce_read_config(self.h, os.fsencode(config_yaml))
        self.K = np.ascontiguousarray(K, dtype=np.float64).reshape(9)
        self.L.refce_set_intrinsics(self.h, _dp(self.K))

    def __del__(self):
        if getattr(self, "h", None):
            self.L.refce_destroy(self.h)
            self.h = None

    def set_frames(self, gray0, depth0, gray1):
        g0 = np.ascontiguousarray(gray0, dtype=np.uint8)
        d0 = np.ascontiguousarray(depth0, dtype=np.float64)
        g1 = np.ascontiguousarray(gray1, dtype=np.uint8)
        r, c = g0.shape
        self.L.refce_set_source(self.h, g0.ctypes.data, d0.ctypes.data, r, c)
        self.L.refce_set_target(self.h, g1.ctypes.data, r, c)

    def evaluate(self, level_shape, state, want_jacobian=True):
        """Residuals (rows x cols) and Jacobian (rows*cols x 6) of the level with that shape at `state`:
        the reference functor on T = Jet<double,6> (or on T = double when want_jacobian is False)."""
        n = int(level_shape[0]) * int(level_shape[1])
        st = np.ascontiguousarray(state, dtype=np.float64)
        res = np.zeros(n)
        jac = np.zeros((n, 6)) if want_jacobian else None
        ok = self.L.refce_evaluate(self.h, n, _dp(st), _dp(res), _dp(jac) if want_jacobian else None)
        if not ok:
            raise RuntimeError("no optimised level with %d pixels in this configuration" % n)
        return res.reshape(level_shape), jac

    def optimize(self, state0=None):
        import oracle_py
        s0 = np.zeros(6) if state0 is None else np.ascontiguousarray(state0, dtype=np.float64)
        self.L.refce_set_initial_state(self.h, _dp(s0))
        self.L.refce_optimize(self.h)
        s = np.zeros(6)
        self.L.refce_get_state(self.h, _dp(s))
        log = []
        for i in range(self.L.refce_num_iter_stats(self.h)):
            e = oracle_py.IterStats()
            self.L.refce_get_iter_stats(self.h, i, C.addressof(e))
            log.append(e.as_dict())
        return s, log


def warp_image(gray, depth, rt, K):
    """phovo::warpImage (CPhotoconsistencyOdometry.h:73-134), level 0."""
    L = lib()
    g = np.ascontiguousarray(gray, dtype=np.uint8)
    d = np.ascontiguousarray(depth, dtype=np.float64)
    out = np.zeros_like(g)
    L.ref_warp_image(g.ctypes.data, d.ctypes.data, g.shape[0], g.shape[1],
                     _dp(np.ascontiguousarray(rt, dtype=np.float64).reshape(16)),
                     _dp(np.ascontiguousarray(K, dtype=np.float64).reshape(9)), out.ctypes.data)
    return out
