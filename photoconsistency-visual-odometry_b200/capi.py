"""ctypes binding of libphovo_b200.so -- the C ABI declared in include/phovo_b200.h.

This is the only way Python reaches the CUDA path; there is no CPU fallback: loading fails loudly
if the library has not been built, and `phovo_create` fails if no CUDA device is present.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libphovo_b200.so")
MAXL = 10

OK, E_INVALID, E_CUDA, E_CONFIG, E_NOMEM, E_UNSUPPORTED, E_NUMERIC = 0, -1, -2, -3, -4, -5, -6
MODE_ANALYTIC_REF, MODE_ANALYTIC_FIXED, MODE_CERES, MODE_BIOBJECTIVE = 0, 1, 2, 3
DEPTH_F64, DEPTH_F32, DEPTH_U16 = 0, 1, 2


class Config(C.Structure):
    """`phovo_config`"""
    _fields_ = [
        ("mode", C.c_int32), ("num_levels", C.c_int32),
        ("blur_filter_size", C.c_int32 * MAXL), ("max_num_iterations", C.c_int32 * MAXL),
        ("grad_scale", C.c_double * MAXL), ("lambda_step", C.c_double * MAXL),
        ("min_gradient_norm", C.c_double * MAXL),
        ("min_depth", C.c_double), ("max_depth", C.c_double),
        ("visualize_iterations", C.c_int32),
        ("function_tolerance", C.c_double * MAXL), ("gradient_tolerance", C.c_double * MAXL),
        ("parameter_tolerance", C.c_double * MAXL),
        ("initial_trust_region_radius", C.c_double * MAXL),
        ("max_trust_region_radius", C.c_double * MAXL),
        ("min_trust_region_radius", C.c_double * MAXL),
        ("min_relative_decrease", C.c_double * MAXL),
        ("num_threads", C.c_int32), ("num_linear_solver_threads", C.c_int32),
        ("minimizer_progress_to_stdout", C.c_int32), ("reserved", C.c_int32),
    ]


class IterStats(C.Structure):
    """`phovo_iter_stats`"""
    _fields_ = [
        ("level", C.c_int32), ("iteration", C.c_int32), ("num_valid", C.c_int32), ("accepted", C.c_int32),
        ("H", C.c_double * 21), ("g", C.c_double * 6), ("grad_norm", C.c_double), ("cost", C.c_double),
        ("radius", C.c_double), ("state_in", C.c_double * 6), ("state_out", C.c_double * 6),
    ]

    def as_dict(self):
        return dict(level=self.level, iteration=self.iteration, num_valid=self.num_valid,
                    accepted=self.accepted, H=np.array(self.H[:]), g=np.array(self.g[:]),
                    grad_norm=self.grad_norm, cost=self.cost, radius=self.radius,
                    state_in=np.array(self.state_in[:]), state_out=np.array(self.state_out[:]))


# name -> (restype, argtypes); every symbol include/phovo_b200.h declares
_vp, _dp, _ip = C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int32)
_cfgp, _stp = C.POINTER(Config), C.POINTER(IterStats)
SIGNATURES = {
    "phovo_create": (C.c_int, [C.c_int, C.POINTER(_vp)]),
    "phovo_destroy": (C.c_int, [_vp]),
    "phovo_last_error": (C.c_char_p, [_vp]),
    "phovo_version": (C.c_char_p, []),
    "phovo_config_default": (C.c_int, [_cfgp]),
    "phovo_set_config": (C.c_int, [_vp, _cfgp]),
    "phovo_get_config": (C.c_int, [_vp, _cfgp]),
    "phovo_load_config_yaml": (C.c_int, [_vp, C.c_char_p]),
    "phovo_parse_config_yaml": (C.c_int, [C.c_char_p, _cfgp, C.c_char_p, C.c_size_t]),
    "phovo_set_mode": (C.c_int, [_vp, C.c_int]),
    "phovo_set_depth_range": (C.c_int, [_vp, C.c_double, C.c_double]),
    "phovo_set_intrinsics": (C.c_int, [_vp, _dp]),
    "phovo_set_source": (C.c_int, [_vp, _vp, C.c_size_t, _vp, C.c_int, C.c_size_t, C.c_double, C.c_int, C.c_int]),
    "phovo_set_target": (C.c_int, [_vp, _vp, C.c_size_t, C.c_int, C.c_int]),
    "phovo_promote_target_to_source": (C.c_int, [_vp, _vp, C.c_int, C.c_size_t, C.c_double]),
    "phovo_set_target_depth": (C.c_int, [_vp, _vp, C.c_int, C.c_size_t, C.c_double]),
    "phovo_set_initial_state": (C.c_int, [_vp, _dp]),
    "phovo_optimize": (C.c_int, [_vp]),
    "phovo_get_state": (C.c_int, [_vp, _dp]),
    "phovo_get_rt": (C.c_int, [_vp, _dp]),
    "phovo_state_to_rt": (None, [_dp, _dp]),
    "phovo_warp_image": (C.c_int, [_vp, _vp, C.c_size_t, _vp, C.c_int, C.c_size_t, C.c_double, C.c_int, C.c_int, _dp, _dp, C.c_int,
                                   _vp, C.c_size_t, _vp, C.c_size_t, _vp, C.c_size_t]),
    "phovo_num_iter_stats": (C.c_int, [_vp]),
    "phovo_get_iter_stats": (C.c_int, [_vp, C.c_int, _stp]),
    "phovo_get_level_image": (C.c_int, [_vp, C.c_int, C.c_int, _vp, _ip, _ip]),
    "phovo_eval_normal_equations": (C.c_int, [_vp, C.c_int, _dp, _stp]),
    "phovo_eval_residuals": (C.c_int, [_vp, C.c_int, _dp, _vp, _vp]),
    "phovo_get_timings": (C.c_int, [_vp, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "phovo_launch_count": (C.c_int64, [_vp]),
    "phovo_set_stream": (C.c_int, [_vp, _vp]),
    "phovo_set_use_graph": (C.c_int, [_vp, C.c_int]),
    "phovo_last_optimize_used_graph": (C.c_int, [_vp]),
    "phovo_set_execution": (C.c_int, [_vp, C.c_int]),
    "phovo_last_optimize_path": (C.c_int, [_vp]),
    "phovo_graph_error": (C.c_char_p, [_vp]),
    "phovo_set_build_all_levels": (C.c_int, [_vp, C.c_int]),
    "phovo_batch_align": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, _vp, _vp, C.c_int, C.c_double, _vp, _vp, _vp, _vp]),
    "phovo_batch_align_with_target_depth": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, _vp, _vp, C.c_int, C.c_double, _vp, _vp, _vp, _vp, _vp]),
    "phovo_batch_last_path": (C.c_int, [_vp]),
    "phovo_batch_align_device": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, _vp, _vp, C.c_int, C.c_double, _vp, _vp, _vp, _vp]),
    "phovo_batch_align_device_with_target_depth": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, _vp, _vp, C.c_int, C.c_double, _vp, _vp,
                                                             _vp, _vp, _vp]),
    "phovo_batch_set_record_stats": (C.c_int, [_vp, C.c_int]),
    "phovo_batch_get_iter_stats": (C.c_int, [_vp, C.c_int, C.c_int, _stp]),
    "phovo_batch_num_iter_stats": (C.c_int, [_vp, C.c_int]),
    "phovo_batch_set_debug_flags": (C.c_int, [_vp, C.c_int]),
    "phovo_batch_warp_image": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, _vp, _vp, C.c_int, C.c_double, _vp, _dp, C.c_int, _vp,
                                         _vp, _vp, _vp, _vp]),
    "phovo_batch_eval_normal_equations": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, _vp, _vp, C.c_int, C.c_double, _vp, _vp,
                                                    C.c_int, _vp, _vp, _vp, _vp]),
    "phovo_batch_eval_normal_equations_with_target_depth": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, _vp, _vp, C.c_int, C.c_double,
                                                                      _vp, _vp, _vp, C.c_int, _vp, _vp, _vp, _vp]),
    "phovo_batch_release_memory": (C.c_int, [_vp]),
    "phovo_batch_get_last_h2d_bytes": (C.c_int, [_vp, C.POINTER(C.c_uint64)]),
    "phovo_synchronize": (C.c_int, [_vp]),
    "phovo_batch_get_kernel_times": (C.c_int, [_vp, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "phovo_shard_configure": (C.c_int, [_vp, C.c_int, C.c_int]),
    "phovo_shard_buffer": (C.c_int, [_vp, C.POINTER(_vp)]),
    "phovo_shard_read_buffer": (C.c_int, [_vp, _dp]),
    "phovo_shard_write_buffer": (C.c_int, [_vp, _dp]),
    "phovo_shard_begin": (C.c_int, [_vp]),
    "phovo_shard_begin_level": (C.c_int, [_vp, C.c_int]),
    "phovo_shard_partial": (C.c_int, [_vp]),
    "phovo_shard_step": (C.c_int, [_vp, _ip]),
    "phovo_shard_finish": (C.c_int, [_vp]),
    "phovo_shard_peer_export": (C.c_int, [_vp, _vp]),
    "phovo_shard_peer_import": (C.c_int, [_vp, C.c_int, _vp]),
    "phovo_shard_partial_exchange": (C.c_int, [_vp]),
    "phovo_shard_optimize": (C.c_int, [_vp, C.c_int]),
}

_lib = None


class PhovoError(RuntimeError):
    def __init__(self, code, text):
        super().__init__("phovo error %d: %s" % (code, text))
        self.code = code


def lib():
    """Load libphovo_b200.so (no CPU fallback: raises if it has not been built)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("libphovo_b200.so is not built (run __graft_entry__.build() or "
                              "python photoconsistency-visual-odometry_b200/build.py); there is no CPU fallback")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


def _ptr(a):
    """data pointer of a numpy array, torch tensor (host or device) or raw int."""
    if a is None:
        return None
    if isinstance(a, int):
        return a
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    if hasattr(a, "data_ptr"):
        return a.data_ptr()
    raise TypeError(type(a))


def default_config():
    cfg = Config()
    lib().phovo_config_default(C.byref(cfg))
    return cfg


def parse_config_yaml(path):
    cfg = default_config()
    err = C.create_string_buffer(512)
    rc = lib().phovo_parse_config_yaml(os.fsencode(path), C.byref(cfg), err, 512)
    if rc != OK:
        raise PhovoError(rc, err.value.decode())
    return cfg


def state_to_rt(state):
    s = np.ascontiguousarray(state, dtype=np.float64)
    out = np.zeros(16)
    lib().phovo_state_to_rt(s.ctypes.data_as(_dp), out.ctypes.data_as(_dp))
    return out.reshape(4, 4)
