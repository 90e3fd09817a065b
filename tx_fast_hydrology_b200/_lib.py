"""ctypes binding of libtxh.so (the C ABI declared in include/txh.h).

This is the whole Python<->CUDA boundary: plain pointers and sizes, no torch
types.  There is no CPU fallback: if the library is missing or no CUDA device
is visible, compute entry points raise.
"""
import ctypes
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libtxh.so")

c_i64 = ctypes.c_int64
c_i32 = ctypes.c_int32
c_f64 = ctypes.c_double
c_vp = ctypes.c_void_p
p_i64 = ctypes.POINTER(ctypes.c_int64)
p_i32 = ctypes.POINTER(ctypes.c_int32)
p_u32 = ctypes.POINTER(ctypes.c_uint32)
p_f64 = ctypes.POINTER(ctypes.c_double)

# name -> (restype, argtypes); every symbol include/txh.h declares
SIGNATURES = {
    "txh_last_error": (ctypes.c_char_p, []),
    "txh_version": (ctypes.c_int, []),
    "txh_device_count": (ctypes.c_int, []),
    "txh_create": (ctypes.c_int, [c_i64, p_i64, p_i32, ctypes.POINTER(c_vp)]),
    "txh_destroy": (None, [c_vp]),
    "txh_n": (c_i64, [c_vp]),
    "txh_get_indegree": (ctypes.c_int, [c_vp, p_i64]),
    "txh_get_headwaters": (ctypes.c_int, [c_vp, p_i64, p_i64]),
    "txh_get_levels": (ctypes.c_int, [c_vp, p_i64, p_i64]),
    "txh_get_level_order": (ctypes.c_int, [c_vp, p_i64, p_i64]),
    "txh_get_chains": (ctypes.c_int, [c_vp, p_i64, p_i64, p_i64, p_i64]),
    "txh_get_paths": (ctypes.c_int, [c_vp, p_i64, p_i64]),
    "txh_get_visit_order": (ctypes.c_int, [c_vp, p_i64]),
    "txh_get_schedule_info": (ctypes.c_int, [c_vp, p_i64]),
    "txh_get_schedule": (ctypes.c_int, [c_vp, p_i64, p_i32, p_i32, p_u32, p_u32]),
    "txh_get_window_info": (ctypes.c_int, [c_vp, p_i64]),
    "txh_get_window_schedule": (ctypes.c_int, [c_vp, p_i32, p_u32, p_u32, p_i32]),
    "txh_get_lane_info": (ctypes.c_int, [c_vp, c_i64, c_i64, p_i64]),
    "txh_get_lane_schedule": (ctypes.c_int, [c_vp, c_i64, p_i32, p_i32, p_i32]),
    "txh_scan_nhd_geojson": (ctypes.c_int, [ctypes.c_char_p, c_i64, p_i64, p_i64, p_f64, p_i64]),
    "txh_compute_coeffs": (ctypes.c_int, [c_vp, p_f64, p_f64, c_f64, p_f64, p_f64, p_f64, p_f64]),
    "txh_set_coeffs": (ctypes.c_int, [c_vp, p_f64, p_f64, p_f64, p_f64]),
    "txh_row_stride": (c_i64, [c_i64]),
    "txh_pack_host": (ctypes.c_int, [c_vp, p_f64, c_i64, ctypes.c_int, c_vp, c_vp]),
    "txh_unpack_host": (ctypes.c_int, [c_vp, c_vp, c_i64, ctypes.c_int, p_f64, c_vp]),
    "txh_pack_dev": (ctypes.c_int, [c_vp, c_vp, c_i64, c_vp, c_vp]),
    "txh_unpack_dev": (ctypes.c_int, [c_vp, c_vp, c_i64, c_vp, c_vp]),
    "txh_gather_rows": (ctypes.c_int, [c_vp, c_vp, c_i64, p_i64, c_i64, c_vp, c_vp]),
    "txh_init_inflows": (ctypes.c_int, [c_vp, c_vp, c_vp, c_i64, c_vp]),
    "txh_forcing_create": (ctypes.c_int, [c_vp, c_i64, p_f64, c_vp, c_i64, c_vp, c_vp, ctypes.POINTER(c_vp)]),
    "txh_forcing_update": (ctypes.c_int, [c_vp, p_f64, c_vp, c_vp, c_vp]),
    "txh_forcing_update_async": (ctypes.c_int, [c_vp, p_f64, c_vp, c_vp, c_vp]),
    "txh_forcing_wait": (ctypes.c_int, [c_vp]),
    "txh_forcing_destroy": (None, [c_vp]),
    "txh_route_run": (ctypes.c_int, [c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, c_i64, c_i64, ctypes.c_int,
                                     p_i64, c_i64, c_i64, c_vp, c_vp]),
    "txh_route_step": (ctypes.c_int, [c_vp, c_vp, c_vp, c_i64, c_vp, c_vp]),
    "txh_route_step_levels": (ctypes.c_int, [c_vp, c_vp, c_vp, c_i64, c_vp, c_vp]),
    "txh_route_apply": (ctypes.c_int, [c_vp, c_vp, c_vp, c_i64, c_vp]),
    "txh_apply_gain": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "txh_enkf_stats": (ctypes.c_int, [c_vp, c_vp, c_i64, p_i64, c_i64, c_f64, c_vp, c_vp, c_vp]),
    "txh_set_stats_output": (ctypes.c_int, [c_vp, c_vp, c_f64]),
    "txh_enkf_work_size": (c_i64, [c_i64, c_i64]),
    "txh_enkf_solve": (ctypes.c_int, [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, p_i64, c_vp, c_vp, c_vp, ctypes.c_int,
                                      c_vp, c_vp, c_vp, c_vp]),
    "txh_enkf_apply": (ctypes.c_int, [c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, c_i64, c_i64, c_i64, c_vp, c_vp, p_i64, c_i64,
                                      c_vp, c_vp, c_vp, c_vp]),
    "txh_enkf_apply_peers": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, ctypes.POINTER(c_vp), c_i64, c_i64, c_i64, c_vp,
                                            c_vp, p_i64, c_i64, c_vp, c_vp, c_vp, c_vp]),
    "txh_run_assimilating": (ctypes.c_int, [c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, c_i64, c_i64, c_i64, ctypes.c_int,
                                            p_i64, c_i64, c_vp, c_vp, c_vp, c_vp, ctypes.c_int, c_vp, c_vp, c_vp, c_vp,
                                            c_vp, c_vp, c_i64, c_vp, c_vp]),
    "txh_run_assimilating_rec": (ctypes.c_int, [c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, c_i64, c_i64, c_i64, ctypes.c_int,
                                                p_i64, c_i64, c_vp, c_vp, c_vp, c_vp, ctypes.c_int, c_vp, c_vp, c_vp, c_vp,
                                                c_vp, c_vp, c_i64, c_vp, p_i64, c_i64, c_i64, c_vp, c_vp, c_vp]),
    "txh_get_route_timings": (ctypes.c_int, [c_vp, p_f64, c_i64, p_i64]),
    "txh_set_transform_history": (ctypes.c_int, [c_vp, c_vp, c_i64]),
    "txh_enks_work_size": (c_i64, [c_i64, c_i64]),
    "txh_enks_smooth": (ctypes.c_int, [c_i64, c_i64, c_i64, c_vp, c_i64, c_i64, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp]),
    "txh_dgemm": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, c_i64, c_i64, c_i64, c_f64, c_vp, c_i64, c_vp, c_i64,
                                 c_f64, c_vp, c_i64, c_vp]),
    "txh_spd_solve": (ctypes.c_int, [c_i64, c_i64, c_vp, c_vp, c_vp]),
    "txh_inverse": (ctypes.c_int, [c_i64, c_vp, c_vp, c_vp]),
    "txh_kf_work_size": (c_i64, [c_vp, c_i64]),
    "txh_kf_filter": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, p_i64, c_i64, p_f64, c_vp, c_vp, c_vp,
                                     c_vp, c_vp, c_vp, c_vp]),
    "txh_kfb_max_gauges": (c_i64, []),
    "txh_kfb_create": (ctypes.c_int, [c_vp, c_i64, p_i64, p_i64, p_i64, ctypes.POINTER(c_vp)]),
    "txh_kfb_destroy": (None, [c_vp]),
    "txh_kfb_set": (ctypes.c_int, [c_vp, c_i64, ctypes.c_int, p_f64, c_vp]),
    "txh_kfb_get": (ctypes.c_int, [c_vp, c_i64, ctypes.c_int, p_f64, c_vp]),
    "txh_kfb_filter": (ctypes.c_int, [c_vp, ctypes.POINTER(ctypes.c_uint8), p_f64, c_vp, c_vp, c_vp]),
    "txh_check": (ctypes.c_int, [c_vp, c_vp]),
    "txh_launch_count": (c_i64, []),
}

_lib = None


class TxhError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libtxh error {code}: {msg}")
        self.code = code


def load():
    """Load libtxh.so (never builds, never falls back)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -m tx_fast_hydrology_b200.build` "
                "(nvcc, sm_100a).  There is no CPU fallback.")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc):
    if rc != 0:
        raise TxhError(rc, load().txh_last_error().decode())


def as_i64(a):
    return np.ascontiguousarray(a, dtype=np.int64)


def as_f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def ptr_i64(a):
    return a.ctypes.data_as(p_i64)


def ptr_f64(a):
    return a.ctypes.data_as(p_f64)
