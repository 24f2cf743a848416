"""ctypes binding of libcoverage_cuda.so (include/coverage_cuda.h).

The shared library is built in-tree by `make` / `__graft_entry__.build()`.  There is no fallback:
if the library is missing, importing this module raises, and if no CUDA device is usable
`cov_create` fails with COV_ERR_CUDA.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("COVERAGE_CUDA_LIB") or os.path.join(_HERE, "libcoverage_cuda.so")  # override: kernel experiments

COV_OK = 0
COV_ERR_INVALID = -1
COV_ERR_STATE = -2
COV_ERR_CUDA = -3
COV_ERR_OFF_LATTICE = -4
COV_ERR_LIMIT = -5
COV_ERR_NOMEM = -6

KERNEL_AUTO, KERNEL_SPAN, KERNEL_BRUTE, KERNEL_EXACT, KERNEL_SPAN_GENERAL, KERNEL_ORDERED = 0, 1, 2, 3, 4, 5
OPT_KERNEL, OPT_WARPS_PER_CTA, OPT_CTAS_PER_SM, OPT_BAND_ROWS, OPT_FORCE_EXACT, OPT_CHUNK, OPT_TRACE, OPT_ZEROCOPY_OUT, OPT_PLANE_MODE = 1, 2, 3, 4, 5, 6, 7, 8, 9
OPT_PROGRESSIVE_INDEX = 10
OPT_LIST_ORDER_HORIZON = 11
PACK_F32, PACK_I32, PACK_I16 = 1, 2, 3


class GridInfo(C.Structure):
    _fields_ = [("nx", C.c_int64), ("ny", C.c_int64), ("dx", C.c_double), ("dy", C.c_double),
                ("n_entries", C.c_int64), ("n_cells", C.c_int64), ("n_planes", C.c_int64),
                ("n_classes", C.c_int64), ("area_exact", C.c_int32), ("planes_in_smem", C.c_int32)]


class LaunchInfo(C.Structure):
    _fields_ = [("kernel", C.c_int32), ("grid", C.c_int32), ("block", C.c_int32), ("smem_bytes", C.c_int32),
                ("band_rows", C.c_int32), ("planes_in_smem", C.c_int32), ("multi", C.c_int32), ("chunk", C.c_int32),
                ("max_warps", C.c_int32), ("plane_mode", C.c_int32)]


class Limits(C.Structure):
    _fields_ = [("max_uavs", C.c_int64), ("max_nx", C.c_int64), ("max_ny", C.c_int64),
                ("max_planes", C.c_int64), ("max_classes", C.c_int64)]


_vp, _i, _i64, _d = C.c_void_p, C.c_int, C.c_int64, C.c_double
_pd, _pi64, _pu8, _pu32 = C.POINTER(C.c_double), C.POINTER(C.c_int64), C.POINTER(C.c_uint8), C.POINTER(C.c_uint32)

# name -> (restype, argtypes); every symbol include/coverage_cuda.h declares
SIGNATURES = {
    "cov_abi_version": (_i, []),
    "cov_device_count": (_i, []),
    "cov_create": (_i, [_i, C.POINTER(_vp)]),
    "cov_destroy": (None, [_vp]),
    "cov_last_error": (C.c_char_p, [_vp]),
    "cov_set_option": (_i, [_vp, _i, _i64]),
    "cov_get_option": (_i, [_vp, _i, _pi64]),
    "cov_set_grid_bits": (_i, [_vp, _i64, _i64, _d, _d, _vp, _d]),
    "cov_set_grid_cells": (_i, [_vp, _i64, _i64, _d, _d, _vp, _vp, _i64, _vp]),
    "cov_set_points": (_i, [_vp, _vp, _i64, _i64, _i64, _d, _d]),
    "cov_set_grid_full": (_i, [_vp, _i64, _i64, _d, _d]),
    "cov_add_points": (_i, [_vp, _vp, _i64]),
    "cov_get_grid_info": (_i, [_vp, C.POINTER(GridInfo)]),
    "cov_get_grid_cells": (_i, [_vp, _vp]),
    "cov_get_class_weights": (_i, [_vp, _pd, _i64]),
    "cov_remove_covered": (_i, [_vp, _vp, _i64, _pi64]),
    "cov_fire_init": (_i, [_vp, _i64, _i64, _d, _d, _vp, C.c_int32]),
    "cov_fire_step": (_i, [_vp, _d, _d, _d, C.c_uint64, _i64, C.c_int32, _pi64]),
    "cov_fire_get_state": (_i, [_vp, _vp]),
    "cov_set_params": (_i, [_vp, _i64, _vp, _d, _vp, _vp, _d, _d, C.c_int32]),
    "cov_eval_batch": (_i, [_vp, _vp, _i64, _vp, _vp, _vp]),
    "cov_eval_batch_ex": (_i, [_vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp]),
    "cov_eval_batch_device": (_i, [_vp, _vp, _i64, _vp, _vp, _vp]),
    "cov_eval_one": (_i, [_vp, _vp, _pd]),
    "cov_eval_batch_best": (_i, [_vp, _vp, _i64, _vp, _vp, _vp, C.c_int32, _pd, _pi64]),
    "cov_eval_batch_packed": (_i, [_vp, _vp, C.c_int32, _d, _i64, _vp, _vp, _vp, C.c_int32, _pd, _pi64]),
    "cov_argmin": (_i, [_vp, _vp, _i64, C.c_int32, _pd, _pi64]),
    "cov_union_area_batch": (_i, [_vp, _vp, _i64, _i64, _vp]),
    "cov_mads_solve": (_i, [_vp, _vp, _i64, _d, C.c_uint64, _vp, _pd, _pi64]),
    "cov_mads_solve_batch": (_i, [_vp, _vp, _i64, _i64, _d, C.c_uint64, _vp, _vp, _vp]),
    "cov_run_horizon": (_i, [_vp, _vp, _i64, _i64, _d, _i64, _d, C.c_uint64, _vp, _i64, _d, _d, _vp, _vp, _vp, _vp]),
    "cov_run_horizon_points": (_i, [_vp, _vp, _i64, _i64, _d, _i64, _d, C.c_uint64, _vp, _i64, _d, _d, _vp, _vp,
                                    _vp, _vp, _vp, _vp, _vp]),
    "cov_run_horizon_ensemble": (_i, [_vp, _vp, _i64, _i64, _i64, _d, _i64, _d, C.c_uint64, _vp, _i64, _d, _d, _vp, _vp,
                                      _vp, _vp, _vp]),
    "cov_run_horizon_fire": (_i, [_vp, _vp, _i64, _i64, _d, _i64, _d, C.c_uint64, _vp, _i64, _d, _d, _vp, _d, _d, _d,
                                  C.c_uint64, _i64, _vp, _vp, _vp, _vp]),
    "cov_run_horizon_fire_ensemble": (_i, [_vp, _vp, _i64, _i64, _i64, _d, _i64, _d, C.c_uint64, _vp, _i64, _d, _d,
                                           _vp, _vp, C.c_uint64, C.c_uint64, _i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "cov_run_horizon_points_ensemble": (_i, [_vp, _vp, _i64, _i64, _i64, _d, _i64, _d, C.c_uint64, _vp, _i64, _d, _d,
                                             _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "cov_covered_mask": (_i, [_vp, _vp, _vp]),
    "cov_set_region": (_i, [_vp, _d, _d, _d, _d, _vp, _i64]),
    "cov_eval_region_batch": (_i, [_vp, _vp, _i64, _vp, _vp, _vp, C.c_int32, _pd, _pi64]),
    "cov_mads_solve_batch_region": (_i, [_vp, _vp, _i64, _i64, _d, C.c_uint64, _vp, _vp, _vp]),
    "cov_run_horizon_region": (_i, [_vp, _vp, _i64, _i64, _d, _i64, _d, C.c_uint64, _vp, _i64, _d, _d, _vp, _vp, _vp,
                                    _vp]),
    "cov_sync": (_i, [_vp]),
    "cov_stream": (_vp, [_vp]),
    "cov_set_stream": (_i, [_vp, _vp]),
    "cov_host_alloc": (_i, [_vp, _i64, C.POINTER(_vp)]),
    "cov_host_free": (_i, [_vp, _vp]),
    "cov_device_alloc": (_i, [_vp, _i64, C.POINTER(_vp)]),
    "cov_device_free": (_i, [_vp, _vp]),
    "cov_memcpy_h2d": (_i, [_vp, _vp, _vp, _i64]),
    "cov_memcpy_d2h": (_i, [_vp, _vp, _vp, _i64]),
    "cov_launch_count": (_i64, [_vp]),
    "cov_get_trace": (_i64, [_vp, _pd, _i64]),
    "cov_last_kernel_ms": (_i, [_vp, _pd]),
    "cov_kernel_time_total": (_i, [_vp, _pd, _pi64]),
    "cov_last_launch": (_i, [_vp, C.POINTER(LaunchInfo)]),
    "cov_generate_candidates": (_i, [_vp, _vp, _i64, _i64, C.c_uint64, _i64, _d, _d, _d, _d, _d]),
    "cov_multi_create": (_i, [C.POINTER(C.c_int), _i, C.POINTER(_vp)]),
    "cov_multi_destroy": (None, [_vp]),
    "cov_multi_last_error": (C.c_char_p, [_vp]),
    "cov_multi_size": (_i, [_vp]),
    "cov_multi_handle": (_vp, [_vp, _i]),
    "cov_multi_eval_batch": (_i, [_vp, _vp, _i64, _vp, _vp, _vp]),
    "cov_multi_run_horizon_ensemble": (_i, [_vp, _vp, _i64, _i64, _i64, _d, _i64, _d, C.c_uint64, _vp, _i64, _d, _d,
                                            _vp, _vp, _vp, _vp]),
    "cov_multi_run_horizon_fire_ensemble": (_i, [_vp, _vp, _i64, _i64, _i64, _d, _i64, _d, C.c_uint64, _vp, _i64, _d,
                                                 _d, _vp, _vp, C.c_uint64, C.c_uint64, _i64, _vp, _vp, _vp, _vp, _vp]),
    "cov_multi_run_horizon_points_ensemble": (_i, [_vp, _vp, _i64, _i64, _i64, _d, _i64, _d, C.c_uint64, _vp, _i64,
                                                   _d, _d, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "cov_multi_argmin": (_i, [_vp, _vp, _i64, C.c_int32, _pd, _pi64]),
    "cov_get_limits": (None, [C.POINTER(Limits)]),
    "cov_threshold": (_d, [_d]),
}


def load(path: str = LIB_PATH) -> C.CDLL:
    if not os.path.exists(path):
        raise ImportError(
            f"{path} is missing: build it with `make` (or __graft_entry__.build()). "
            "libcoverage_cuda has no CPU fallback.")
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    return lib


lib = load()


class CoverageError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"libcoverage_cuda error {code}: {message}")
        self.code = code
        self.message = message
