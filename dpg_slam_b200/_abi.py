"""ctypes view of the C ABI in include/dpgicp.h (types + loader).

The structures mirror ``dpgicp_params`` / ``dpgicp_result`` field for field; the loader binds the
in-tree ``libdpgicp.so`` built by ``__graft_entry__.build()`` and raises if it is missing — there
is no CPU fallback in the product path.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))

# ---- constants (include/dpgicp.h) -----------------------------------------------------------------
ABI_VERSION = 4
METRIC_POINT_TO_POINT, METRIC_POINT_TO_LINE = 0, 1
SEARCH_BRUTE, SEARCH_PRUNED, SEARCH_PROJECTIVE = 0, 1, 2
COV_REFERENCE_LIVE, COV_CENSI_INDEXPAIR, COV_CENSI_CORR = 0, 1, 2
OUTLIER_NONE, OUTLIER_TRIMMED, OUTLIER_MEDIAN = 0, 1, 2
ENUM_REOPTIMIZE, ENUM_ONLINE = 0, 1
STOP_MASK = 0xFF
STOP_NONE, STOP_ITERATIONS, STOP_TRANSFORM, STOP_ABS_MSE, STOP_NO_CORRESPONDENCES, STOP_DEGENERATE = 0, 1, 2, 3, 4, 5
FLAG_CONVERGED, FLAG_COV_SINGULAR, FLAG_EMPTY_INPUT, FLAG_FACTOR_INVALID = 0x100, 0x200, 0x400, 0x800
MAX_ABS_COORD = 1000.0
MAX_POINTS = 8192
IPC_HANDLE_BYTES = 64
MAX_GATHER_RANKS = 16

ERRORS = {0: "OK", -1: "E_INVALID", -2: "E_NODEVICE", -3: "E_CUDA", -4: "E_NOMEM", -5: "E_RANGE",
          -6: "E_STATE", -7: "E_TOOBIG"}


class Params(C.Structure):
    """``dpgicp_params``; defaults are the reference's parameters.h values."""
    _fields_ = [
        ("max_iterations", C.c_int32),
        ("use_reciprocal", C.c_int32),
        ("ransac_iterations", C.c_int32),
        ("downsample_divisor", C.c_int32),
        ("metric", C.c_int32),
        ("search", C.c_int32),
        ("cov_mode", C.c_int32),
        ("cov_cap", C.c_int32),
        ("transformation_epsilon", C.c_double),
        ("max_correspondence_distance", C.c_double),
        ("cov_sensor_variance", C.c_double),
        ("laser_x_variance", C.c_float),
        ("laser_y_variance", C.c_float),
        ("laser_theta_variance", C.c_float),
        ("projective_window", C.c_int32),
        ("sensor_x", C.c_float),
        ("sensor_y", C.c_float),
        ("outlier_mode", C.c_int32),
        ("reserved0", C.c_int32),
        ("outlier_param", C.c_double),
    ]

    @classmethod
    def defaults(cls, **overrides) -> "Params":
        """parameters.h:146,159,173,191,201,374,385,396,402; cov_func_point_to_point.h:307,554."""
        p = cls(max_iterations=500, use_reciprocal=1, ransac_iterations=50, downsample_divisor=5,
                metric=METRIC_POINT_TO_POINT, search=SEARCH_PRUNED, cov_mode=COV_REFERENCE_LIVE,
                cov_cap=200, transformation_epsilon=5e-9, max_correspondence_distance=0.6,
                cov_sensor_variance=0.01, laser_x_variance=0.5, laser_y_variance=0.5,
                laser_theta_variance=0.3, projective_window=8, sensor_x=0.2, sensor_y=0.0,
                outlier_mode=OUTLIER_NONE, reserved0=0, outlier_param=0.0)
        for k, v in overrides.items():
            if not hasattr(p, k):
                raise AttributeError(f"dpgicp_params has no field {k!r}")
            setattr(p, k, v)
        return p

    def copy(self, **overrides) -> "Params":
        q = Params.from_buffer_copy(bytes(self))
        for k, v in overrides.items():
            if not hasattr(q, k):
                raise AttributeError(f"dpgicp_params has no field {k!r}")
            setattr(q, k, v)
        return q


class Result(C.Structure):
    """``dpgicp_result`` (112 bytes)."""
    _fields_ = [
        ("tx", C.c_float), ("ty", C.c_float), ("theta", C.c_float),
        ("rot_c", C.c_float), ("rot_s", C.c_float),
        ("iterations", C.c_int32), ("status", C.c_uint32), ("n_correspondences", C.c_int32),
        ("mse", C.c_double),
        ("cov", C.c_double * 9),
    ]


RESULT_DTYPE = np.dtype([
    ("tx", "<f4"), ("ty", "<f4"), ("theta", "<f4"), ("rot_c", "<f4"), ("rot_s", "<f4"),
    ("iterations", "<i4"), ("status", "<u4"), ("n_correspondences", "<i4"),
    ("mse", "<f8"), ("cov", "<f8", (9,)),
], align=True)

FACTOR_DTYPE = np.dtype([
    ("from_node", "<i4"), ("to_node", "<i4"), ("tx", "<f4"), ("ty", "<f4"), ("theta", "<f4"), ("status", "<u4"),
    ("sqrt_info", "<f8", (9,)),
], align=True)

assert C.sizeof(Result) == 112 and RESULT_DTYPE.itemsize == 112 and FACTOR_DTYPE.itemsize == 96
assert C.sizeof(Params) == 96

EXPORTS = [
    "dpgicp_abi_version", "dpgicp_default_params", "dpgicp_create", "dpgicp_destroy",
    "dpgicp_last_error", "dpgicp_set_stream", "dpgicp_synchronize", "dpgicp_upload_scans",
    "dpgicp_upload_ranges", "dpgicp_upload_ranges_subset", "dpgicp_scan_count", "dpgicp_download_scan", "dpgicp_submit_pairs",
    "dpgicp_set_pairs", "dpgicp_set_pair_cost_hints", "dpgicp_run", "dpgicp_fetch_results", "dpgicp_fetch_factors", "dpgicp_results_device_ptr",
    "dpgicp_gather_export", "dpgicp_gather_attach", "dpgicp_gather_detach", "dpgicp_gather_fetch",
    "dpgicp_gather_device_ptr", "dpgicp_last_run_counters", "dpgicp_single_pair", "dpgicp_cov", "dpgicp_cov_pairs", "dpgicp_correspondences",
    "dpgicp_enumerate_pairs", "dpgicp_relative_guess", "dpgicp_fp32_probe", "dpgicp_fp32x2_probe",
    "dpgicp_correspondences_seeded", "dpgicp_set_nodes", "dpgicp_enumerate_pairs_device", "dpgicp_fetch_pairs",
    "dpgicp_convert_ranges_device", "dpgicp_gather_attach_local", "dpgicp_gather_set_root_only",
    "dpgicp_enable_stage_timing", "dpgicp_last_run_stage_ms", "dpgicp_run_range", "dpgicp_fetch_results_range",
    "dpgicp_gather_fetch_range", "dpgicp_gather_declare", "dpgicp_append_ranges", "dpgicp_append_scans",
]

_lib = None


def library_path() -> str:
    # DPGICP_LIBRARY selects a development build variant of the same library (A/B timing)
    return os.environ.get("DPGICP_LIBRARY") or os.path.join(_HERE, "libdpgicp.so")


def load_library() -> C.CDLL:
    """Bind libdpgicp.so.  Raises (never falls back) when the CUDA extension is not built."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        raise RuntimeError(
            f"{path} is missing: build the CUDA back end first (python -c 'import __graft_entry__ as g; "
            "g.build()' or make -C dpg_slam_b200/csrc). dpg_slam_b200 has no CPU fallback.")
    lib = C.CDLL(path)
    vp, i32, i64, sz = C.c_void_p, C.c_int32, C.c_int64, C.c_size_t
    PP, PR = C.POINTER(Params), C.POINTER(Result)
    sig = {
        "dpgicp_abi_version": (C.c_int, []),
        "dpgicp_default_params": (C.c_int, [PP]),
        "dpgicp_create": (C.c_int, [C.c_int, C.POINTER(vp)]),
        "dpgicp_destroy": (None, [vp]),
        "dpgicp_last_error": (C.c_char_p, [vp]),
        "dpgicp_set_stream": (C.c_int, [vp, vp]),
        "dpgicp_synchronize": (C.c_int, [vp]),
        "dpgicp_upload_scans": (C.c_int, [vp, vp, sz, vp, i32]),
        "dpgicp_upload_ranges": (C.c_int, [vp, vp, i32, i32] + [C.c_float] * 6),
        "dpgicp_upload_ranges_subset": (C.c_int, [vp, vp, i32, i32, vp, i32] + [C.c_float] * 6),
        "dpgicp_append_ranges": (C.c_int, [vp, vp, i32, i32] + [C.c_float] * 6),
        "dpgicp_append_scans": (C.c_int, [vp, vp, sz, vp, i32]),
        "dpgicp_scan_count": (C.c_int, [vp]),
        "dpgicp_download_scan": (C.c_int, [vp, i32, vp, C.POINTER(i32)]),
        "dpgicp_submit_pairs": (C.c_int, [vp, vp, vp, vp, i64, PP, vp]),
        "dpgicp_set_pairs": (C.c_int, [vp, vp, vp, vp, i64]),
        "dpgicp_set_pair_cost_hints": (C.c_int, [vp, vp, i64]),
        "dpgicp_run": (C.c_int, [vp, PP]),
        "dpgicp_fetch_results": (C.c_int, [vp, vp, i64]),
        "dpgicp_fetch_factors": (C.c_int, [vp, vp, i64]),
        "dpgicp_results_device_ptr": (C.c_int, [vp, C.POINTER(vp), C.POINTER(i64)]),
        "dpgicp_gather_export": (C.c_int, [vp, i64, vp]),
        "dpgicp_gather_attach": (C.c_int, [vp, vp, i32, i32]),
        "dpgicp_gather_declare": (C.c_int, [vp, i64, vp]),
        "dpgicp_gather_detach": (C.c_int, [vp]),
        "dpgicp_gather_fetch": (C.c_int, [vp, vp, i64]),
        "dpgicp_gather_device_ptr": (C.c_int, [vp, C.POINTER(vp), C.POINTER(i64)]),
        "dpgicp_last_run_counters": (C.c_int, [vp, C.POINTER(C.c_uint64 * 8)]),
        "dpgicp_single_pair": (C.c_int, [vp, vp, i32, vp, i32, sz, vp, PP, PR]),
        "dpgicp_cov": (C.c_int, [vp, vp, i32, vp, i32, sz, vp, PP, vp, C.POINTER(C.c_uint32)]),
        "dpgicp_cov_pairs": (C.c_int, [vp, vp, vp, vp, i64, PP, vp, vp, C.POINTER(C.c_float)]),
        "dpgicp_correspondences": (C.c_int, [vp, vp, i32, vp, i32, sz, vp, PP, vp, vp]),
        "dpgicp_relative_guess": (C.c_int, [vp, vp, vp]),
        "dpgicp_fp32_probe": (C.c_int, [vp, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
        "dpgicp_fp32x2_probe": (C.c_int, [vp, C.POINTER(C.c_double)]),
        "dpgicp_enumerate_pairs": (C.c_int, [vp, vp, vp, i32, C.c_float, C.c_float, vp, vp,
                                              C.POINTER(i64)]),
        "dpgicp_correspondences_seeded": (C.c_int, [vp, vp, i32, vp, i32, sz, vp, PP, vp, vp, vp, vp]),
        "dpgicp_set_nodes": (C.c_int, [vp, vp, vp, i32]),
        "dpgicp_enumerate_pairs_device": (C.c_int, [vp, i32, C.c_float, C.c_float, i32, i32, C.POINTER(i64), C.POINTER(i64)]),
        "dpgicp_fetch_pairs": (C.c_int, [vp, vp, vp, vp, i64]),
        "dpgicp_convert_ranges_device": (C.c_int, [vp, vp, i32, i32] + [C.c_float] * 6),
        "dpgicp_gather_attach_local": (C.c_int, [C.POINTER(vp), i32, i64, i32]),
        "dpgicp_gather_set_root_only": (C.c_int, [vp, i32]),
        "dpgicp_enable_stage_timing": (C.c_int, [vp, i32]),
        "dpgicp_last_run_stage_ms": (C.c_int, [vp, C.POINTER(C.c_float * 8), C.POINTER(i32)]),
        "dpgicp_run_range": (C.c_int, [vp, PP, i64, i64]),
        "dpgicp_fetch_results_range": (C.c_int, [vp, vp, i64, i64]),
        "dpgicp_gather_fetch_range": (C.c_int, [vp, vp, i64, i64]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)      # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.dpgicp_abi_version() != ABI_VERSION:
        raise RuntimeError("libdpgicp.so ABI version mismatch")
    _lib = lib
    return lib
