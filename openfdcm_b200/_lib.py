"""ctypes binding of libfdcm_b200.so (include/fdcm_b200.h). No fallback: a missing library or a
missing CUDA device is a hard error."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libfdcm_b200.so")

FDCM_OK = 0
FDCM_ERR_INVALID, FDCM_ERR_CUDA, FDCM_ERR_NOMEM, FDCM_ERR_OUT_OF_RANGE, FDCM_ERR_CAPACITY = 1, 2, 3, 4, 5
FDCM_SCENE_RESIDENT = -1   # n_scene value: search the scene the map was built from (resident on the device)

MATCH_DTYPE = np.dtype([("tmpl_idx", "<i4"), ("score", "<f4"), ("transform", "<f4", (6,))])
assert MATCH_DTYPE.itemsize == 32


class Dt3Params(C.Structure):
    _fields_ = [("depth", C.c_int32), ("dt3_coeff", C.c_float), ("padding", C.c_float), ("distance", C.c_int32)]


class SearchParams(C.Structure):
    _fields_ = [("max_tmpl_lines", C.c_int32), ("max_scene_lines", C.c_int32), ("batch_size", C.c_int32),
                ("penalty_kind", C.c_int32), ("penalty_tau", C.c_float), ("top_k", C.c_int32),
                ("tmpl_idx_base", C.c_int32), ("concentric", C.c_int32), ("center_x", C.c_float), ("center_y", C.c_float),
                ("low_radius", C.c_float), ("high_radius", C.c_float)]


class SelectParams(C.Structure):
    _fields_ = [("max_per_template", C.c_int32), ("radius", C.c_float), ("max_angle", C.c_float), ("across_templates", C.c_int32)]


class RefineParams(C.Structure):
    _fields_ = [("levels", C.c_int32), ("rot_steps", C.c_int32), ("rot_step", C.c_float), ("trans_steps", C.c_int32),
                ("trans_step", C.c_float)]


class DenseParams(C.Structure):
    _fields_ = [("rotations", C.c_int32), ("rot_start", C.c_float), ("rot_step", C.c_float), ("stride", C.c_int32), ("cell", C.c_int32),
                ("roi_on", C.c_int32), ("roi", C.c_float * 4)]


class CoverageParams(C.Structure):
    _fields_ = [("radius", C.c_int32), ("bin_tolerance", C.c_int32), ("min_coverage", C.c_float)]


class FitParams(C.Structure):
    _fields_ = [("iterations", C.c_int32), ("max_distance", C.c_float), ("sample_step", C.c_float), ("bin_tolerance", C.c_int32),
                ("tolerance", C.c_float), ("min_inliers", C.c_int32)]


class ScaleGridParams(C.Structure):
    _fields_ = [("scales", C.c_int32), ("scale_start", C.c_float), ("scale_ratio", C.c_float)]


class FitScaleParams(C.Structure):
    _fields_ = [("min_scale", C.c_float), ("max_scale", C.c_float)]


FIT_STATS_DTYPE = np.dtype([("n_samples", "<i4"), ("n_inliers", "<i4"), ("iterations", "<i4"), ("rms", "<f4")])
assert FIT_STATS_DTYPE.itemsize == 16


class Dt3Info(C.Structure):
    _fields_ = [("depth", C.c_int32), ("width", C.c_int32), ("height", C.c_int32), ("pitch", C.c_int32),
                ("scene_translation", C.c_float * 2), ("distance", C.c_int32), ("device", C.c_int32),
                ("n_scene_lines", C.c_int32), ("exact_dt_path", C.c_int32)]


class SearchStats(C.Structure):
    _fields_ = [("n_hypotheses", C.c_int64), ("n_valid", C.c_int64), ("n_evaluations", C.c_int64),
                ("n_lookups", C.c_int64)]


# every symbol include/fdcm_b200.h declares: name -> (restype, argtypes)
_P = C.c_void_p
SIGNATURES = {
    "fdcm_last_error": (C.c_char_p, []),
    "fdcm_abi_version": (C.c_int32, []),
    "fdcm_device_count": (C.c_int, [C.POINTER(C.c_int32)]),
    "fdcm_set_stream": (C.c_int, [C.c_int32, _P]),
    "fdcm_dt3_build": (C.c_int, [_P, C.c_int32, C.POINTER(Dt3Params), C.c_int32, C.c_int32, C.POINTER(_P)]),
    "fdcm_dt3_rebuild": (C.c_int, [_P, _P, C.c_int32]),
    "fdcm_dt3_rebuild_async": (C.c_int, [_P, _P, C.c_int32]),
    "fdcm_dt3_rerun": (C.c_int, [_P]),
    "fdcm_dt3_rerun_async": (C.c_int, [_P]),
    "fdcm_dt3_retain": (C.c_int, [_P]),
    "fdcm_dt3_release": (C.c_int, [_P]),
    "fdcm_dt3_get_info": (C.c_int, [_P, C.POINTER(Dt3Info)]),
    "fdcm_dt3_angles": (C.c_int, [_P, _P]),
    "fdcm_dt3_download_plane": (C.c_int, [_P, C.c_int32, _P]),
    "fdcm_dt3_download_mask": (C.c_int, [_P, C.c_int32, _P]),
    "fdcm_dt3_scene_bins": (C.c_int, [_P, _P]),
    "fdcm_dt3_device_ptr": (C.c_int, [_P, C.POINTER(_P), C.POINTER(C.c_uint64)]),
    "fdcm_dt3_minmax_translation": (C.c_int, [_P, _P, C.c_int32, _P, _P]),
    "fdcm_dt3_evaluate": (C.c_int, [_P, _P, _P, C.c_int32, _P, _P, _P]),
    "fdcm_dt3_classify": (C.c_int, [_P, _P, C.c_int32, _P]),
    "fdcm_templates_create": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.POINTER(_P)]),
    "fdcm_templates_release": (C.c_int, [_P]),
    "fdcm_templates_lengths": (C.c_int, [_P, _P]),
    "fdcm_search": (C.c_int, [_P, _P, _P, C.c_int32, C.POINTER(SearchParams), _P, C.c_int64, C.POINTER(C.c_int64)]),
    "fdcm_search_select": (C.c_int, [_P, _P, _P, C.c_int32, C.POINTER(SearchParams), C.POINTER(SelectParams), _P, C.c_int64,
                                     C.POINTER(C.c_int64)]),
    "fdcm_template_anchors": (C.c_int, [_P, _P, C.c_int32, _P]),
    "fdcm_refine_matches": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_float, C.POINTER(RefineParams), _P, C.c_int64, _P]),
    "fdcm_search_refine": (C.c_int, [_P, _P, _P, C.c_int32, C.POINTER(SearchParams), C.POINTER(SelectParams), C.POINTER(RefineParams), _P,
                                     C.c_int64, C.POINTER(C.c_int64)]),
    "fdcm_refine_poses": (C.c_int, [_P, _P, C.POINTER(RefineParams), C.c_int32, _P]),
    "fdcm_search_dense": (C.c_int, [_P, _P, C.POINTER(DenseParams), C.c_int32, C.c_float, C.c_int32, C.c_int32, C.POINTER(SelectParams),
                                    C.POINTER(RefineParams), _P, C.c_int64, C.POINTER(C.c_int64)]),
    "fdcm_dense_poses": (C.c_int, [C.POINTER(DenseParams), _P, _P, C.c_int32, C.c_int32, C.c_int32, _P, C.c_int64, C.POINTER(C.c_int64),
                                   _P]),
    "fdcm_match_coverage": (C.c_int, [_P, _P, C.c_int32, C.POINTER(CoverageParams), _P, C.c_int64, _P]),
    "fdcm_search_verify": (C.c_int, [_P, _P, _P, C.c_int32, C.POINTER(SearchParams), C.POINTER(SelectParams), C.POINTER(RefineParams),
                                     C.POINTER(CoverageParams), _P, C.c_int64, C.POINTER(C.c_int64)]),
    "fdcm_search_dense_verify": (C.c_int, [_P, _P, C.POINTER(DenseParams), C.c_int32, C.c_float, C.c_int32, C.c_int32, C.POINTER(SelectParams),
                                           C.POINTER(RefineParams), C.POINTER(CoverageParams), _P, C.c_int64, C.POINTER(C.c_int64)]),
    "fdcm_fit_matches": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_float, C.POINTER(FitParams), _P, C.c_int64, _P, _P]),
    "fdcm_search_dense_scales": (C.c_int, [_P, _P, C.POINTER(DenseParams), C.POINTER(ScaleGridParams), C.c_int32, C.c_float, C.c_int32,
                                           C.c_int32, C.POINTER(SelectParams), C.POINTER(RefineParams), C.POINTER(CoverageParams), _P,
                                           C.c_int64, C.POINTER(C.c_int64)]),
    "fdcm_dense_scaled_poses": (C.c_int, [C.POINTER(DenseParams), C.POINTER(ScaleGridParams), _P, _P, C.c_int32, C.c_int32, C.c_int32,
                                          C.c_int32, _P, C.c_int64, C.POINTER(C.c_int64), _P]),
    "fdcm_fit_matches_scaled": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_float, C.POINTER(FitParams), C.POINTER(FitScaleParams), _P,
                                          C.c_int64, _P, _P]),
    "fdcm_search_scales": (C.c_int, [_P, _P, _P, C.c_int32, C.POINTER(SearchParams), C.POINTER(ScaleGridParams), C.POINTER(SelectParams),
                                     C.POINTER(RefineParams), C.POINTER(CoverageParams), _P, C.c_int64, C.POINTER(C.c_int64)]),
    "fdcm_fit_samples": (C.c_int, [_P, C.c_int32, C.c_float, _P, C.c_int64, C.POINTER(C.c_int64)]),
    "fdcm_optimize": (C.c_int, [_P, _P, _P, C.c_int32, _P, C.c_int32, _P, _P, _P]),
    "fdcm_search_host": (C.c_int, [_P, _P, _P, C.c_int32, _P, C.c_int32, C.POINTER(SearchParams), _P, C.c_int64,
                                   C.POINTER(C.c_int64)]),
    "fdcm_search_last_hypotheses": (C.c_int, [_P, _P, C.c_int64, C.POINTER(C.c_int64)]),
    "fdcm_search_last_stats": (C.c_int, [_P, C.POINTER(SearchStats)]),
    "fdcm_default_search": (C.c_int, [_P, C.c_int32, _P, C.c_int32, C.c_int32, C.c_int32, _P, C.c_int32,
                                      C.POINTER(C.c_int32)]),
    "fdcm_debug_dt_rows": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P]),
    "fdcm_debug_sqrt_check": (C.c_int, [C.c_int32, C.POINTER(C.c_int64), C.POINTER(C.c_uint32)]),
    "fdcm_concentric_search": (C.c_int, [_P, C.c_int32, _P, C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_float, C.c_float,
                                         C.c_float, _P, C.c_int32, C.POINTER(C.c_int32)]),
    "fdcm_orientation_bins": (C.c_int, [C.c_int32, _P, C.c_int32, _P, _P]),
    "fdcm_penalize": (C.c_int, [C.c_int32, C.c_float, _P, C.c_int64, _P, C.c_int64]),
    "fdcm_sort_matches": (C.c_int, [_P, C.c_int64]),
    "fdcm_template_lengths": (C.c_int, [_P, _P, C.c_int32, _P]),
    "fdcm_profile_enable": (C.c_int, [C.c_int32]),
    "fdcm_profile_reset": (C.c_int, []),
    "fdcm_profile_get": (C.c_int, [C.c_int32, C.c_char_p, C.c_int32, C.POINTER(C.c_double), C.POINTER(C.c_int64),
                                   C.POINTER(C.c_double)]),
    "fdcm_profile_count": (C.c_int, [C.POINTER(C.c_int32)]),
    "fdcm_kernel_launch_count": (C.c_int64, []),
    "fdcm_comm_unique_id": (C.c_int, [_P]),
    "fdcm_comm_init": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.POINTER(_P)]),
    "fdcm_comm_destroy": (C.c_int, [_P]),
    "fdcm_comm_info": (C.c_int, [_P, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "fdcm_comm_shard": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "fdcm_comm_search_topk": (C.c_int, [_P, _P, _P, _P, C.c_int32, C.POINTER(SearchParams), _P, C.c_int64, C.POINTER(C.c_int64)]),
    "fdcm_comm_search_select": (C.c_int, [_P, _P, _P, _P, C.c_int32, C.POINTER(SearchParams), C.POINTER(SelectParams), _P, C.c_int64,
                                          C.POINTER(C.c_int64)]),
    "fdcm_comm_search_host_topk": (C.c_int, [_P, _P, _P, _P, C.c_int32, _P, C.c_int32, C.POINTER(SearchParams), _P, C.c_int64,
                                             C.POINTER(C.c_int64)]),
    "fdcm_comm_rebuild_broadcast": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32]),
    "fdcm_set_host_threads": (C.c_int, [C.c_int32]),
    "fdcm_scene_batch_create": (C.c_int, [C.POINTER(Dt3Params), C.c_int32, C.POINTER(_P)]),
    "fdcm_scene_batch_destroy": (C.c_int, [_P]),
    "fdcm_search_scenes": (C.c_int, [_P, _P, _P, C.c_int32, _P, C.POINTER(SearchParams), _P, _P]),
    "fdcm_search_scenes_select": (C.c_int, [_P, _P, _P, C.c_int32, _P, C.POINTER(SearchParams), C.POINTER(SelectParams), _P, _P]),
}


class FdcmError(RuntimeError):
    def __init__(self, status, message):
        super().__init__(f"libfdcm_b200 status {status}: {message}")
        self.status = status


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: build it with `make -C openfdcm_b200/csrc` "
                              "(or __graft_entry__.build()); there is no CPU fallback")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)   # AttributeError if a declared symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(status):
    if status != FDCM_OK:
        msg = lib().fdcm_last_error()
        raise FdcmError(status, msg.decode() if msg else "")


def ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None
