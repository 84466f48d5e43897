"""ctypes binding of ``include/apc.h`` - the only door from Python into the CUDA path.

There is no CPU fallback: if ``libapc.so`` is missing or cannot be loaded the import of
this module raises, and every wrapper raises ``RuntimeError`` on a non-zero status (the
reference's node swallows exceptions per frame, pp.py:701-702, so behaviour is preserved).
"""
from __future__ import annotations

import ctypes as C
import os

PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG, "libapc.so")

APC_MAX_FIELDS = 16
APC_MAX_CLOUDS = 8
APC_MAX_NEIGHBORS = 1024   # statistical nb_neighbors, normals and FPFH max_nn
APC_MAX_TRANSFORMS = 3
APC_MAX_MIRRORS = 8

APC_OK, APC_ERR_CUDA, APC_ERR_BAD_ARG, APC_ERR_KEY_RANGE, APC_ERR_CAPACITY, APC_ERR_TOO_FEW = 0, -1, -2, -3, -4, -5
CROP_NUMPY, CROP_TORCH, CROP_OPEN3D = 0, 1, 2
DEDUP_OFF, DEDUP_OPEN3D, DEDUP_NUMPY, DEDUP_TORCH_COMPAT = 0, 1, 2, 3
STAGE_NANSKIP, STAGE_DEDUP, STAGE_FINITE, STAGE_CROP = 1, 2, 4, 8
APC_ICP_POINT_TO_POINT, APC_ICP_POINT_TO_PLANE, APC_ICP_GENERALIZED = 0, 1, 2
APC_ICP_OK, APC_ICP_NO_CORRESPONDENCE, APC_ICP_DEGENERATE = 0, 1, 2
APC_FGR_OK, APC_FGR_TOO_FEW, APC_FGR_DEGENERATE = 0, 1, 2
(CNT_INPUT, CNT_FILTERED, CNT_VOXELS, CNT_AFTER_STAT, CNT_AFTER_RADIUS, CNT_GROUND_INLIERS, CNT_OUTPUT,
 CNT_STATUS) = range(8)


class Field(C.Structure):
    _fields_ = [("offset", C.c_int32), ("datatype", C.c_int32)]


class CloudDesc(C.Structure):
    _fields_ = [("data_dev", C.c_void_p), ("n_points", C.c_uint32), ("point_step", C.c_uint32),
                ("x", Field), ("y", Field), ("z", Field), ("intensity", Field),
                ("n_nan_fields", C.c_uint32), ("nan_fields", Field * APC_MAX_FIELDS),
                ("has_transform", C.c_int32), ("transform", C.c_float * 16)]


class FilterCfg(C.Structure):
    _fields_ = [("skip_nans", C.c_int32), ("dedup_mode", C.c_int32), ("remove_nan", C.c_int32),
                ("remove_inf", C.c_int32), ("n_transforms", C.c_uint32),
                ("transforms", (C.c_float * 16) * APC_MAX_TRANSFORMS),
                ("crop_enable", C.c_int32), ("crop_mode", C.c_int32), ("crop_invert", C.c_int32),
                ("roi_min", C.c_double * 3), ("roi_max", C.c_double * 3)]


class OutField(C.Structure):
    _fields_ = [("offset", C.c_int32), ("datatype", C.c_int32), ("source", C.c_int32),
                ("attr_datatype", C.c_int32), ("attr_dev", C.c_void_p)]


class PipelineMaps(C.Structure):
    _fields_ = [("src_idx_dev", C.c_void_p), ("p2v_dev", C.c_void_p), ("voxel_counts_dev", C.c_void_p),
                ("out_row_dev", C.c_void_p), ("normals_dev", C.c_void_p)]


class OutMirror(C.Structure):
    _fields_ = [("n_xyzi", C.c_uint32), ("xyzi_multicast", C.c_int32), ("xyzi_dev", C.c_void_p * APC_MAX_MIRRORS),
                ("n_counts", C.c_uint32), ("counts_dev", C.c_void_p * APC_MAX_MIRRORS)]


class PipelineCfg(C.Structure):
    _fields_ = [("filter", FilterCfg), ("voxel_size", C.c_float),
                ("stat_enable", C.c_int32), ("stat_nb_neighbors", C.c_int32), ("stat_std_ratio", C.c_double),
                ("radius_enable", C.c_int32), ("radius_nb_points", C.c_int32),
                ("radius_search_radius", C.c_double),
                ("ground_enable", C.c_int32), ("ground_distance_threshold", C.c_double),
                ("ground_ransac_n", C.c_int32), ("ground_num_iterations", C.c_int32),
                ("ground_probability", C.c_double), ("ground_seed", C.c_uint64),
                ("normals_enable", C.c_int32), ("normals_max_nn", C.c_int32), ("normals_radius", C.c_double)]


def _load():
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: build it with `python -m autodriver_pointcloud_preprocessor_b200._build` "
            "(nvcc, sm_100a).  This package has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, u32, i32, f64 = C.c_void_p, C.c_uint32, C.c_int, C.c_double
    sig = {
        "apc_ctx_create": [i32, u32, C.POINTER(vp)],
        "apc_ctx_destroy": [vp],
        "apc_check": [vp, vp],
        "apc_ctx_set_low_latency": [vp, i32],
        "apc_version": [],
        "apc_frontend": [vp, C.POINTER(CloudDesc), u32, C.POINTER(FilterCfg), vp, vp, vp, vp, vp],
        "apc_unpack": [vp, C.POINTER(CloudDesc), vp, vp],
        "apc_transform": [vp, vp, u32, vp, C.POINTER(C.c_float), vp, vp],
        "apc_crop_mask": [vp, vp, u32, vp, C.POINTER(f64), C.POINTER(f64), i32, i32, vp, vp],
        "apc_non_finite_mask": [vp, vp, u32, vp, i32, i32, vp, vp],
        "apc_duplicate_mask": [vp, vp, u32, vp, vp, vp],
        "apc_unique_rows": [vp, vp, u32, vp, vp, vp, vp, vp],
        "apc_select_by_mask": [vp, vp, u32, vp, vp, i32, vp, vp, vp, vp],
        "apc_gather": [vp, vp, u32, vp, u32, vp, vp, vp],
        "apc_pack_xyzi": [vp, vp, vp, u32, vp, vp],
        "apc_split_xyzi": [vp, vp, u32, vp, vp, vp, vp],
        "apc_voxel_downsample": [vp, vp, u32, vp, C.c_float, vp, vp, vp, vp, vp],
        "apc_voxel_downsample_sorted": [vp, vp, u32, vp, C.c_float, vp, vp, vp, vp],
        "apc_voxel_mean_attr": [vp, vp, vp, u32, vp, vp, i32, vp, vp],
        "apc_radius_outliers": [vp, vp, u32, vp, i32, f64, vp, vp, vp],
        "apc_statistical_outliers": [vp, vp, u32, vp, i32, f64, vp, vp, vp, vp],
        "apc_estimate_normals": [vp, vp, u32, vp, i32, f64, vp, vp, vp, vp],
        "apc_estimate_normals_knn": [vp, vp, u32, vp, i32, vp, vp, vp, vp],
        "apc_estimate_normals_radius": [vp, vp, u32, vp, f64, vp, vp, vp, vp],
        "apc_cluster_dbscan": [vp, vp, u32, vp, f64, i32, vp, vp, vp, vp],
        "apc_evaluate_registration": [vp, vp, u32, vp, vp, u32, vp, f64, C.POINTER(f64), vp, vp, vp, vp],
        "apc_icp": [vp, vp, u32, vp, vp, vp, u32, vp, f64, C.POINTER(f64), i32, i32, f64, f64, vp, vp, vp, vp, vp],
        "apc_icp_generalized": [vp, vp, vp, u32, vp, vp, vp, u32, vp, f64, C.POINTER(f64), f64, i32, f64, f64, vp, vp,
                                vp, vp, vp, vp, vp],
        "apc_compute_fpfh": [vp, vp, vp, u32, vp, i32, f64, vp, vp, vp, vp],
        "apc_compute_fpfh_knn": [vp, vp, vp, u32, vp, i32, vp, vp, vp, vp],
        "apc_correspondences_from_features": [vp, vp, u32, vp, vp, u32, vp, i32, i32, f64, vp, vp, vp, vp],
        "apc_fgr_from_features": [vp, vp, u32, vp, vp, u32, vp, vp, vp, i32, f64, i32, i32, f64, i32, f64, i32, i32,
                                  C.c_uint64, vp, vp, vp, vp],
        "apc_fgr": [vp, vp, u32, vp, vp, u32, vp, vp, u32, vp, f64, i32, i32, f64, i32, vp, vp, vp, vp],
        "apc_segment_plane": [vp, vp, u32, vp, f64, i32, i32, f64, C.c_uint64, vp, vp, vp, vp, vp],
        "apc_segment_plane_scores": [vp, vp, u32, vp],
        "apc_repack": [vp, vp, u32, vp, C.POINTER(OutField), u32, u32, vp, vp],
        "apc_pipeline_run": [vp, C.POINTER(CloudDesc), u32, C.POINTER(PipelineCfg), vp, vp, vp, vp],
        "apc_pipeline_run_maps": [vp, C.POINTER(CloudDesc), u32, C.POINTER(PipelineCfg), vp, vp, vp,
                                  C.POINTER(PipelineMaps), vp],
        "apc_graph_capture_pipeline": [vp, C.POINTER(CloudDesc), u32, C.POINTER(PipelineCfg), vp, vp, vp,
                                       C.POINTER(vp)],
        "apc_pipeline_run_ex": [vp, C.POINTER(CloudDesc), u32, C.POINTER(PipelineCfg), vp, vp, vp,
                                C.POINTER(PipelineMaps), C.POINTER(OutMirror), vp],
        "apc_graph_capture_pipeline_ex": [vp, C.POINTER(CloudDesc), u32, C.POINTER(PipelineCfg), vp, vp, vp,
                                          C.POINTER(PipelineMaps), C.POINTER(OutMirror), C.POINTER(vp)],
        "apc_pipeline_run_mirrored": [vp, C.POINTER(CloudDesc), u32, C.POINTER(PipelineCfg), vp, vp, vp,
                                      C.POINTER(OutMirror), vp],
        "apc_graph_capture_pipeline_mirrored": [vp, C.POINTER(CloudDesc), u32, C.POINTER(PipelineCfg), vp, vp, vp,
                                                C.POINTER(OutMirror), C.POINTER(vp)],
        "apc_graph_launch": [vp, vp, vp],
        "apc_graph_destroy": [vp],
        "apc_graph_kernel_count": [vp],
        "apc_profile_enable": [vp, i32],
        "apc_profile_report": [vp, C.c_char_p, u32],
    }
    for name, args in sig.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = C.c_int
    lib.apc_last_error.argtypes = [vp]
    lib.apc_last_error.restype = C.c_char_p
    lib.apc_ctx_max_points.argtypes = [vp]
    lib.apc_ctx_max_points.restype = u32
    return lib


lib = _load()

#: every symbol include/apc.h declares (checked by tests/test_capi_symbols.py)
SYMBOLS = ["apc_ctx_create", "apc_ctx_destroy", "apc_ctx_set_low_latency", "apc_last_error", "apc_check", "apc_version",
           "apc_ctx_max_points", "apc_frontend", "apc_unpack", "apc_transform", "apc_crop_mask",
           "apc_non_finite_mask", "apc_duplicate_mask", "apc_unique_rows", "apc_select_by_mask", "apc_gather",
           "apc_voxel_downsample", "apc_voxel_downsample_sorted", "apc_voxel_mean_attr", "apc_radius_outliers",
           "apc_statistical_outliers", "apc_estimate_normals", "apc_estimate_normals_knn",
           "apc_estimate_normals_radius", "apc_cluster_dbscan", "apc_evaluate_registration", "apc_icp", "apc_icp_generalized", "apc_compute_fpfh",
           "apc_compute_fpfh_knn", "apc_correspondences_from_features", "apc_fgr_from_features", "apc_fgr", "apc_segment_plane", "apc_segment_plane_scores", "apc_repack", "apc_pipeline_run", "apc_pipeline_run_maps",
           "apc_pipeline_run_mirrored", "apc_pipeline_run_ex", "apc_graph_capture_pipeline_ex",
           "apc_graph_capture_pipeline", "apc_graph_capture_pipeline_mirrored",
           "apc_graph_launch", "apc_graph_destroy",
           "apc_graph_kernel_count", "apc_profile_enable", "apc_profile_report", "apc_pack_xyzi",
           "apc_split_xyzi"]


class ApcError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(msg)
        self.code = code


def check(ctx_handle, rc):
    if rc != APC_OK:
        msg = lib.apc_last_error(ctx_handle)
        raise ApcError(rc, msg.decode() if msg else f"apc error {rc}")
