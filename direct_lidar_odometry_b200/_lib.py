"""Loader and ctypes prototypes for csrc/libnanogicp_b200.so (C ABI in include/nanogicp_c.h).

There is no CPU fallback: if the CUDA library is missing or cannot be loaded this raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("NGICP_LIB_PATH") or os.path.join(_HERE, "csrc", "libnanogicp_b200.so")   # override: A/B builds of the same library

OK, E_INVALID, E_STATE, E_TOO_FEW_POINTS, E_COV_SIZE, E_CUDA, E_UNSUPPORTED, E_COMM, W_VOXEL_OVERFLOW = 0, -1, -2, -3, -4, -5, -6, -7, 1
REG_NONE, REG_MIN_EIG, REG_NORMALIZED_MIN_EIG, REG_PLANE, REG_FROBENIUS = range(5)
OPT_GAUSS_NEWTON, OPT_LEVENBERG_MARQUARDT = 0, 1
SOURCE, TARGET = 0, 1
ALIGN_FUSED, ALIGN_STEPPED = 0, 1
KNN_AUTO, KNN_WARP, KNN_TILE = 0, 1, 2

# every symbol include/nanogicp_c.h declares (checked by tests/test_abi.py)
EXPORTS = [
    "ngicp_create", "ngicp_destroy", "ngicp_last_error", "ngicp_set_stream", "ngicp_get_stream", "ngicp_sync",
    "ngicp_get_timings", "ngicp_params_default", "ngicp_set_params", "ngicp_get_params", "ngicp_set_source",
    "ngicp_set_target", "ngicp_register_source", "ngicp_share_source", "ngicp_share_source_covs", "ngicp_swap",
    "ngicp_clear_source", "ngicp_clear_target", "ngicp_cloud_size", "ngicp_calc_source_covs", "ngicp_calc_target_covs",
    "ngicp_set_source_covs", "ngicp_set_target_covs", "ngicp_clear_covs", "ngicp_covs_size", "ngicp_get_source_covs",
    "ngicp_get_target_covs", "ngicp_align", "ngicp_transform_source", "ngicp_voxel_filter", "ngicp_voxel_assignment",
    "ngicp_knn", "ngicp_linearize", "ngicp_compute_error", "ngicp_linearize_partial", "ngicp_compute_error_partial",
    "ngicp_version", "ngicp_launch_count", "ngicp_grid_info", "ngicp_set_owner_slab", "ngicp_lm_trial",
    "ngicp_lm_is_converged", "ngicp_comm_export", "ngicp_comm_connect", "ngicp_comm_connect_local", "ngicp_comm_close", "ngicp_comm_reset", "ngicp_preprocess", "ngicp_preprocess_pointcloud2", "ngicp_calc_source_covs_part", "ngicp_covs_device", "ngicp_transform_voxel_filter", "ngicp_kfstore_create", "ngicp_kfstore_destroy", "ngicp_kfstore_size",
    "ngicp_kfstore_points", "ngicp_kfstore_push", "ngicp_kfstore_set_target", "ngicp_cov_neighbors", "ngicp_align_batch", "ngicp_imu_prior",
    "ngicp_nn1_packed", "ngicp_linearize_won", "ngicp_fitness_score", "ngicp_fitness_batch",
    "ngicp_submap_push_indices", "ngicp_submap_convex_hull", "ngicp_submap_concave_hull", "ngicp_submap_selector_create",
    "ngicp_submap_selector_destroy", "ngicp_submap_select", "ngicp_submap_selector_hulls", "ngicp_keyframe_wanted",
]


class Params(C.Structure):
    _fields_ = [("k_correspondences", C.c_int), ("max_correspondence_distance", C.c_double),
                ("max_iterations", C.c_int), ("transformation_epsilon", C.c_double), ("rotation_epsilon", C.c_double),
                ("optimizer", C.c_int), ("lm_max_iterations", C.c_int), ("lm_init_lambda_factor", C.c_double),
                ("regularization_method", C.c_int), ("grid_cell_size", C.c_float), ("grid_table_cells", C.c_int),
                ("align_mode", C.c_int), ("knn_path", C.c_int), ("knn_tile_min_points", C.c_int),
                ("voxel_path", C.c_int), ("index_path", C.c_int)]


class Result(C.Structure):
    _fields_ = [("final_transformation", C.c_float * 16), ("final_x", C.c_double * 16),
                ("final_hessian", C.c_double * 36), ("lm_lambda", C.c_double), ("last_error", C.c_double),
                ("nr_iterations", C.c_int), ("converged", C.c_int), ("n_linearize", C.c_int),
                ("n_compute_error", C.c_int), ("lm_failed", C.c_int), ("reserved", C.c_int)]


class Timings(C.Structure):
    _fields_ = [("set_source_ms", C.c_float), ("set_target_ms", C.c_float), ("source_covs_ms", C.c_float),
                ("target_covs_ms", C.c_float), ("align_ms", C.c_float), ("voxel_ms", C.c_float),
                ("reserved", C.c_float * 10)]


_LIB = None


def load() -> C.CDLL:
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `make -C direct_lidar_odometry_b200/csrc` "
            "(or __graft_entry__.build()).  This package has no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, sz, i32, f32 = C.c_void_p, C.c_size_t, C.c_int, C.c_float
    dp, fp, ip = C.POINTER(C.c_double), C.POINTER(C.c_float), C.POINTER(C.c_int)

    def proto(name, res, *args):
        f = getattr(L, name)
        f.restype = res
        f.argtypes = list(args)

    proto("ngicp_create", i32, i32, C.POINTER(vp))
    proto("ngicp_destroy", None, vp)
    proto("ngicp_last_error", C.c_char_p, vp)
    proto("ngicp_set_stream", i32, vp, vp)
    proto("ngicp_get_stream", vp, vp)
    proto("ngicp_sync", i32, vp)
    proto("ngicp_get_timings", i32, vp, C.POINTER(Timings))
    proto("ngicp_params_default", None, C.POINTER(Params))
    proto("ngicp_set_params", i32, vp, C.POINTER(Params))
    proto("ngicp_get_params", i32, vp, C.POINTER(Params))
    for n in ("ngicp_set_source", "ngicp_set_target", "ngicp_register_source"):
        proto(n, i32, vp, vp, sz, sz)
    proto("ngicp_share_source", i32, vp, vp)
    proto("ngicp_share_source_covs", i32, vp, vp)
    for n in ("ngicp_swap", "ngicp_clear_source", "ngicp_clear_target", "ngicp_calc_source_covs", "ngicp_calc_target_covs"):
        proto(n, i32, vp)
    proto("ngicp_cloud_size", sz, vp, i32)
    proto("ngicp_covs_size", sz, vp, i32)
    proto("ngicp_clear_covs", i32, vp, i32)
    for n in ("ngicp_set_source_covs", "ngicp_set_target_covs", "ngicp_get_source_covs", "ngicp_get_target_covs"):
        proto(n, i32, vp, vp, sz)
    proto("ngicp_align", i32, vp, fp, C.POINTER(Result))
    proto("ngicp_align_batch", i32, C.POINTER(vp), sz, fp, C.POINTER(Result))
    proto("ngicp_transform_source", i32, vp, fp, vp, sz)
    proto("ngicp_fitness_score", i32, vp, fp, C.c_double, dp, C.POINTER(sz))
    proto("ngicp_fitness_batch", i32, C.POINTER(vp), sz, fp, C.c_double, dp, C.POINTER(sz))
    proto("ngicp_voxel_filter", i32, vp, vp, sz, sz, f32, vp, sz, C.POINTER(sz))
    proto("ngicp_voxel_assignment", i32, vp, ip, sz)
    proto("ngicp_transform_voxel_filter", i32, vp, vp, sz, sz, fp, f32, vp, sz, C.POINTER(sz))
    proto("ngicp_preprocess", i32, vp, vp, sz, sz, fp, fp, f32, vp, sz, C.POINTER(sz))
    proto("ngicp_preprocess_pointcloud2", i32, vp, vp, vp, fp, fp, f32, vp, sz, C.POINTER(sz))
    proto("ngicp_calc_source_covs_part", i32, vp, i32, i32)
    proto("ngicp_covs_device", i32, vp, i32, C.POINTER(vp), C.POINTER(sz))
    proto("ngicp_knn", i32, vp, i32, vp, sz, sz, i32, ip, fp)
    proto("ngicp_cov_neighbors", i32, vp, i32, ip, fp)
    proto("ngicp_linearize", i32, vp, dp, dp, dp, dp, ip, fp, dp)
    proto("ngicp_compute_error", i32, vp, dp, dp)
    proto("ngicp_linearize_partial", i32, vp, dp, vp)
    proto("ngicp_nn1_packed", i32, vp, dp, C.c_uint, vp)
    proto("ngicp_linearize_won", i32, vp, dp, C.c_uint, vp, vp)
    proto("ngicp_compute_error_partial", i32, vp, dp, vp)
    proto("ngicp_version", C.c_char_p)
    proto("ngicp_launch_count", C.c_ulonglong)
    proto("ngicp_grid_info", i32, vp, i32, fp, ip, ip)
    proto("ngicp_set_owner_slab", i32, vp, i32, f32, f32)
    proto("ngicp_lm_trial", i32, dp, dp, C.c_double, dp, dp, dp, dp)
    proto("ngicp_lm_is_converged", i32, dp, C.c_double, C.c_double)
    proto("ngicp_imu_prior", i32, dp, dp, sz, C.c_double, C.c_double, fp)
    proto("ngicp_submap_push_indices", i32, fp, ip, i32, i32, ip, i32)
    proto("ngicp_submap_convex_hull", i32, fp, i32, ip, i32)
    proto("ngicp_submap_concave_hull", i32, fp, i32, C.c_double, ip, i32)
    proto("ngicp_submap_selector_create", i32, i32, i32, i32, C.c_double, C.POINTER(vp))
    proto("ngicp_submap_selector_destroy", None, vp)
    proto("ngicp_submap_select", i32, vp, fp, i32, fp, ip, i32, ip)
    proto("ngicp_submap_selector_hulls", i32, vp, i32, ip, i32)
    proto("ngicp_keyframe_wanted", i32, fp, fp, i32, fp, fp, C.c_double, C.c_double)
    proto("ngicp_kfstore_create", i32, i32, C.POINTER(vp))
    proto("ngicp_kfstore_destroy", None, vp)
    proto("ngicp_kfstore_size", sz, vp)
    proto("ngicp_kfstore_points", sz, vp, sz)
    proto("ngicp_kfstore_push", i32, vp, vp, C.POINTER(sz))
    proto("ngicp_kfstore_set_target", i32, vp, vp, ip, sz)
    proto("ngicp_comm_export", i32, vp, vp)
    proto("ngicp_comm_connect", i32, vp, i32, i32, vp)
    proto("ngicp_comm_connect_local", i32, vp, i32, i32, C.POINTER(vp))
    proto("ngicp_comm_close", i32, vp)
    proto("ngicp_comm_reset", i32, vp)
    _LIB = L
    return L
