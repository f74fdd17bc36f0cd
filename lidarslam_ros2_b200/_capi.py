"""ctypes loader of the C-ABI library (include/b200reg.h). There is no fallback: if the CUDA library is missing
or cannot be loaded this module raises, and every compute call goes through sm_100a kernels."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
REPO_ROOT = os.path.dirname(_HERE)
LIB_PATH = os.path.join(_HERE, "csrc", os.environ.get("B200REG_LIB_VARIANT", "libb200reg.so"))  # variant: developer A/B builds

OK, ERR_ARG, ERR_NO_TARGET, ERR_NO_SOURCE, ERR_CUDA, ERR_TIMEOUT, ERR_GRID = 0, -1, -2, -3, -4, -5, -6
NDT, GICP = 0, 1
KDTREE, DIRECT26, DIRECT7, DIRECT1 = 0, 1, 2, 3

# every symbol include/b200reg.h declares
SYMBOLS = [
    "b200reg_create", "b200reg_destroy", "b200reg_last_error",
    "b200reg_set_transformation_epsilon", "b200reg_set_maximum_iterations",
    "b200reg_set_max_correspondence_distance", "b200reg_set_euclidean_fitness_epsilon",
    "b200reg_set_ransac_iterations",
    "b200reg_ndt_set_resolution", "b200reg_ndt_set_step_size", "b200reg_ndt_set_outlier_ratio",
    "b200reg_ndt_set_neighborhood_search_method", "b200reg_ndt_set_num_threads",
    "b200reg_ndt_get_transformation_probability", "b200reg_ndt_get_final_num_iteration",
    "b200reg_ndt_calculate_score",
    "b200reg_gicp_set_rotation_epsilon", "b200reg_gicp_set_correspondence_randomness",
    "b200reg_gicp_set_maximum_optimizer_iterations", "b200reg_gicp_set_epsilon",
    "b200reg_set_input_target", "b200reg_set_input_source",
    "b200reg_set_input_target_device", "b200reg_set_input_source_device",
    "b200reg_align", "b200reg_get_final_transformation", "b200reg_has_converged",
    "b200reg_get_fitness_score", "b200reg_get_aligned", "b200reg_align_batch",
    "b200reg_ndt_align_batch", "b200reg_ndt_align_batch_device", "b200reg_ndt_set_batch_slots", "b200reg_ndt_sweep",
    "b200reg_gicp_align_batch", "b200reg_gicp_align_batch_device",
    "b200reg_ndt_attach_pose_board", "b200reg_ndt_gathered_poses",
    "b200reg_voxelgrid", "b200reg_get_stats", "b200reg_ndt_derivatives", "b200reg_ndt_hessian_radius",
    "b200reg_ndt_num_voxels", "b200reg_ndt_get_voxels", "b200reg_nn1",
    "b200reg_gicp_get_covariances", "b200reg_gicp_num_correspondences", "b200reg_get_kind",
    "b200sm_create", "b200sm_destroy", "b200sm_last_error", "b200sm_set_params", "b200sm_set_initial_pose",
    "b200sm_set_scan", "b200sm_update_map", "b200sm_receive_cloud", "b200sm_num_submaps", "b200sm_get_targeted",
    "b200sm_get_submap", "b200sm_get_filtered_scan", "b200sm_get_stats", "b200sm_search_loop", "b200sm_search_loop_all", "b200sm_import_submap",
    "b200sm_imu_set_scan_period", "b200sm_imu_push", "b200sm_deskew_next_scan", "b200sm_imu_adjust_distortion",
    "b200sm_imu_get_state", "b200sm_imu_get_sample",
    # include/b200comm.h
    "b200comm_unique_id", "b200comm_create", "b200comm_destroy", "b200comm_all_gather_rows", "b200comm_rank", "b200comm_last_error",
    "b200comm_board_create", "b200comm_board_destroy", "b200comm_board_info",
]


class SmLoopResult(C.Structure):
    _fields_ = [("is_candidate", C.c_int), ("id_min", C.c_int), ("accepted", C.c_int), ("pad", C.c_int),
                ("min_dist", C.c_double), ("fitness", C.c_double), ("final_T", C.c_float * 16),
                ("relative_pose", C.c_double * 16), ("n_source", C.c_size_t), ("n_target", C.c_size_t)]


class SmStats(C.Structure):
    _fields_ = [("n_scan", C.c_size_t), ("n_filtered", C.c_size_t), ("n_targeted", C.c_size_t), ("n_submaps", C.c_size_t),
                ("kernel_launches", C.c_int), ("trans", C.c_double), ("latest_distance", C.c_double)]


class BatchResult(C.Structure):
    _fields_ = [("final_T", C.c_float * 16), ("trans_probability", C.c_double), ("converged", C.c_int), ("iterations", C.c_int),
                ("evaluations", C.c_int), ("status", C.c_int), ("hits_total", C.c_longlong)]


class GicpBatchResult(C.Structure):
    _fields_ = [("final_T", C.c_float * 16), ("converged", C.c_int), ("iterations", C.c_int), ("evaluations", C.c_int),
                ("correspondences", C.c_int), ("status", C.c_int), ("pad", C.c_int)]


class SweepResult(C.Structure):
    _fields_ = [("final_T", C.c_float * 16), ("fitness", C.c_double), ("trans_probability", C.c_double), ("converged", C.c_int),
                ("iterations", C.c_int), ("status", C.c_int), ("pad", C.c_int)]


class Stats(C.Structure):
    _fields_ = [
        ("evaluations", C.c_int), ("iterations", C.c_int),
        ("hits", C.c_longlong), ("hits_total", C.c_longlong),
        ("solve_ms", C.c_float), ("target_build_ms", C.c_float),
        ("kernel_launches", C.c_int),
        ("grid_ctas", C.c_int), ("block_threads", C.c_int), ("index_in_smem", C.c_int),
        ("n_voxels", C.c_longlong), ("n_cells", C.c_longlong), ("n_source", C.c_longlong), ("n_target", C.c_longlong),
        ("gicp_inner_ms", C.c_float), ("gicp_inner_launches", C.c_int), ("gicp_pair_evaluations", C.c_double),
    ]


def build(force: bool = False) -> str:
    """Compile the sm_100a library in-tree with nvcc (build.sh)."""
    env = dict(os.environ)
    if force:
        for f in os.listdir(os.path.join(_HERE, "csrc")):
            if f.endswith(".o"):
                os.remove(os.path.join(_HERE, "csrc", f))
    subprocess.check_call(["bash", os.path.join(REPO_ROOT, "build.sh")], env=env)
    return LIB_PATH


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    vp, sz, i, d, f = C.c_void_p, C.c_size_t, C.c_int, C.c_double, C.c_float
    L.b200reg_create.argtypes = [i, i, C.POINTER(vp)]
    L.b200reg_destroy.argtypes = [vp]
    L.b200reg_last_error.argtypes = [vp]
    L.b200reg_last_error.restype = C.c_char_p
    for name in ("b200reg_set_transformation_epsilon", "b200reg_set_max_correspondence_distance",
                 "b200reg_set_euclidean_fitness_epsilon", "b200reg_ndt_set_step_size", "b200reg_ndt_set_outlier_ratio",
                 "b200reg_gicp_set_rotation_epsilon", "b200reg_gicp_set_epsilon"):
        getattr(L, name).argtypes = [vp, d]
    for name in ("b200reg_set_maximum_iterations", "b200reg_set_ransac_iterations",
                 "b200reg_ndt_set_neighborhood_search_method", "b200reg_ndt_set_num_threads",
                 "b200reg_gicp_set_correspondence_randomness", "b200reg_gicp_set_maximum_optimizer_iterations"):
        getattr(L, name).argtypes = [vp, i]
    L.b200reg_ndt_set_resolution.argtypes = [vp, f]
    L.b200reg_ndt_get_transformation_probability.argtypes = [vp, C.POINTER(d)]
    L.b200reg_ndt_get_final_num_iteration.argtypes = [vp, C.POINTER(i)]
    L.b200reg_ndt_calculate_score.argtypes = [vp, vp, sz, sz, C.POINTER(d)]
    L.b200reg_set_input_target.argtypes = [vp, vp, sz, sz]
    L.b200reg_set_input_source.argtypes = [vp, vp, sz, sz]
    L.b200reg_set_input_target_device.argtypes = [vp, vp, sz]
    L.b200reg_set_input_source_device.argtypes = [vp, vp, sz]
    L.b200reg_align.argtypes = [vp, vp, vp]
    L.b200reg_get_final_transformation.argtypes = [vp, vp]
    L.b200reg_has_converged.argtypes = [vp, C.POINTER(i)]
    L.b200reg_get_fitness_score.argtypes = [vp, d, C.POINTER(d)]
    L.b200reg_get_aligned.argtypes = [vp, vp, sz]
    L.b200reg_align_batch.argtypes = [vp, i, vp, vp]
    L.b200reg_ndt_align_batch.argtypes = [vp, i, vp, vp, sz, vp, vp]
    L.b200reg_ndt_align_batch_device.argtypes = [vp, i, vp, vp, vp, vp]
    L.b200reg_ndt_set_batch_slots.argtypes = [vp, i]
    L.b200reg_gicp_align_batch.argtypes = [vp, i, vp, vp, sz, vp, vp]
    L.b200reg_gicp_align_batch_device.argtypes = [vp, i, vp, vp, vp, vp]
    L.b200reg_ndt_attach_pose_board.argtypes = [vp, vp]
    L.b200reg_ndt_gathered_poses.argtypes = [vp, vp, vp, i]
    L.b200reg_ndt_sweep.argtypes = [vp, i, vp, vp, vp, vp, sz, vp, d, vp]
    L.b200reg_voxelgrid.argtypes = [i, vp, sz, sz, C.c_long, f, vp, sz, C.POINTER(sz)]
    L.b200reg_get_stats.argtypes = [vp, C.POINTER(Stats)]
    L.b200reg_ndt_derivatives.argtypes = [vp, vp, vp, i, C.POINTER(d), vp, vp]
    L.b200reg_ndt_hessian_radius.argtypes = [vp, vp, vp, vp]
    L.b200reg_ndt_num_voxels.argtypes = [vp, C.POINTER(sz)]
    L.b200reg_ndt_get_voxels.argtypes = [vp, vp, vp, vp, vp, vp]
    L.b200reg_nn1.argtypes = [vp, vp, sz, sz, vp, vp]
    L.b200reg_gicp_get_covariances.argtypes = [vp, i, vp, C.POINTER(sz)]
    L.b200reg_gicp_num_correspondences.argtypes = [vp, C.POINTER(i)]
    L.b200reg_get_kind.argtypes = [vp, C.POINTER(i)]
    L.b200sm_create.argtypes = [i, C.POINTER(vp)]
    L.b200sm_destroy.argtypes = [vp]
    L.b200sm_destroy.restype = None
    L.b200sm_last_error.argtypes = [vp]
    L.b200sm_last_error.restype = C.c_char_p
    L.b200sm_set_params.argtypes = [vp, f, f, i, d, i, d, d]
    L.b200sm_set_initial_pose.argtypes = [vp, vp, vp]
    L.b200sm_set_scan.argtypes = [vp, vp, vp, sz, sz, C.c_long, C.POINTER(sz)]
    L.b200sm_update_map.argtypes = [vp, vp, vp, vp, vp, i]
    L.b200sm_receive_cloud.argtypes = [vp, vp, vp, sz, sz, C.c_long, vp, vp, C.POINTER(i)]
    L.b200sm_num_submaps.argtypes = [vp, C.POINTER(sz)]
    L.b200sm_get_targeted.argtypes = [vp, vp, sz, C.POINTER(sz)]
    L.b200sm_get_submap.argtypes = [vp, sz, vp, sz, C.POINTER(sz), vp, C.POINTER(d)]
    L.b200sm_get_filtered_scan.argtypes = [vp, vp, sz, C.POINTER(sz)]
    L.b200sm_get_stats.argtypes = [vp, C.POINTER(SmStats)]
    L.b200sm_search_loop.argtypes = [vp, vp, f, d, d, d, i, C.POINTER(SmLoopResult)]
    L.b200sm_search_loop_all.argtypes = [vp, vp, f, d, d, d, i, i, i, vp, sz, C.POINTER(sz), C.POINTER(sz)]
    L.b200sm_import_submap.argtypes = [vp, vp, sz, sz, C.c_long, vp, d]
    L.b200sm_imu_set_scan_period.argtypes = [vp, d]
    L.b200sm_imu_push.argtypes = [vp, vp, vp, vp, d]
    L.b200sm_deskew_next_scan.argtypes = [vp, d]
    L.b200sm_imu_adjust_distortion.argtypes = [vp, vp, sz, sz, C.c_long, d]
    L.b200sm_imu_get_state.argtypes = [vp, C.POINTER(i), C.POINTER(i), C.POINTER(i)]
    L.b200sm_imu_get_sample.argtypes = [vp, i, C.POINTER(d), vp, vp, vp]
    L.b200comm_unique_id.argtypes = [vp]
    L.b200comm_create.argtypes = [vp, i, i, i, C.POINTER(vp)]
    L.b200comm_destroy.argtypes = [vp]
    L.b200comm_all_gather_rows.argtypes = [vp, vp, i, i, vp]
    L.b200comm_rank.argtypes = [vp, C.POINTER(i), C.POINTER(i)]
    L.b200comm_board_create.argtypes = [vp, i, C.POINTER(vp)]
    L.b200comm_board_destroy.argtypes = [vp]
    L.b200comm_board_info.argtypes = [vp, C.POINTER(i), C.POINTER(i), C.POINTER(i)]
    L.b200comm_last_error.argtypes = []
    L.b200comm_last_error.restype = C.c_char_p
    for name in SYMBOLS:
        fn = getattr(L, name)
        if name not in ("b200reg_last_error", "b200sm_last_error", "b200sm_destroy", "b200comm_last_error"):
            fn.restype = i
    _lib = L
    return L
