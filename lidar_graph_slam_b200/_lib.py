"""ctypes loader for liblgs_b200.so (the C-ABI declared in include/lgs_c.h).

The library is the product: there is no Python or CPU fallback.  Importing this module without the built
shared object, or calling into it on a box without a CUDA device, fails loudly.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "liblgs_b200.so")

LGS_OK = 0


class LgsError(RuntimeError):
    pass


class VoxelGridInfo(C.Structure):
    _fields_ = [("status", C.c_int32), ("reserved", C.c_int32), ("n_kept", C.c_int64), ("n_out", C.c_int64),
                ("min_b", C.c_int32 * 3), ("max_b", C.c_int32 * 3), ("div_b", C.c_int32 * 3)]


class SorInfo(C.Structure):
    _fields_ = [("n_out", C.c_int64), ("mean", C.c_double), ("stddev", C.c_double), ("threshold", C.c_double)]


class Pc2Layout(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("point_step", C.c_uint32), ("row_step", C.c_uint32),
                ("offset_x", C.c_int32), ("offset_y", C.c_int32), ("offset_z", C.c_int32), ("datatype_xyz", C.c_int32),
                ("offset_intensity", C.c_int32), ("datatype_intensity", C.c_int32), ("is_bigendian", C.c_int32), ("reserved", C.c_int32)]


class AlignResult(C.Structure):
    _fields_ = [("T", C.c_float * 16), ("fitness", C.c_double), ("trans_probability", C.c_double), ("iterations", C.c_int32),
                ("converged", C.c_int32), ("evaluations", C.c_int32), ("line_search_trials", C.c_int32),
                ("hessian_recomputes", C.c_int32), ("pair_id", C.c_int32)]


class NdtGridInfo(C.Structure):
    _fields_ = [("refused", C.c_int32), ("dense", C.c_int32), ("n_voxels", C.c_int64), ("n_valid", C.c_int64),
                ("min_b", C.c_int32 * 3), ("max_b", C.c_int32 * 3), ("div_b", C.c_int32 * 3), ("reserved", C.c_int32)]


class BatchParams(C.Structure):
    _fields_ = [("method", C.c_int32), ("max_iterations", C.c_int32), ("transformation_epsilon", C.c_double),
                ("max_correspondence_distance", C.c_double), ("k_correspondences", C.c_int32), ("ndt_resolution", C.c_float),
                ("ndt_step_size", C.c_double), ("submap_leaf", C.c_float), ("fitness_max_range", C.c_double),
                ("n_workers", C.c_int32), ("max_optimizer_iterations", C.c_int32), ("euclidean_fitness_epsilon", C.c_double)]


class BatchDistInfo(C.Structure):
    _fields_ = [("rank", C.c_int32), ("world", C.c_int32), ("n_local", C.c_int64), ("n_received", C.c_int64), ("gather_bytes", C.c_int64),
                ("verify_ms", C.c_double), ("gather_ms", C.c_double)]


class OdometryParams(C.Structure):
    _fields_ = [("method", C.c_int32), ("max_iterations", C.c_int32), ("transformation_epsilon", C.c_double),
                ("max_correspondence_distance", C.c_double), ("k_correspondences", C.c_int32), ("ndt_resolution", C.c_float),
                ("ndt_step_size", C.c_double), ("max_optimizer_iterations", C.c_int32), ("max_scan_accumulate_num", C.c_int32),
                ("keyframe_displacement", C.c_double), ("range_min", C.c_double), ("leaf", C.c_float), ("sor_mean_k", C.c_int32),
                ("sor_stddev_mul", C.c_double), ("base_from_sensor", C.c_float * 16)]


class OdometryFrame(C.Structure):
    _fields_ = [("T", C.c_float * 16), ("trans_probability", C.c_double), ("accum_distance", C.c_double), ("sequence", C.c_int32),
                ("frame", C.c_int32), ("converged", C.c_int32), ("iterations", C.c_int32), ("evaluations", C.c_int32),
                ("keyframe_id", C.c_int32), ("n_source", C.c_int64)]


class OdometryDistInfo(C.Structure):
    _fields_ = [("rank", C.c_int32), ("world", C.c_int32), ("n_local_sequences", C.c_int64), ("n_local_frames", C.c_int64),
                ("n_received", C.c_int64), ("gather_bytes", C.c_int64), ("run_ms", C.c_double), ("gather_ms", C.c_double)]


# every symbol include/lgs_c.h declares: name -> (restype, argtypes)
_vp, _i32, _i64, _f32, _f64 = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_double
SYMBOLS = {
    "lgs_ctx_create": (_i32, [_i32, _vp, C.POINTER(_vp)]),
    "lgs_ctx_destroy": (None, [_vp]),
    "lgs_ctx_synchronize": (_i32, [_vp]),
    "lgs_last_error": (C.c_char_p, []),
    "lgs_version": (C.c_char_p, []),
    "lgs_ctx_launch_count": (_i64, [_vp]),
    "lgs_voxelgrid_filter": (_i32, [_vp, _vp, _i64, _i32, _vp, _i32, _f64, _vp, _vp, _vp, _vp, C.POINTER(VoxelGridInfo)]),
    "lgs_voxelgrid_filter_dev": (_i32, [_vp, _vp, _i64, _vp, _i32, _f64, _vp, _vp, _vp, _vp, C.POINTER(VoxelGridInfo)]),
    "lgs_voxelgrid_filter_wide": (_i32, [_vp, _vp, _i64, _i32, _vp, _i32, _f64, _vp, _vp, _vp, _vp, C.POINTER(VoxelGridInfo)]),
    "lgs_voxelgrid_filter_wide_dev": (_i32, [_vp, _vp, _i64, _vp, _i32, _f64, _vp, _vp, _vp, _vp, C.POINTER(VoxelGridInfo)]),
    "lgs_cloud_from_pointcloud2": (_i32, [_vp, _vp, C.POINTER(Pc2Layout), _vp, C.POINTER(_i64)]),
    "lgs_sor_create": (_i32, [_vp, C.POINTER(_vp)]),
    "lgs_sor_destroy": (None, [_vp]),
    "lgs_sor_set_mean_k": (_i32, [_vp, _i32]),
    "lgs_sor_set_stddev_mul_thresh": (_i32, [_vp, _f64]),
    "lgs_sor_set_negative": (_i32, [_vp, _i32]),
    "lgs_sor_filter": (_i32, [_vp, _vp, _i64, _i32, _vp, _vp, _vp, C.POINTER(SorInfo)]),
    "lgs_sor_filter_dev": (_i32, [_vp, _vp, _i64, _vp, _vp, _vp, C.POINTER(SorInfo)]),
    "lgs_ndt_create": (_i32, [_vp, C.POINTER(_vp)]),
    "lgs_ndt_destroy": (None, [_vp]),
    "lgs_ndt_set_resolution": (_i32, [_vp, _f32]),
    "lgs_ndt_set_step_size": (_i32, [_vp, _f64]),
    "lgs_ndt_set_transformation_epsilon": (_i32, [_vp, _f64]),
    "lgs_ndt_set_maximum_iterations": (_i32, [_vp, _i32]),
    "lgs_ndt_set_outlier_ratio": (_i32, [_vp, _f64]),
    "lgs_ndt_set_search_method": (_i32, [_vp, _i32]),
    "lgs_ndt_set_exact_newton_step": (_i32, [_vp, _i32]),
    "lgs_ndt_set_target": (_i32, [_vp, _vp, _i64, _i32]),
    "lgs_ndt_set_source": (_i32, [_vp, _vp, _i64, _i32]),
    "lgs_ndt_set_target_dev": (_i32, [_vp, _vp, _i64]),
    "lgs_ndt_set_source_dev": (_i32, [_vp, _vp, _i64]),
    "lgs_ndt_set_target_keyframes": (_i32, [_vp, _vp, _vp, _i32, C.POINTER(_i32)]),
    "lgs_ndt_align": (_i32, [_vp, _vp, C.POINTER(AlignResult), _vp]),
    "lgs_ndt_align_many": (_i32, [_vp, _i32, _vp, _vp, C.POINTER(AlignResult), _vp]),
    "lgs_ndt_fitness": (_i32, [_vp, _f64, C.POINTER(_f64)]),
    "lgs_ndt_calculate_score": (_i32, [_vp, _vp, C.POINTER(_f64)]),
    "lgs_ndt_grid_info_get": (_i32, [_vp, C.POINTER(NdtGridInfo)]),
    "lgs_ndt_export_voxels": (_i32, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "lgs_ndt_derivatives": (_i32, [_vp, _vp, _vp, _i32, C.POINTER(_f64), _vp, _vp]),
    "lgs_ndt_convert_transform": (_i32, [_vp, _vp]),
    "lgs_ndt_profile": (_i32, [_vp, _i32, _vp]),
    "lgs_ndt_align_breakdown": (_i32, [_vp, _vp]),
    "lgs_gicp_create": (_i32, [_vp, C.POINTER(_vp)]),
    "lgs_gicp_destroy": (None, [_vp]),
    "lgs_gicp_set_correspondence_randomness": (_i32, [_vp, _i32]),
    "lgs_gicp_set_max_correspondence_distance": (_i32, [_vp, _f64]),
    "lgs_gicp_set_transformation_epsilon": (_i32, [_vp, _f64]),
    "lgs_gicp_set_rotation_epsilon": (_i32, [_vp, _f64]),
    "lgs_gicp_set_maximum_iterations": (_i32, [_vp, _i32]),
    "lgs_gicp_set_regularization_method": (_i32, [_vp, _i32]),
    "lgs_gicp_set_initial_lambda_factor": (_i32, [_vp, _f64]),
    "lgs_gicp_set_source": (_i32, [_vp, _vp, _i64, _i32]),
    "lgs_gicp_set_target": (_i32, [_vp, _vp, _i64, _i32]),
    "lgs_gicp_set_source_dev": (_i32, [_vp, _vp, _i64]),
    "lgs_gicp_set_target_dev": (_i32, [_vp, _vp, _i64]),
    "lgs_gicp_swap_source_and_target": (_i32, [_vp]),
    "lgs_gicp_clear_source": (_i32, [_vp]),
    "lgs_gicp_clear_target": (_i32, [_vp]),
    "lgs_gicp_align": (_i32, [_vp, _vp, C.POINTER(AlignResult), _vp]),
    "lgs_gicp_fitness": (_i32, [_vp, _f64, C.POINTER(_f64)]),
    "lgs_gicp_final_hessian": (_i32, [_vp, _vp]),
    "lgs_gicp_export_covariances": (_i32, [_vp, _i32, _vp]),
    "lgs_gicp_evaluate_cost": (_i32, [_vp, _vp, C.POINTER(_f64)]),
    "lgs_gicp_set_covariances": (_i32, [_vp, _i32, _vp, _i64]),
    "lgs_gicp_linearize": (_i32, [_vp, _vp, C.POINTER(_f64), _vp, _vp, _vp]),
    "lgs_gicp_omp_create": (_i32, [_vp, C.POINTER(_vp)]),
    "lgs_gicp_omp_destroy": (None, [_vp]),
    "lgs_gicp_omp_set_correspondence_randomness": (_i32, [_vp, _i32]),
    "lgs_gicp_omp_set_max_correspondence_distance": (_i32, [_vp, _f64]),
    "lgs_gicp_omp_set_transformation_epsilon": (_i32, [_vp, _f64]),
    "lgs_gicp_omp_set_rotation_epsilon": (_i32, [_vp, _f64]),
    "lgs_gicp_omp_set_maximum_iterations": (_i32, [_vp, _i32]),
    "lgs_gicp_omp_set_maximum_optimizer_iterations": (_i32, [_vp, _i32]),
    "lgs_gicp_omp_set_source": (_i32, [_vp, _vp, _i64, _i32]),
    "lgs_gicp_omp_set_target": (_i32, [_vp, _vp, _i64, _i32]),
    "lgs_gicp_omp_set_source_dev": (_i32, [_vp, _vp, _i64]),
    "lgs_gicp_omp_set_target_dev": (_i32, [_vp, _vp, _i64]),
    "lgs_gicp_omp_align": (_i32, [_vp, _vp, C.POINTER(AlignResult), _vp]),
    "lgs_gicp_omp_fitness": (_i32, [_vp, _f64, C.POINTER(_f64)]),
    "lgs_gicp_omp_export_covariances": (_i32, [_vp, _i32, _vp]),
    "lgs_gicp_omp_functor": (_i32, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "lgs_icp_create": (_i32, [_vp, C.POINTER(_vp)]),
    "lgs_icp_destroy": (None, [_vp]),
    "lgs_icp_set_max_correspondence_distance": (_i32, [_vp, _f64]),
    "lgs_icp_set_maximum_iterations": (_i32, [_vp, _i32]),
    "lgs_icp_set_transformation_epsilon": (_i32, [_vp, _f64]),
    "lgs_icp_set_transformation_rotation_epsilon": (_i32, [_vp, _f64]),
    "lgs_icp_set_euclidean_fitness_epsilon": (_i32, [_vp, _f64]),
    "lgs_icp_reset_convergence_criteria": (_i32, [_vp]),
    "lgs_icp_set_source": (_i32, [_vp, _vp, _i64, _i32]),
    "lgs_icp_set_target": (_i32, [_vp, _vp, _i64, _i32]),
    "lgs_icp_set_source_dev": (_i32, [_vp, _vp, _i64]),
    "lgs_icp_set_target_dev": (_i32, [_vp, _vp, _i64]),
    "lgs_icp_align": (_i32, [_vp, _vp, C.POINTER(AlignResult), _vp]),
    "lgs_icp_fitness": (_i32, [_vp, _f64, C.POINTER(_f64)]),
    "lgs_icp_step": (_i32, [_vp, _vp, _vp, _vp, C.POINTER(_i32)]),
    "lgs_knn": (_i32, [_vp, _vp, _i64, _i32, _vp, _i64, _i32, _i32, _vp, _vp]),
    "lgs_nn_search1": (_i32, [_vp, _vp, _i64, _i32, _vp, _i64, _i32, _vp, _vp, _vp]),
    "lgs_sort_pairs": (_i32, [_vp, _vp, _vp, _i64, _i32]),
    "lgs_linalg_batch": (_i32, [_vp, _i32, _i64, _vp, _vp]),
    "lgs_grid_fold_check": (_i32, [_vp, _vp, _i32, _i32, _i32, _vp]),
    "lgs_keyframes_create": (_i32, [_vp, C.POINTER(_vp)]),
    "lgs_keyframes_destroy": (None, [_vp]),
    "lgs_keyframes_push": (_i32, [_vp, _vp, _i64, _i32, _vp, C.POINTER(_i32)]),
    "lgs_keyframes_push_dev": (_i32, [_vp, _vp, _i64, _vp, C.POINTER(_i32)]),
    "lgs_keyframes_set_pose": (_i32, [_vp, _i32, _vp]),
    "lgs_keyframes_size": (_i32, [_vp, C.POINTER(_i64), C.POINTER(_i64)]),
    "lgs_keyframes_assemble": (_i32, [_vp, _vp, _i32, _f32, C.POINTER(_vp), C.POINTER(_i64)]),
    "lgs_keyframes_export_map": (_i32, [_vp, _vp, _i32, _f32, C.POINTER(_vp), C.POINTER(_i64), C.POINTER(VoxelGridInfo)]),
    "lgs_keyframes_set_accum_distance": (_i32, [_vp, _i32, _f64]),
    "lgs_keyframes_set_position": (_i32, [_vp, _i32, _vp]),
    "lgs_keyframes_detect_loop": (_i32, [_vp, _i32, _f64, _f64, _vp, _i32, C.POINTER(_i32), C.POINTER(_i32)]),
    "lgs_batch_align_keyframes": (_i32, [_vp, _vp, C.POINTER(BatchParams), _i64, _vp, _vp, _i32, _vp, _i32, _vp, _vp]),
    "lgs_batch_align": (_i32, [_i32, _vp, C.POINTER(BatchParams), _i64, _vp, _vp, _vp, _vp, _i32, _vp, _i32, _vp, _vp]),
    "lgs_odometry_run": (_i32, [_vp, C.POINTER(OdometryParams), _i32, _vp, _vp, _vp, _i32, _vp, _vp, _vp]),
    "lgs_odometry_run_dev": (_i32, [_vp, C.POINTER(OdometryParams), _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "lgs_odometry_profile": (_i32, [_vp]),
    "lgs_odometry_run_dist": (_i32, [_vp, _vp, C.POINTER(OdometryParams), _i32, _vp, _vp, _vp, _i32, _vp, _vp, C.POINTER(OdometryDistInfo)]),
    "lgs_odometry_run_dist_dev": (_i32, [_vp, _vp, C.POINTER(OdometryParams), _i32, _vp, _vp, _vp, _vp, _vp, C.POINTER(OdometryDistInfo)]),
    "lgs_batch_release": (None, []),
    "lgs_comm_get_unique_id": (_i32, [_vp]),
    "lgs_comm_init_rank": (_i32, [_vp, _i32, _i32, _i32, C.POINTER(_vp)]),
    "lgs_comm_adopt": (_i32, [_vp, _i32, C.POINTER(_vp)]),
    "lgs_comm_destroy": (None, [_vp]),
    "lgs_comm_info": (_i32, [_vp, C.POINTER(_i32), C.POINTER(_i32), C.POINTER(_i32)]),
    "lgs_batch_partition": (_i32, [_vp, _i64, _i32, _i32, _vp, _i64, C.POINTER(_i64)]),
    "lgs_batch_align_keyframes_dist": (_i32, [_vp, _vp, C.POINTER(BatchParams), _i64, _vp, _vp, _i32, _vp, _vp, C.POINTER(BatchDistInfo)]),
    "lgs_batch_align_dist": (_i32, [_vp, C.POINTER(BatchParams), _i64, _vp, _vp, _vp, _vp, _i32, _vp, _vp, C.POINTER(BatchDistInfo)]),
}

_lib = None


def load():
    """Loads liblgs_b200.so and binds every symbol of include/lgs_c.h.  Raises if anything is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise LgsError("%s is missing: build it with `python -m lidar_graph_slam_b200.build` (nvcc, sm_100a). "
                       "There is no CPU fallback." % SO_PATH)
    lib = C.CDLL(SO_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the export is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != LGS_OK:
        msg = load().lgs_last_error()
        raise LgsError("liblgs_b200 error %d: %s" % (rc, msg.decode("utf-8", "replace") if msg else "?"))
