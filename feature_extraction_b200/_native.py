"""ctypes binding of csrc/libfe_b200.so — the C-ABI declared in include/fe_b200.h.

The library is the product: there is no Python or CPU fallback.  Importing this module fails
loudly if the shared object is missing, and creating a context fails if no B200 is visible.
"""
import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libfe_b200.so")

DESC_LEN = 1980
RECORD_FLOATS = 1996

FE_OK, FE_ERR_INVALID, FE_ERR_CUDA, FE_ERR_CAPACITY, FE_ERR_NO_DEVICE, FE_ERR_UNSUPPORTED = range(6)

# every symbol include/fe_b200.h declares
EXPORTS = [
    "fe_params_node_default", "fe_params_launch_playback", "fe_version", "fe_create", "fe_set_params",
    "fe_destroy", "fe_last_error", "fe_device_count", "fe_host_alloc", "fe_host_free",
    "fe_process_batch", "fe_process_batch_layout", "fe_imu_to_roll_pitch", "fe_process_batch_device", "fe_download",
    "fe_multi_create", "fe_multi_process_batch", "fe_multi_destroy", "fe_multi_last_error", "fe_enable_cloud_outputs", "fe_get_cloud_outputs", "fe_enable_record_output", "fe_multi_enable_record_output",
    "fe_get_stage_times", "fe_enable_stage_timing", "fe_timer_begin", "fe_timer_end", "fe_get_batch_stats", "fe_get_elevation_angles", "fe_rotate_cloud", "fe_rotation_matrix",
    "fe_filter_cloud", "fe_extract_clusters", "fe_get_cylinder_segments", "fe_estimate_keypoints",
    "fe_estimate_descriptors", "fe_pack_point_descriptors",
    "fe_set_angle_libm", "fe_enable_boundary_report", "fe_get_boundary_report",
    "fe_enable_boundary_report_all", "fe_get_boundary_report_all",
    "fe_multi_enable_cloud_outputs", "fe_multi_get_cloud_outputs",
    "fe_match_descriptors", "fe_match_descriptors_device",
    "fe_register_params_default", "fe_register_matches", "fe_register_matches_device", "fe_match_device_best",
]


class Params(C.Structure):
    """fe_params_t: the ROS parameters of reference src:9-34."""
    _fields_ = [
        ("x_min", C.c_double), ("x_max", C.c_double),
        ("y_min", C.c_double), ("y_max", C.c_double),
        ("z_min", C.c_double), ("z_max", C.c_double),
        ("cluster_tolerance", C.c_double),
        ("cluster_min_count", C.c_int32), ("cluster_max_count", C.c_int32),
        ("cluster_radius_threshold", C.c_double),
        ("number_detection_channels", C.c_int32),
        ("estimate_descriptors", C.c_int32),
        ("descriptor_radius", C.c_double),
    ]

    def copy(self):
        return Params.from_buffer_copy(self)


class Limits(C.Structure):
    _fields_ = [
        ("max_points_per_call", C.c_int64),
        ("max_scans_per_call", C.c_int32),
        ("max_keypoints_per_call", C.c_int64),
        ("max_ring_clusters_per_call", C.c_int64),
    ]


class PointLayout(C.Structure):
    """fe_point_layout_t: PointCloud2-style record layout (stride = point_step)."""
    _fields_ = [("stride", C.c_int32), ("x_off", C.c_int32), ("y_off", C.c_int32), ("z_off", C.c_int32)]


class BatchResult(C.Structure):
    _fields_ = [
        ("n_scans", C.c_int32),
        ("n_keypoints", C.c_int64),
        ("keypoint_offsets", C.POINTER(C.c_int64)),
        ("keypoints", C.c_void_p),
        ("descriptors", C.c_void_p),
        ("on_device", C.c_int32),
        ("gpu_launches", C.c_int64),
    ]


class MatchResult(C.Structure):
    """fe_match_result_t: per query row, the best reference row and shift, its distance and the second-best row's."""
    _fields_ = [
        ("n_queries", C.c_int64),
        ("best", C.POINTER(C.c_int64)),
        ("shift", C.POINTER(C.c_int32)),
        ("dist2", C.POINTER(C.c_float)),
        ("second_dist2", C.POINTER(C.c_float)),
    ]


class RegisterParams(C.Structure):
    """fe_register_params_t: inlier radius and minimum separation (m), hypothesis cap, inliers for status 2, refinement
    rounds."""
    _fields_ = [
        ("inlier_radius", C.c_double),
        ("min_separation", C.c_double),
        ("max_hypotheses", C.c_int32),
        ("min_inliers", C.c_int32),
        ("refine_iterations", C.c_int32),
    ]


class RegisterResult(C.Structure):
    """fe_register_result_t: per group the motion {c, s, tx, ty}, rms, counts and status; per query row its inlier."""
    _fields_ = [
        ("n_groups", C.c_int32),
        ("n_queries", C.c_int64),
        ("pose", C.POINTER(C.c_double)),
        ("rms", C.POINTER(C.c_double)),
        ("n_inliers", C.POINTER(C.c_int32)),
        ("n_hypotheses", C.POINTER(C.c_int32)),
        ("status", C.POINTER(C.c_int32)),
        ("assoc", C.POINTER(C.c_int64)),
    ]


def build():
    """Compile libfe_b200.so for sm_100a (nvcc cross-compiles without a GPU)."""
    subprocess.check_call(["make", "-s", "-C", os.path.join(_HERE, "csrc")])


_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "feature_extraction_b200: %s is missing — build it with `python -c 'import __graft_entry__ as g; "
                "g.build()'` or `make -C feature_extraction_b200/csrc`.  There is no CPU fallback." % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        L.fe_version.restype = C.c_char_p
        L.fe_last_error.restype = C.c_char_p
        L.fe_last_error.argtypes = [C.c_void_p]
        L.fe_host_alloc.restype = C.c_void_p
        L.fe_host_alloc.argtypes = [C.c_int64]
        L.fe_host_free.argtypes = [C.c_void_p]
        L.fe_create.argtypes = [C.c_int, C.POINTER(Params), C.POINTER(Limits), C.POINTER(C.c_void_p)]
        L.fe_destroy.argtypes = [C.c_void_p]
        L.fe_set_params.argtypes = [C.c_void_p, C.POINTER(Params)]
        L.fe_process_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(BatchResult)]
        L.fe_process_batch_layout.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(PointLayout), C.c_void_p, C.c_void_p, C.c_int32,
                                              C.POINTER(BatchResult)]
        L.fe_imu_to_roll_pitch.argtypes = [C.c_void_p, C.c_int32, C.POINTER(C.c_double), C.POINTER(C.c_double)]
        L.fe_process_batch_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(BatchResult)]
        L.fe_multi_create.argtypes = [C.c_void_p, C.c_int32, C.POINTER(Params), C.POINTER(Limits), C.POINTER(C.c_void_p)]
        L.fe_multi_process_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(BatchResult)]
        L.fe_multi_destroy.argtypes = [C.c_void_p]
        L.fe_multi_last_error.restype = C.c_char_p
        L.fe_multi_last_error.argtypes = [C.c_void_p]
        L.fe_download.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]
        L.fe_enable_cloud_outputs.argtypes = [C.c_void_p, C.c_int32]
        L.fe_enable_record_output.argtypes = [C.c_void_p, C.c_int32]
        L.fe_enable_stage_timing.argtypes = [C.c_void_p, C.c_int32]
        L.fe_multi_enable_record_output.argtypes = [C.c_void_p, C.c_int32]
        L.fe_get_cloud_outputs.argtypes = [C.c_void_p, C.POINTER(C.POINTER(C.c_int64)), C.POINTER(C.c_void_p),
                                           C.POINTER(C.POINTER(C.c_int64)), C.POINTER(C.c_void_p)]
        L.fe_get_stage_times.argtypes = [C.c_void_p, C.c_int32, C.POINTER(C.c_char_p), C.POINTER(C.c_float), C.POINTER(C.c_int32)]
        L.fe_timer_begin.argtypes = [C.c_void_p]
        L.fe_timer_end.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
        L.fe_get_batch_stats.argtypes = [C.c_void_p, C.c_void_p]
        L.fe_get_elevation_angles.argtypes = [C.c_void_p, C.c_void_p, C.c_int64]
        L.fe_rotate_cloud.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_double, C.c_double]
        L.fe_rotation_matrix.argtypes = [C.c_double, C.c_double, C.c_void_p]
        L.fe_filter_cloud.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]
        L.fe_extract_clusters.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_double, C.c_int32, C.c_int32,
                                          C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.POINTER(C.c_int32)]
        L.fe_get_cylinder_segments.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.POINTER(C.c_int64),
                                               C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]
        L.fe_estimate_keypoints.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.POINTER(C.c_int64),
                                            C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]
        L.fe_estimate_descriptors.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]
        L.fe_pack_point_descriptors.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
        L.fe_debug_sort_replay.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
        L.fe_set_angle_libm.argtypes = [C.c_void_p, C.c_int32]
        L.fe_enable_boundary_report.argtypes = [C.c_void_p, C.c_double]
        L.fe_get_boundary_report.argtypes = [C.c_void_p, C.POINTER(C.POINTER(C.c_int64)), C.POINTER(C.c_int32)]
        L.fe_enable_boundary_report_all.argtypes = [C.c_void_p, C.c_double]
        L.fe_get_boundary_report_all.argtypes = [C.c_void_p, C.POINTER(C.POINTER(C.c_int64)), C.POINTER(C.c_int32)]
        L.fe_multi_enable_cloud_outputs.argtypes = [C.c_void_p, C.c_int32]
        L.fe_multi_get_cloud_outputs.argtypes = [C.c_void_p, C.POINTER(C.POINTER(C.c_int64)), C.POINTER(C.c_void_p),
                                                 C.POINTER(C.POINTER(C.c_int64)), C.POINTER(C.c_void_p)]
        for f in (L.fe_match_descriptors, L.fe_match_descriptors_device):
            f.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int32,
                          C.POINTER(MatchResult)]
        L.fe_register_params_default.argtypes = [C.POINTER(RegisterParams)]
        L.fe_register_params_default.restype = None
        for f in (L.fe_register_matches, L.fe_register_matches_device):
            f.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                          C.POINTER(RegisterParams), C.POINTER(RegisterResult)]
        L.fe_match_device_best.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
        L.fe_debug_enable_graphs.argtypes = [C.c_void_p, C.c_int32, C.POINTER(C.c_int64)]
        L.fe_debug_lean_reruns.argtypes = [C.c_void_p, C.POINTER(C.c_int64)]
        L.fe_debug_density_work.argtypes = [C.c_void_p, C.c_void_p]
        L.fe_debug_h2d_probe.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_float)]
        L.fe_debug_force_grid_clustering.argtypes = [C.c_void_p, C.c_int32]
        L.fe_debug_libm_f32.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]
        _LIB = L
    return _LIB
