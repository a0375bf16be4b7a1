"""ctypes binding of the C-ABI in include/dvo_b200.h (libdvo_b200.so).  Fails loudly when the CUDA library is missing."""
import ctypes as C
import os

from . import build as _build

MAX_LEVELS = 6
STAGES = ["h2d", "pyramid", "canny", "edt_rows", "normgrad", "solve", "d2h"]


class Config(C.Structure):
    _fields_ = [("width", C.c_int), ("height", C.c_int), ("levels", C.c_int), ("max_batch", C.c_int), ("device", C.c_int),
                ("keep_now_depth", C.c_int), ("trace_iters", C.c_int)]


class SolverParams(C.Structure):
    _fields_ = [("solver", C.c_int), ("jacobian", C.c_int), ("weight", C.c_int), ("arithmetic", C.c_int),
                ("huber_k", C.c_float), ("lm_lambda0", C.c_double), ("iters", C.c_int * MAX_LEVELS), ("residual", C.c_int)]


class PairInfo(C.Structure):
    _fields_ = [("status", C.c_int), ("npts", C.c_int * MAX_LEVELS), ("best_index", C.c_int * MAX_LEVELS),
                ("iterations_run", C.c_int * MAX_LEVELS), ("best_energy", C.c_float * MAX_LEVELS),
                ("visible_ratio", C.c_float * MAX_LEVELS), ("laplacian_b", C.c_float)]


class CovInfo(C.Structure):
    """dvo_cov_info: status bits (0 no points / edges at the level, 1 nvis < 7, 2 H not positive definite), level, nvis, sigma2, logdet."""
    _fields_ = [("status", C.c_int), ("level", C.c_int), ("nvis", C.c_int), ("sigma2", C.c_double), ("logdet", C.c_double)]


class PhotoConfig(C.Structure):
    _fields_ = [("width", C.c_int), ("height", C.c_int), ("levels", C.c_int), ("max_batch", C.c_int), ("device", C.c_int)]


class PhotoInfo(C.Structure):
    _fields_ = [("status", C.c_int), ("iters_run", C.c_int), ("nreproj", C.c_int), ("sumsq_first", C.c_double),
                ("sumsq_last", C.c_double), ("visible", C.c_double), ("A", C.c_double * 36), ("b", C.c_double * 6)]


class KeyframePolicy(C.Structure):
    _fields_ = [("keyframe_every", C.c_int), ("use_quality_gates", C.c_int), ("laplacian_thresh", C.c_float),
                ("visible_ratio_thresh", C.c_float), ("min_reprojections", C.c_int)]


class PgoParams(C.Structure):
    """dvo_pgo_params: LM iteration cap (damped solves), initial Marquardt damping, relative-decrease stop."""
    _fields_ = [("max_iterations", C.c_int), ("lambda0", C.c_double), ("rel_tol", C.c_double)]


class PgoInfo(C.Structure):
    """dvo_pgo_info: status bits (0 bad edge index, 1 not connected to node 0, 2 H not positive definite), counts, costs."""
    _fields_ = [("status", C.c_int), ("iterations", C.c_int), ("accepted", C.c_int), ("edges_used", C.c_int),
                ("cost_initial", C.c_double), ("cost_final", C.c_double)]


PGO_MAX_LAG = 8

RGBD_MAX_LEVELS = 5


class RgbdConfig(C.Structure):
    _fields_ = [("width", C.c_int), ("height", C.c_int), ("levels", C.c_int), ("max_batch", C.c_int), ("device", C.c_int)]


class RgbdParams(C.Structure):
    _fields_ = [("iterations", C.c_int), ("gradient_threshold", C.c_int), ("min_points", C.c_int), ("max_points", C.c_int),
                ("eps_norm_exit", C.c_double)]


class RgbdInfo(C.Structure):
    _fields_ = [("status", C.c_int), ("npts", C.c_int * RGBD_MAX_LEVELS), ("iters_run", C.c_int * RGBD_MAX_LEVELS),
                ("updates", C.c_int * RGBD_MAX_LEVELS), ("nvis_last", C.c_int * RGBD_MAX_LEVELS),
                ("eps_norm_first", C.c_double * RGBD_MAX_LEVELS), ("eps_norm_last", C.c_double * RGBD_MAX_LEVELS)]


# every symbol include/dvo_b200.h declares
SYMBOLS = [
    "dvo_last_error", "dvo_device_count", "dvo_create", "dvo_destroy", "dvo_set_stream", "dvo_synchronize",
    "dvo_set_intrinsics", "dvo_set_frames", "dvo_set_frames_raw", "dvo_promote_now_to_ref", "dvo_build_pyramids", "dvo_prepare",
    "dvo_set_initial_pose", "dvo_run", "dvo_process", "dvo_join", "dvo_join_stream", "dvo_get_poses", "dvo_align_batch", "dvo_level_dims", "dvo_get_level_buffer",
    "dvo_get_points", "dvo_eval_normal_equations", "dvo_eval_normal_equations_ex", "dvo_get_trace", "dvo_get_energies", "dvo_enable_timing", "dvo_get_stage_ms",
    "dvo_launch_count", "dvo_gop_compose", "dvo_run_sequences", "dvo_run_sequences_gated", "dvo_run_sequences_mem",
    "dvo_pose_covariance", "dvo_run_sequences_cov", "dvo_run_sequences_entropy", "dvo_align_pairs", "dvo_pose_graph_optimize",
    "dvo_photo_create", "dvo_photo_destroy", "dvo_photo_set_stream", "dvo_photo_synchronize", "dvo_photo_launch_count",
    "dvo_photo_set_intrinsics", "dvo_photo_set_frames", "dvo_photo_prepare_ref", "dvo_photo_set_pose", "dvo_photo_estimate",
    "dvo_photo_get_poses", "dvo_photo_get_level", "dvo_photo_get_A", "dvo_photo_eval", "dvo_photo_put_level",
    "dvo_blob_create", "dvo_blob_upload", "dvo_blob_download", "dvo_blob_device_ptr", "dvo_blob_bytes", "dvo_blob_destroy",
    "dvo_undistort",
    "dvo_rgbd_create", "dvo_rgbd_destroy", "dvo_rgbd_set_stream", "dvo_rgbd_synchronize", "dvo_rgbd_launch_count",
    "dvo_rgbd_set_intrinsics", "dvo_rgbd_set_frames", "dvo_rgbd_compute_jacobians", "dvo_rgbd_set_pose", "dvo_rgbd_gauss_newton",
    "dvo_rgbd_get_poses", "dvo_rgbd_level_dims", "dvo_rgbd_get_level", "dvo_rgbd_get_A", "dvo_rgbd_eval",
]

_lib = None


def load(build_if_missing=True):
    """Load libdvo_b200.so (building it in-tree with nvcc when absent).  Raises if it cannot be had."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB
    if build_if_missing:
        path = _build.build_cuda()
    if not os.path.exists(path):
        raise RuntimeError(f"{path} is missing: build it with `python -m rgbd_odometry_b200.build` (no CPU fallback exists)")
    lib = C.CDLL(path)
    lib.dvo_last_error.restype = C.c_char_p
    lib.dvo_launch_count.restype = C.c_longlong
    lib.dvo_launch_count.argtypes = [C.c_void_p]
    lib.dvo_create.argtypes = [C.POINTER(Config), C.POINTER(C.c_void_p)]
    lib.dvo_destroy.argtypes = [C.c_void_p]
    lib.dvo_set_stream.argtypes = [C.c_void_p, C.c_void_p]
    lib.dvo_synchronize.argtypes = [C.c_void_p]
    lib.dvo_set_intrinsics.argtypes = [C.c_void_p, C.c_float, C.c_float, C.c_float, C.c_float]
    lib.dvo_set_frames.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
    lib.dvo_set_frames_raw.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
    lib.dvo_promote_now_to_ref.argtypes = [C.c_void_p, C.c_int, C.c_int]
    lib.dvo_build_pyramids.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int]
    lib.dvo_prepare.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int]
    lib.dvo_set_initial_pose.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int]
    lib.dvo_run.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(SolverParams)]
    lib.dvo_process.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(SolverParams), C.c_void_p]
    lib.dvo_join.argtypes = [C.c_void_p]
    lib.dvo_join_stream.argtypes = [C.c_void_p, C.c_void_p]
    lib.dvo_get_poses.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
    lib.dvo_align_batch.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.POINTER(SolverParams), C.c_void_p, C.c_void_p]
    lib.dvo_level_dims.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.dvo_get_level_buffer.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_size_t]
    lib.dvo_get_points.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int)]
    lib.dvo_eval_normal_equations.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float,
                                              C.c_void_p, C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int),
                                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.dvo_eval_normal_equations_ex.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.POINTER(SolverParams),
                                                 C.c_void_p, C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int),
                                                 C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.dvo_get_trace.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    lib.dvo_get_energies.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int]
    lib.dvo_enable_timing.argtypes = [C.c_void_p, C.c_int]
    lib.dvo_get_stage_ms.argtypes = [C.c_void_p, C.c_void_p]
    lib.dvo_gop_compose.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
    lib.dvo_run_sequences.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.POINTER(SolverParams), C.c_int,
                                      C.c_void_p, C.c_void_p, C.c_void_p]
    lib.dvo_run_sequences_gated.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.POINTER(SolverParams),
                                            C.POINTER(KeyframePolicy), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.dvo_run_sequences_mem.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(SolverParams),
                                          C.POINTER(KeyframePolicy), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.dvo_pose_covariance.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(SolverParams), C.c_int, C.c_void_p, C.c_void_p, C.c_int]
    lib.dvo_align_pairs.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(SolverParams), C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_int]
    lib.dvo_run_sequences_cov.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(SolverParams),
                                          C.POINTER(KeyframePolicy), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.dvo_run_sequences_entropy.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(SolverParams),
                                              C.POINTER(KeyframePolicy), C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                              C.c_void_p, C.c_void_p, C.c_void_p]
    lib.dvo_pose_graph_optimize.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.POINTER(PgoParams), C.c_void_p, C.c_void_p, C.c_int]
    lib.dvo_photo_create.argtypes = [C.POINTER(PhotoConfig), C.POINTER(C.c_void_p)]
    lib.dvo_photo_destroy.argtypes = [C.c_void_p]
    lib.dvo_photo_set_stream.argtypes = [C.c_void_p, C.c_void_p]
    lib.dvo_photo_synchronize.argtypes = [C.c_void_p]
    lib.dvo_photo_launch_count.restype = C.c_longlong
    lib.dvo_photo_launch_count.argtypes = [C.c_void_p]
    lib.dvo_photo_set_intrinsics.argtypes = [C.c_void_p, C.c_double, C.c_double, C.c_double, C.c_double]
    lib.dvo_photo_set_frames.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
    lib.dvo_photo_prepare_ref.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int]
    lib.dvo_photo_set_pose.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    lib.dvo_photo_estimate.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double]
    lib.dvo_photo_get_poses.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    lib.dvo_photo_get_level.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_int]
    lib.dvo_photo_get_A.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    lib.dvo_photo_put_level.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_size_t]
    lib.dvo_blob_create.argtypes = [C.c_size_t, C.c_int, C.POINTER(C.c_void_p)]
    lib.dvo_blob_upload.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    lib.dvo_blob_download.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    lib.dvo_blob_device_ptr.argtypes = [C.c_void_p]
    lib.dvo_blob_device_ptr.restype = C.c_void_p
    lib.dvo_blob_bytes.argtypes = [C.c_void_p]
    lib.dvo_blob_bytes.restype = C.c_size_t
    lib.dvo_blob_destroy.argtypes = [C.c_void_p]
    lib.dvo_photo_eval.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_double, C.c_void_p, C.c_void_p,
                                   C.POINTER(C.c_double), C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_void_p]
    lib.dvo_undistort.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    lib.dvo_rgbd_create.argtypes = [C.POINTER(RgbdConfig), C.POINTER(C.c_void_p)]
    lib.dvo_rgbd_destroy.argtypes = [C.c_void_p]
    lib.dvo_rgbd_set_stream.argtypes = [C.c_void_p, C.c_void_p]
    lib.dvo_rgbd_synchronize.argtypes = [C.c_void_p]
    lib.dvo_rgbd_launch_count.restype = C.c_longlong
    lib.dvo_rgbd_launch_count.argtypes = [C.c_void_p]
    lib.dvo_rgbd_set_intrinsics.argtypes = [C.c_void_p, C.c_double, C.c_double, C.c_double, C.c_double]
    lib.dvo_rgbd_set_frames.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
    lib.dvo_rgbd_compute_jacobians.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int]
    lib.dvo_rgbd_set_pose.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    lib.dvo_rgbd_gauss_newton.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(RgbdParams)]
    lib.dvo_rgbd_get_poses.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    lib.dvo_rgbd_level_dims.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.dvo_rgbd_get_level.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    lib.dvo_rgbd_get_A.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_int)]
    lib.dvo_rgbd_eval.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_int), C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int)]
    _lib = lib
    return lib


class DvoError(RuntimeError):
    pass


def check(rc, what=""):
    if rc != 0:
        msg = load().dvo_last_error().decode(errors="replace")
        raise DvoError(f"{what} failed ({rc}): {msg}")
