"""ctypes loader for libicgvins_b200.so (the C ABI declared in include/icgvins_b200.h).

There is no CPU fallback: if the library is missing this raises, and every create() call fails without a B200.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# ICG_LIB_VARIANT=prof loads libicgvins_b200_prof.so: the same sources built with -DICG_BA_PHASE_CLOCKS (`python -m ic_gvins_b200.build --prof`),
# an instrumented build for the profiling scripts only -- never the measured or shipped library
LIB_PATH = os.path.join(_HERE, "libicgvins_b200_prof.so" if os.environ.get("ICG_LIB_VARIANT") == "prof" else "libicgvins_b200.so")

u8p = C.POINTER(C.c_uint8)
f32p = C.POINTER(C.c_float)
f64p = C.POINTER(C.c_double)
i32p = C.POINTER(C.c_int32)
vp = C.c_void_p

_lib = None


class IcgError(RuntimeError):
    pass


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise IcgError(f"{LIB_PATH} not built: run `python -m ic_gvins_b200.build` (there is no CPU fallback)")
        _lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
        _declare(_lib)
        _declare_r2(_lib)
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib().icg_last_error().decode("utf-8", "replace")
        raise IcgError(f"{what} failed with code {rc}: {msg}")


def _declare(L: C.CDLL) -> None:
    L.icg_last_error.restype = C.c_char_p
    L.icg_version.restype = C.c_int
    L.icg_launch_count.restype = C.c_uint64
    L.icg_launch_count_reset.restype = None
    # ---- KLT
    L.icg_klt_create.argtypes = [C.POINTER(vp), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp]
    L.icg_klt_destroy.argtypes = [vp]
    L.icg_klt_destroy.restype = None
    L.icg_klt_calc_optical_flow_pyr_lk.argtypes = [vp, vp, vp, C.c_int, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int,
                                                   C.c_double, C.c_int]
    L.icg_klt_track_fb.argtypes = [vp, vp, vp, C.c_int, vp, vp, vp, vp, C.c_int]
    L.icg_klt_upload.argtypes = [vp, C.c_int, vp, C.c_int]
    L.icg_klt_upload_level0.argtypes = [vp, C.c_int, vp, C.c_int]
    L.icg_klt_upload_batch.argtypes = [vp, C.c_int, C.c_int, vp, C.c_int]
    L.icg_klt_slot_level0.argtypes = [vp, C.c_int, C.POINTER(vp), C.POINTER(C.c_int)]
    L.icg_klt_slot_level.argtypes = [vp, C.c_int, C.c_int, C.POINTER(vp), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.icg_klt_build_pyramids.argtypes = [vp, C.c_int, C.c_int]
    L.icg_klt_track_batch_dev.argtypes = [vp, C.c_int, vp, vp, vp, vp, vp, vp, C.c_int]
    L.icg_klt_sync.argtypes = [vp]
    L.icg_klt_download_level.argtypes = [vp, C.c_int, C.c_int, vp, C.c_int]
    # ---- detection
    L.icg_detect_create.argtypes = [C.POINTER(vp), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp]
    L.icg_detect_destroy.argtypes = [vp]
    L.icg_detect_destroy.restype = None
    L.icg_detect_blocks.argtypes = [vp, vp, vp, C.c_int, C.c_int, vp, vp, C.c_double, C.c_double, C.c_int, vp, vp]
    L.icg_detect_blocks_dev.argtypes = [vp, C.c_int, vp, C.c_int, C.c_size_t, vp, C.c_int, vp, vp, C.c_double, C.c_double, C.c_int, vp, vp]
    L.icg_corner_subpix.argtypes = [vp, vp, C.c_int, vp, C.c_int]
    # ---- camera model (host functions)
    L.icg_camera_undistort_points.argtypes = [vp, vp, C.c_int]
    L.icg_camera_distort_points.argtypes = [vp, vp, C.c_int]
    L.icg_camera_distort_camera_points.argtypes = [vp, vp, vp, C.c_int]
    L.icg_camera_pixel2cam.argtypes = [vp, vp, vp, C.c_int]
    L.icg_camera_world2pixel.argtypes = [vp, vp, vp, vp, vp, C.c_int]
    L.icg_tracking_histogram.argtypes = [vp, C.c_int, C.c_int, C.c_int, vp]
    L.icg_triangulate_points.argtypes = [vp, vp, vp, vp, C.c_int, vp]
    L.icg_find_fundamental_mat_ransac.argtypes = [vp, vp, C.c_int, C.c_double, C.c_double, C.c_int, vp, vp]
    # ---- CLAHE
    L.icg_clahe_create.argtypes = [C.POINTER(vp), C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_int, vp]
    L.icg_clahe_destroy.argtypes = [vp]
    L.icg_clahe_destroy.restype = None
    L.icg_clahe_apply.argtypes = [vp, vp, C.c_int, vp, C.c_int]
    L.icg_clahe_apply_dev.argtypes = [vp, vp, C.c_int, vp, C.c_int]
    L.icg_clahe_sync.argtypes = [vp]
    # ---- BA
    L.icg_imu_preintegrate.argtypes = [vp, vp, vp, vp, vp, C.c_int, vp, vp]
    L.icg_ba_create.argtypes = [C.POINTER(vp), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp]
    L.icg_ba_destroy.argtypes = [vp]
    L.icg_ba_destroy.restype = None
    L.icg_ba_solve.argtypes = [vp, C.c_int, vp, C.c_int, vp]
    L.icg_ba_upload.argtypes = [vp, C.c_int, vp]
    L.icg_ba_run.argtypes = [vp, C.c_int, C.c_int]
    L.icg_ba_download.argtypes = [vp, C.c_int, vp, vp]
    L.icg_ba_sync.argtypes = [vp]
    L.icg_ba_shard_export.argtypes = [vp, C.c_int, C.c_int, vp]
    L.icg_ba_shard_connect.argtypes = [vp, vp]
    L.icg_ba_shard_error.argtypes = [vp]
    L.icg_ba_gvins_optimization.argtypes = [vp, C.c_int, vp, C.c_int, vp, vp]
    L.icg_ba_run_gvins.argtypes = [vp, C.c_int, C.c_int]
    L.icg_ba_gvins_optimization_begin.argtypes = [vp, C.c_int, vp, C.c_int]
    L.icg_ba_gvins_optimization_end.argtypes = [vp, C.c_int, vp, vp, vp]
    L.icg_ba_residual_costs.argtypes = [vp, vp, vp, vp]
    L.icg_ba_reproj_evaluate.argtypes = [vp, vp, vp, vp, vp, vp, vp, C.c_double, vp, vp]
    L.icg_ba_imu_evaluate.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp]
    L.icg_ba_marginalize.argtypes = [vp, C.c_int, vp, vp, vp]
    L.icg_ba_marginalize_resident.argtypes = [vp, C.c_int, vp, vp, vp]
    L.icg_ba_outlier_culling_resident.argtypes = [vp, C.c_int, vp, vp, vp]
    L.icg_ba_gnss_evaluate.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    L.icg_ba_pose_prior_evaluate.argtypes = [vp, vp, vp, vp, vp, vp]
    L.icg_ba_mix_prior_evaluate.argtypes = [vp, vp, vp, vp, vp, vp]
    L.icg_ba_imu_error_evaluate.argtypes = [vp, vp, vp, vp]
    L.icg_ba_marg_factor_evaluate.argtypes = [vp, C.c_int, C.c_int, vp, vp, vp, vp, vp, vp, vp]


def _declare_r2(L: C.CDLL) -> None:
    L.icg_clahe_apply_batch_dev.argtypes = [vp, C.c_int, vp, C.c_int, C.c_size_t, vp, C.c_int, C.c_size_t, vp]
    L.icg_geom_create.argtypes = [C.POINTER(vp), C.c_int, vp]
    L.icg_geom_destroy.argtypes = [vp]
    L.icg_geom_destroy.restype = None
    L.icg_geom_undistort_points.argtypes = [vp, vp, vp, C.c_int]
    L.icg_geom_distort_points.argtypes = [vp, vp, vp, C.c_int]
    L.icg_geom_find_fundamental_mat_ransac.argtypes = [vp, vp, vp, C.c_int, C.c_double, C.c_double, C.c_int, vp, vp]
    L.icg_geom_triangulate_points.argtypes = [vp, vp, vp, vp, vp, C.c_int, vp]
    L.icg_geom_imu_preintegrate_batch.argtypes = [vp, C.c_int, vp, vp, vp, vp, vp, vp, vp, vp]


# every symbol include/icgvins_b200.h declares (checked by tests/test_abi.py against the header text)
EXPORTS = [
    "icg_last_error", "icg_version", "icg_launch_count", "icg_launch_count_reset",
    "icg_klt_create", "icg_klt_destroy", "icg_klt_calc_optical_flow_pyr_lk", "icg_klt_track_fb", "icg_klt_upload",
    "icg_klt_upload_level0", "icg_klt_upload_batch", "icg_klt_slot_level0", "icg_klt_slot_level", "icg_klt_build_pyramids",
    "icg_klt_track_batch_dev", "icg_klt_sync", "icg_klt_download_level",
    "icg_detect_create", "icg_detect_destroy", "icg_detect_blocks", "icg_detect_blocks_dev", "icg_corner_subpix",
    "icg_camera_undistort_points", "icg_camera_distort_points", "icg_camera_distort_camera_points", "icg_camera_pixel2cam", "icg_camera_world2pixel", "icg_tracking_histogram", "icg_find_fundamental_mat_ransac", "icg_triangulate_points",
    "icg_clahe_create", "icg_clahe_destroy", "icg_clahe_apply", "icg_clahe_apply_dev", "icg_clahe_apply_batch_dev", "icg_geom_create", "icg_geom_destroy", "icg_geom_undistort_points", "icg_geom_distort_points", "icg_geom_find_fundamental_mat_ransac", "icg_geom_triangulate_points", "icg_geom_imu_preintegrate_batch", "icg_clahe_sync",
    "icg_imu_preintegrate", "icg_ba_create", "icg_ba_destroy", "icg_ba_solve", "icg_ba_upload", "icg_ba_run", "icg_ba_download",
    "icg_ba_sync", "icg_ba_shard_export", "icg_ba_shard_connect", "icg_ba_shard_error", "icg_ba_gvins_optimization", "icg_ba_run_gvins", "icg_ba_gvins_optimization_begin", "icg_ba_gvins_optimization_end", "icg_ba_residual_costs", "icg_ba_reproj_evaluate", "icg_ba_imu_evaluate", "icg_ba_marginalize", "icg_ba_marginalize_resident", "icg_ba_outlier_culling_resident", "icg_ba_gnss_evaluate", "icg_ba_pose_prior_evaluate", "icg_ba_mix_prior_evaluate", "icg_ba_imu_error_evaluate", "icg_ba_marg_factor_evaluate",
]
