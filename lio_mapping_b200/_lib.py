"""ctypes loader of liblio_b200.so (the C-ABI in include/lio_b200.h).

There is no CPU fallback: if the shared library is missing or no CUDA device is usable, every
entry point of this package raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "liblio_b200.so")
_LIB = None


class LioError(RuntimeError):
    pass


STATUS = {0: "LIO_OK", -1: "LIO_ERR_CUDA", -2: "LIO_ERR_INVALID", -3: "LIO_ERR_CAPACITY", -4: "LIO_ERR_NO_DEVICE",
          -5: "LIO_ERR_NUMERIC"}

f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
f64p = np.ctypeslib.ndpointer(np.float64, flags="C_CONTIGUOUS")
i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
u8p = np.ctypeslib.ndpointer(np.uint8, flags="C_CONTIGUOUS")
i8p = np.ctypeslib.ndpointer(np.int8, flags="C_CONTIGUOUS")


class EstConfig(C.Structure):
    """lio_est_config (include/lio_b200.h) == lidar/solver subset of EstimatorConfig (Estimator.h:77-108)."""
    _fields_ = [("window_size", C.c_int), ("opt_window_size", C.c_int), ("min_match_sq_dis", C.c_float),
                ("min_plane_dis", C.c_float), ("surf_filter_size", C.c_float), ("keep_features", C.c_int),
                ("estimate_extrinsic", C.c_int), ("opt_extrinsic", C.c_int), ("imu_factor", C.c_int),
                ("point_distance_factor", C.c_int), ("prior_factor", C.c_int), ("marginalization_factor", C.c_int),
                ("enable_deskew", C.c_int), ("cutoff_deskew", C.c_int), ("acc_n", C.c_double), ("gyr_n", C.c_double),
                ("acc_w", C.c_double), ("gyr_w", C.c_double), ("g_norm", C.c_double), ("max_num_iterations", C.c_int),
                ("odom_max_iterations", C.c_int), ("max_frame_points", C.c_int), ("max_scan_points", C.c_int),
                ("device_solver", C.c_int), ("overlap_marginalization", C.c_int), ("solver_graph", C.c_int)]


class DevCloud(C.Structure):
    """lio_dev_cloud (include/lio_b200.h): a device cloud whose point count lives in device memory, bounded by n_max."""
    _fields_ = [("xyzi", C.c_void_p), ("n_dev", C.c_void_p), ("n_max", C.c_int)]


ALLREDUCE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_int)


class PPConfig(C.Structure):
    """lio_pp_config (include/lio_b200.h) == PointProcessorConfig (PointProcessor.h:104-120)."""
    _fields_ = [("lower_bound", C.c_float), ("upper_bound", C.c_float), ("num_rings", C.c_int),
                ("scan_period", C.c_double), ("num_scan_subregions", C.c_int), ("num_curvature_regions", C.c_int),
                ("surf_curv_th", C.c_float), ("max_corner_sharp", C.c_int), ("max_corner_less_sharp", C.c_int),
                ("max_surf_flat", C.c_int), ("less_flat_filter_size", C.c_float)]


def lib():
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise LioError(f"{LIB_PATH} not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                       "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    L.lio_last_error.restype = C.c_char_p
    L.lio_version.restype = C.c_int
    L.lio_device_count.restype = C.c_int
    vp, ip = C.c_void_p, C.c_int
    L.lio_pp_default_config.argtypes = [C.POINTER(PPConfig)]
    L.lio_pp_create.argtypes = [C.POINTER(PPConfig), ip, ip, vp, C.POINTER(vp)]
    L.lio_pp_destroy.argtypes = [vp]
    L.lio_pp_process_host.argtypes = [vp, f32p, ip]
    L.lio_pp_process_dev.argtypes = [vp, vp, ip]
    L.lio_pp_process_host_ring.argtypes = [vp, f32p, np.ctypeslib.ndpointer(np.uint16, flags="C_CONTIGUOUS"), ip]
    L.lio_pp_cloud_sizes.argtypes = [vp, i32p]
    L.lio_pp_download_cloud.argtypes = [vp, ip, f32p, ip, C.POINTER(ip)]
    L.lio_pp_cloud_dev.argtypes = [vp, ip, C.POINTER(vp)]
    L.lio_pp_download_index.argtypes = [vp, ip, i32p, ip, C.POINTER(ip)]
    L.lio_pp_download_scan_ranges.argtypes = [vp, i32p]
    L.lio_pp_download_mask_labels.argtypes = [vp, u8p, i8p, ip]
    L.lio_pp_start_ori.argtypes = [vp, C.POINTER(C.c_float)]
    L.lio_pp_last_launches.argtypes = [vp]
    L.lio_voxel_grid_host.argtypes = [f32p, ip, C.c_float, f32p, ip, C.POINTER(ip), ip]
    L.lio_calculate_features_host.argtypes = [f32p, ip, f32p, ip, f32p, C.c_float, C.c_float, f32p, f32p, i32p,
                                              C.POINTER(ip), ip]
    L.lio_calculate_line_features_host.argtypes = [f32p, ip, f32p, ip, f32p, C.c_float, f32p, f32p, i32p, C.POINTER(ip), ip]
    L.lio_host_cholesky_solve.argtypes = [ip, f64p, f64p, f64p, f64p]
    L.lio_host_sym_eigen.argtypes = [ip, f64p, f64p, f64p, ip]
    L.lio_host_dogleg_toy.argtypes = [ip, ip, f64p, f64p, f64p, C.c_double, ip, f64p, ip, f64p]
    L.lio_compact_encode.argtypes = [f32p, f32p, ip, f32p, ip, f32p, ip, f32p, ip, C.POINTER(ip)]
    L.lio_compact_sizes.argtypes = [f32p, ip, i32p]
    L.lio_compact_decode.argtypes = [f32p, ip, f32p, f32p, f32p, f32p]
    L.lio_xyzi_to_pcl32.argtypes = [f32p, ip, u8p]
    L.lio_pcl32_to_xyzi.argtypes = [u8p, ip, f32p]
    L.lio_scan_to_map_host.argtypes = [f32p, ip, f32p, ip, f32p, ip, f32p, ip, f32p, C.c_float, C.c_float, ip, C.c_double, C.c_double,
                                       ip, f32p, f32p, i32p, C.POINTER(ip), C.POINTER(ip), ip]
    L.lio_pm_create.argtypes = [ip, C.c_float, C.c_float, C.c_float, C.c_float, ip, ip, vp, C.POINTER(vp)]
    L.lio_pm_destroy.argtypes = [vp]
    L.lio_pm_process_host.argtypes = [vp, f32p, ip, f32p, ip, f32p, f32p, i32p]
    L.lio_pm_map_centre.argtypes = [vp, i32p]
    L.lio_pm_cube_size.argtypes = [vp, ip, ip, C.POINTER(ip)]
    L.lio_pm_cube_download.argtypes = [vp, ip, ip, f32p, ip]
    L.lio_po_create.argtypes = [C.c_float, ip, ip, ip, ip, ip, vp, C.POINTER(vp)]
    L.lio_po_destroy.argtypes = [vp]
    L.lio_po_set_enable_odom.argtypes = [vp, ip]
    L.lio_po_process_host.argtypes = [vp] + [f32p, ip] * 5 + [f32p, f32p, i32p]
    L.lio_po_cloud_size.argtypes = [vp, ip, C.POINTER(ip)]
    L.lio_po_cloud_download.argtypes = [vp, ip, f32p, ip]
    L.lio_po_compact_data.argtypes = [vp, f32p, ip, C.POINTER(ip)]
    L.lio_po_last_launches.argtypes = [vp]
    L.lio_po_matches.argtypes = [vp, ip, i32p, ip]
    L.lio_po_process_dev.argtypes = [vp, C.POINTER(DevCloud), f32p, f32p, i32p]
    L.lio_po_cloud_dev.argtypes = [vp, ip, C.POINTER(vp), C.POINTER(vp)]
    L.lio_pm_process_dev.argtypes = [vp, C.POINTER(DevCloud), C.POINTER(DevCloud), f32p, f32p, i32p]
    i64p = np.ctypeslib.ndpointer(np.int64, flags="C_CONTIGUOUS")
    L.lio_po_last_stats.argtypes = [vp, i64p]
    L.lio_pm_last_stats.argtypes = [vp, i64p]
    L.lio_transform_to_end_host.argtypes = [f32p, ip, f32p, C.c_float, ip]
    L.lio_laser_odom_host.argtypes = [f32p, ip, f32p, ip, f32p, C.c_float, C.c_float, ip, ip, f32p, f32p, i32p,
                                      C.POINTER(ip), C.POINTER(ip), ip]
    L.lio_pp_cloud_count_dev.argtypes = [vp, ip, C.POINTER(vp)]
    L.lio_ppp_evaluate.argtypes = [f64p, f64p, f64p, f64p, f64p, f64p, f64p, f64p, f64p]
    L.lio_ppp_evaluate_batch_host.argtypes = [f32p, f32p, ip, f64p, f64p, f64p, f64p, f64p, ip]
    L.lio_asm_ppp_host.argtypes = [f32p, f32p, ip, f64p, f64p, f64p, ip]
    L.lio_asm_set_fold_chunks.argtypes = [ip]
    L.lio_asm_stream_bench.argtypes = [C.c_longlong, ip, ip, f64p]
    L.lio_dev_cholesky_solve_host.argtypes = [f64p, f64p, ip, f64p, C.POINTER(ip), vp, ip]
    L.lio_pim_create.argtypes = [f64p, f64p, f64p, f64p, f64p, C.POINTER(vp)]
    L.lio_pim_destroy.argtypes = [vp]
    L.lio_pim_push_back.argtypes = [vp, C.c_double, f64p, f64p]
    L.lio_pim_get.argtypes = [vp, f64p, f64p, f64p]
    L.lio_imu_factor_evaluate.argtypes = [vp, f64p, f64p, f64p, f64p, f64p, f64p, f64p, f64p, f64p]
    L.lio_est_default_config.argtypes = [C.POINTER(EstConfig)]
    L.lio_est_create.argtypes = [C.POINTER(EstConfig), ip, vp, C.POINTER(vp)]
    L.lio_est_destroy.argtypes = [vp]
    L.lio_est_set_extrinsic.argtypes = [vp, f32p]
    L.lio_est_get_extrinsic.argtypes = [vp, f32p]
    L.lio_est_init_frame.argtypes = [vp, ip, f64p, f32p, ip, vp]
    L.lio_est_finish_init.argtypes = [vp, f64p, f64p]
    L.lio_est_process_imu.argtypes = [vp, C.c_double, f64p, f64p, C.c_double]
    L.lio_est_process_scan_host.argtypes = [vp, f32p, ip]
    L.lio_est_begin_scan.argtypes = [vp]
    L.lio_est_open_scan_host.argtypes = [vp, f32p, ip]
    L.lio_est_open_scan_dev.argtypes = [vp, vp, vp, ip]
    L.lio_est_get_parameters.argtypes = [vp, f64p, f64p, f64p]
    L.lio_est_assemble.argtypes = [vp, vp, vp, vp, f64p, f64p, C.POINTER(C.c_double), C.POINTER(ip)]
    L.lio_est_solve.argtypes = [vp, f64p, f64p, f64p, ip, f64p]
    L.lio_est_close_scan.argtypes = [vp, vp, vp, vp]
    L.lio_est_exchange_buffer.argtypes = [vp, C.POINTER(vp), C.POINTER(C.c_size_t)]
    L.lio_est_set_peers.argtypes = [vp, ip, C.POINTER(vp)]
    L.lio_est_feature_slab.argtypes = [vp, C.POINTER(vp), C.POINTER(C.c_size_t)]
    L.lio_est_set_feature_peers.argtypes = [vp, ip, C.POINTER(vp)]
    L.lio_ipc_export.argtypes = [vp, u8p]
    L.lio_ipc_open.argtypes = [u8p, C.POINTER(vp)]
    L.lio_ipc_close.argtypes = [vp]
    L.lio_est_process_imu_batch.argtypes = [vp, ip, f64p, f64p, f64p, f64p]
    L.lio_est_process_scan_dev.argtypes = [vp, vp, vp, ip]
    L.lio_est_get_states.argtypes = [vp, f64p]
    L.lio_est_summary.argtypes = [vp, f64p]
    L.lio_est_feature_count.argtypes = [vp, ip, C.POINTER(ip)]
    L.lio_est_get_features.argtypes = [vp, ip, f32p, f32p, i32p, ip]
    L.lio_est_map_size.argtypes = [vp, C.POINTER(ip)]
    L.lio_est_get_map.argtypes = [vp, f32p, ip]
    L.lio_est_frame_size.argtypes = [vp, ip, C.POINTER(ip)]
    L.lio_est_get_frame.argtypes = [vp, ip, f32p, ip]
    L.lio_est_get_local_transform.argtypes = [vp, ip, f32p]
    L.lio_est_prior_dim.argtypes = [vp, C.POINTER(ip)]
    L.lio_est_get_prior.argtypes = [vp, f64p, f64p]
    L.lio_est_last_normal_equations.argtypes = [vp, f64p, f64p, C.POINTER(C.c_double), C.POINTER(ip)]
    L.lio_est_last_launches.argtypes = [vp]
    L.lio_est_last_error.argtypes = [vp]
    L.lio_est_last_error.restype = C.c_char_p
    L.lio_est_solver_trace.argtypes = [vp, np.ctypeslib.ndpointer(np.int64, flags="C_CONTIGUOUS"), ip]
    L.lio_est_frame_owner.argtypes = [ip, ip]
    L.lio_est_kernel_profile.argtypes = [vp, f64p, ip]
    L.lio_est_set_shard.argtypes = [vp, ip, ip, ALLREDUCE_FN, vp]
    _LIB = L
    return L


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = lib().lio_last_error()
        raise LioError(f"{what}: {STATUS.get(rc, rc)} {msg.decode() if msg else ''}")


def require_device():
    n = lib().lio_device_count()
    if n <= 0:
        raise LioError("no CUDA device: lio_mapping_b200 has no CPU fallback")
    return n
