"""ctypes binding of libcupoch_b200.so (the C ABI in include/cupoch_b200.h).

The product path has NO fallback: if the CUDA library is missing or no GPU is
visible every compute entry point raises.  (The CPU oracle under oracle/ is
test infrastructure and is never imported from here.)
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libcupoch_b200.so")

OK = 0
EST_UNSPECIFIED, EST_POINT_TO_POINT, EST_POINT_TO_PLANE, EST_SYMMETRIC, EST_COLORED_ICP, EST_GENERALIZED_ICP = range(6)


class CphbError(RuntimeError):
    pass


class Cloud(C.Structure):
    _fields_ = [("points", C.c_void_p), ("normals", C.c_void_p), ("colors", C.c_void_p),
                ("covariances", C.c_void_p), ("color_gradient", C.c_void_p), ("n", C.c_size_t),
                ("cov_col_major", C.c_int)]


class IcpParams(C.Structure):
    _fields_ = [("estimation", C.c_int), ("max_correspondence_distance", C.c_float),
                ("relative_fitness", C.c_float), ("relative_rmse", C.c_float), ("max_iteration", C.c_int),
                ("det_thresh", C.c_float), ("lambda_geometric", C.c_float), ("flags", C.c_int),
                ("shard_rank", C.c_int), ("shard_world", C.c_int)]


class IcpResult(C.Structure):
    _fields_ = [("transformation", C.c_float * 16), ("fitness", C.c_float), ("inlier_rmse", C.c_float),
                ("n_correspondences", C.c_int64), ("n_local_correspondences", C.c_int64), ("iterations", C.c_int),
                ("converged", C.c_int),
                ("loop_ms", C.c_float), ("loop_launches", C.c_int)]


class OccGridParams(C.Structure):
    _fields_ = [("clamping_thres_min", C.c_float), ("clamping_thres_max", C.c_float), ("prob_hit_log", C.c_float),
                ("prob_miss_log", C.c_float), ("occ_prob_thres_log", C.c_float)]


class FgrOption(C.Structure):
    _fields_ = [("division_factor", C.c_float), ("use_absolute_scale", C.c_int), ("decrease_mu", C.c_int),
                ("maximum_correspondence_distance", C.c_float), ("iteration_number", C.c_int),
                ("tuple_scale", C.c_float), ("maximum_tuple_count", C.c_int)]


_P = C.c_void_p
_F3 = C.POINTER(C.c_float)
_I3 = C.POINTER(C.c_int32)
_SIGNATURES = {
    "cphb_occgrid_default_params": (None, [C.POINTER(OccGridParams)]),
    "cphb_occgrid_create": (C.c_int, [C.c_float, C.c_int, _F3, _P, C.POINTER(_P)]),
    "cphb_occgrid_destroy": (None, [_P]),
    "cphb_occgrid_clear": (C.c_int, [_P, _P]),
    "cphb_occgrid_set_params": (C.c_int, [_P, C.POINTER(OccGridParams)]),
    "cphb_occgrid_set_geometry": (C.c_int, [_P, C.c_float, _F3]),
    "cphb_occgrid_data": (_P, [_P]),
    "cphb_occgrid_resolution": (C.c_int, [_P]),
    "cphb_occgrid_insert": (C.c_int, [_P, _P, C.c_size_t, _F3, C.c_float, _P]),
    "cphb_occgrid_add_voxels": (C.c_int, [_P, _P, C.c_size_t, C.c_int, _P]),
    "cphb_occgrid_add_voxel": (C.c_int, [_P, _I3, C.c_int, _P]),
    "cphb_occgrid_set_free_area": (C.c_int, [_P, _F3, _F3, _P]),
    "cphb_occgrid_bounds": (C.c_int, [_P, _I3, _I3, _P]),
    "cphb_occgrid_extract": (C.c_int, [_P, C.c_int, _P, _P, C.c_size_t, C.POINTER(C.c_size_t), _P]),
    "cphb_occgrid_get_voxel": (C.c_int, [_P, _F3, C.POINTER(C.c_int), C.POINTER(C.c_float), _I3, _P]),
    # name: (restype, argtypes)
    "cphb_version": (C.c_int, []),
    "cphb_last_error": (C.c_char_p, []),
    "cphb_launch_count": (C.c_uint64, []),
    "cphb_device_count": (C.c_int, []),
    "cphb_set_device": (C.c_int, [C.c_int]),
    "cphb_index_create": (C.c_int, [_P, C.c_size_t, _P, C.POINTER(_P)]),
    "cphb_index_destroy": (None, [_P]),
    "cphb_index_size": (C.c_size_t, [_P]),
    "cphb_search_radius": (C.c_int, [_P, _P, C.c_size_t, C.c_float, C.c_int, _P, _P, C.POINTER(C.c_int64), _P]),
    "cphb_search_knn": (C.c_int, [_P, _P, C.c_size_t, C.c_int, _P, _P, C.POINTER(C.c_int64), _P]),
    "cphb_search_hybrid": (C.c_int, [_P, _P, C.c_size_t, C.c_float, C.c_int, _P, _P, C.POINTER(C.c_int64), _P]),
    "cphb_transform": (C.c_int, [_P, _P, _P, C.c_int, C.c_size_t, C.POINTER(C.c_float), _P]),
    "cphb_min_max_bound": (C.c_int, [_P, C.c_size_t, C.POINTER(C.c_float), C.POINTER(C.c_float), _P]),
    "cphb_voxel_down_sample": (C.c_int, [_P, _P, _P, C.c_size_t, C.c_float, _P, _P, _P, C.POINTER(C.c_size_t), _P]),
    "cphb_voxel_down_sample_origin": (C.c_int, [_P, _P, _P, C.c_size_t, C.c_float, C.POINTER(C.c_float), _P, _P, _P,
                                                C.POINTER(C.c_size_t), _P]),
    "cphb_voxel_indices": (C.c_int, [_P, C.c_size_t, C.c_float, C.POINTER(C.c_float), _P, _P]),
    "cphb_estimate_normals": (C.c_int, [_P, C.c_size_t, C.c_int, C.c_float, C.c_int, _P, _P]),
    "cphb_estimate_normals_range": (C.c_int, [_P, C.c_size_t, C.c_int, C.c_float, C.c_int, C.c_size_t, C.c_size_t, _P, _P]),
    "cphb_remove_radius_outliers": (C.c_int, [_P, C.c_size_t, C.c_int, C.c_float, _P, C.POINTER(C.c_size_t), _P]),
    "cphb_remove_statistical_outliers": (C.c_int, [_P, C.c_size_t, C.c_int, C.c_float, _P, C.POINTER(C.c_size_t),
                                                   C.POINTER(C.c_float), _P]),
    "cphb_voxel_grid_from_point_cloud": (C.c_int, [_P, _P, C.c_size_t, C.c_float, C.POINTER(C.c_float), C.POINTER(C.c_float),
                                                   _P, _P, C.POINTER(C.c_size_t), _P]),
    "cphb_gaussian_filter": (C.c_int, [_P, _P, _P, C.c_size_t, C.c_float, C.c_float, C.c_int, _P, _P, _P,
                                       C.POINTER(C.c_size_t), _P]),
    "cphb_select_by_index": (C.c_int, [_P, _P, _P, C.c_size_t, _P, C.c_size_t, _P, _P, _P, _P]),
    "cphb_covariances_from_normals": (C.c_int, [_P, C.c_size_t, C.c_float, _P, C.c_int, _P]),
    "cphb_color_gradient": (C.c_int, [_P, _P, _P, C.c_size_t, C.c_float, C.c_int, _P, _P]),
    "cphb_icp_create": (C.c_int, [C.POINTER(Cloud), C.POINTER(Cloud), C.POINTER(IcpParams), _P, C.POINTER(_P)]),
    "cphb_icp_destroy": (None, [_P]),
    "cphb_icp_run": (C.c_int, [_P, C.POINTER(C.c_float), _P, C.POINTER(IcpResult), _P, _P]),
    "cphb_icp_step": (C.c_int, [_P, C.POINTER(C.c_float), C.POINTER(C.c_double), _P, _P]),
    "cphb_registration_icp": (C.c_int, [C.POINTER(Cloud), C.POINTER(Cloud), C.POINTER(C.c_float),
                                        C.POINTER(IcpParams), _P, C.POINTER(IcpResult), _P, _P]),
    "cphb_registration_icp_host": (C.c_int, [C.POINTER(Cloud), C.POINTER(Cloud), C.POINTER(C.c_float),
                                             C.POINTER(IcpParams), _P, C.POINTER(IcpResult), _P, _P]),
    "cphb_evaluate_registration": (C.c_int, [C.POINTER(Cloud), C.POINTER(Cloud), C.c_float, C.POINTER(C.c_float),
                                             C.POINTER(IcpResult), _P, _P]),
    "cphb_compute_transformation": (C.c_int, [C.c_int, C.POINTER(Cloud), C.POINTER(Cloud), _P, C.c_size_t,
                                              C.POINTER(IcpParams), C.POINTER(C.c_float), _P]),
    "cphb_compute_rmse": (C.c_int, [C.c_int, C.POINTER(Cloud), C.POINTER(Cloud), _P, C.c_size_t, C.POINTER(IcpParams),
                                    C.POINTER(C.c_float), _P]),
    "cphb_kabsch": (C.c_int, [_P, C.c_size_t, _P, _P, C.c_size_t, C.POINTER(C.c_float), _P]),
    "cphb_kabsch_weighted": (C.c_int, [_P, _P, _P, C.c_size_t, C.POINTER(C.c_float), _P]),
    "cphb_compute_jtj_jtr": (C.c_int, [_P, _P, C.c_size_t, C.c_int, C.POINTER(C.c_double), _P]),
    "cphb_compute_weighted_jtj_jtr": (C.c_int, [_P, _P, C.c_size_t, C.c_int, C.c_float, C.c_float, C.POINTER(C.c_double),
                                                 C.POINTER(C.c_float), _P]),
    "cphb_compute_fpfh_feature": (C.c_int, [_P, _P, C.c_size_t, C.c_int, C.c_float, C.c_int, _P, _P]),
    "cphb_fgr_default_option": (None, [C.POINTER(FgrOption)]),
    "cphb_feature_nn": (C.c_int, [_P, C.c_size_t, _P, C.c_size_t, C.c_int, _P, _P, _P, _P, _P]),
    "cphb_fgr_advanced_matching": (C.c_int, [_P, C.c_size_t, _P, C.c_size_t, _P, C.c_size_t, _P, C.c_size_t, C.c_int,
                                             C.POINTER(FgrOption), _P, C.POINTER(C.c_int64), _P]),
    "cphb_fast_global_registration": (C.c_int, [C.POINTER(Cloud), C.POINTER(Cloud), _P, C.c_size_t, _P, C.c_size_t,
                                                C.c_int, C.POINTER(FgrOption), C.POINTER(IcpResult), _P, _P, _P]),
    "cphb_cluster_dbscan": (C.c_int, [_P, C.c_size_t, C.c_float, C.c_int, C.c_int, _P, C.POINTER(C.c_int), _P]),
    "cphb_reserve_pool": (C.c_int, [C.c_size_t]),
    "cphb_malloc": (_P, [C.c_size_t]),
    "cphb_free": (None, [_P]),
    "cphb_malloc_host": (_P, [C.c_size_t]),
    "cphb_free_host": (None, [_P]),
    "cphb_memcpy_h2d": (C.c_int, [_P, _P, C.c_size_t, _P]),
    "cphb_memcpy_d2h": (C.c_int, [_P, _P, C.c_size_t, _P]),
    "cphb_memset": (C.c_int, [_P, C.c_int, C.c_size_t, _P]),
    "cphb_stream_synchronize": (C.c_int, [_P]),
    "cphb_memcpy_d2d": (C.c_int, [_P, _P, C.c_size_t, _P]),
    "cphb_event_create": (_P, []),
    "cphb_event_destroy": (None, [_P]),
    "cphb_event_record": (C.c_int, [_P, _P]),
    "cphb_event_elapsed_ms": (C.c_int, [_P, _P, C.POINTER(C.c_float)]),
    "cphb_nccl_unique_id": (C.c_int, [C.c_char_p]),
    "cphb_comm_nccl_create": (C.c_int, [C.c_char_p, C.c_int, C.c_int, C.POINTER(_P)]),
    "cphb_comm_p2p_create": (C.c_int, [C.c_int, C.c_int, C.c_char_p, C.POINTER(_P)]),
    "cphb_comm_p2p_connect": (C.c_int, [_P, C.c_char_p]),
    "cphb_comm_destroy": (C.c_int, [_P]),
    "cphb_comm_allreduce_f64": (C.c_int, [_P, _P, C.c_int, _P]),
}
EXPORTED_SYMBOLS = sorted(_SIGNATURES)

_lib = None


def lib():
    """Load the shared library (no GPU needed to load it)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise CphbError("libcupoch_b200.so not built: run `python -m cupoch_b200.build` "
                            "(there is no CPU fallback for the product path)")
        L = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
        for name, (res, args) in _SIGNATURES.items():
            f = getattr(L, name)
            f.restype = res
            f.argtypes = args
        _lib = L
    return _lib


def check(rc):
    if rc != OK:
        raise CphbError("cupoch_b200 error %d: %s" % (rc, lib().cphb_last_error().decode(errors="replace")))


def require_gpu():
    if lib().cphb_device_count() <= 0:
        raise CphbError("no CUDA device visible: cupoch_b200 has no CPU fallback")
