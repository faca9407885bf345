"""ctypes binding of libppp_gpu.so (include/ppp_gpu.h).  Fails loudly when the library is missing:
there is no CPU or PyTorch fallback for the hot path."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libppp_gpu.so")

PPP_OK = 0
PPP_ERR_INVALID = -1
PPP_ERR_CUDA = -2
PPP_ERR_NOMEM = -3
PPP_ERR_CAPACITY = -4
PPP_ERR_UNSUPPORTED = -5

PPP_COV_PCL110 = 0
PPP_COV_SHIFTED = 1
PPP_PAIR_GEN2 = 0
PPP_PAIR_SECT = 1

_vp = C.c_void_p
_f32p = C.POINTER(C.c_float)
_i32p = C.POINTER(C.c_int32)
_i64p = C.POINTER(C.c_int64)
_f64p = C.POINTER(C.c_double)

# name -> (restype, argtypes); every symbol include/ppp_gpu.h declares
SIGNATURES = {
    "ppp_abi_version": (C.c_int, []),
    "ppp_create": (C.c_int, [C.c_int, C.POINTER(_vp)]),
    "ppp_destroy": (None, [_vp]),
    "ppp_last_error": (C.c_char_p, []),
    "ppp_stream": (_vp, [_vp]),
    "ppp_sync": (C.c_int, [_vp]),
    "ppp_host_alloc": (_vp, [C.c_size_t]),
    "ppp_host_free": (None, [_vp]),
    "ppp_launch_count": (C.c_int64, [_vp]),
    "ppp_timer_begin": (C.c_int, [_vp, C.c_int]),
    "ppp_timer_end": (C.c_int, [_vp, C.c_int]),
    "ppp_timer_read": (C.c_int, [_vp, C.c_int, _f64p, _i64p, C.c_int]),
    "ppp_kernel_profile": (C.c_int, [_vp, C.c_int]),
    "ppp_kernel_profile_read": (C.c_int, [_vp, C.c_char_p, C.c_size_t, C.c_int]),
    "ppp_kernel_trace": (C.c_int, [_vp, C.c_int]),
    "ppp_kernel_trace_read": (C.c_int, [_vp, C.c_char_p, C.c_size_t]),
    "ppp_cloud_upload": (C.c_int, [_vp, _vp, C.c_size_t, C.c_size_t, C.POINTER(_vp)]),
    "ppp_dev_cloud_attach": (C.c_int, [_vp, _vp, C.c_size_t, C.c_size_t, C.POINTER(_vp)]),
    "ppp_cloud_free": (C.c_int, [_vp]),
    "ppp_cloud_size": (C.c_int64, [_vp]),
    "ppp_cloud_bbox": (C.c_int, [_vp, _f32p, _f32p]),
    "ppp_cloud_set_cell_hint": (C.c_int, [_vp, C.c_float]),
    "ppp_knn": (C.c_int, [_vp, _vp, C.c_size_t, C.c_size_t, C.c_int, _vp, _vp]),
    "ppp_radius": (C.c_int, [_vp, _vp, C.c_size_t, C.c_size_t, C.c_double, _vp, _vp, _vp, _vp]),
    "ppp_normals_knn": (C.c_int, [_vp, C.c_int, _f32p, C.c_uint, _vp, C.c_size_t, _vp]),
    "ppp_normals_radius": (C.c_int, [_vp, C.c_double, _f32p, C.c_uint, _vp, C.c_size_t]),
    "ppp_slice_bands": (C.c_int, [_vp, _vp, C.c_int, C.c_float, C.c_int, _vp, _vp, C.c_int64]),
    "ppp_slice_contours": (C.c_int, [_vp, _vp, C.c_int, C.c_float, C.c_int, C.c_int, _vp, _vp, _vp, _vp, C.c_int64]),
    "ppp_normals_and_contours": (C.c_int, [_vp, C.c_int, C.c_double, _f32p, C.c_uint, _vp, C.c_size_t, _vp, C.c_int, C.c_float,
                                           C.c_int, C.c_int, _vp, _vp, _vp, _vp, C.c_int64]),
    "ppp_insert_point": (C.c_int, [_vp, _vp, C.c_int64, C.c_float, C.c_int, _vp, _vp, _vp, C.c_int64, _i64p]),
    "ppp_principal_curvatures": (C.c_int, [_vp, _vp, C.c_size_t, _vp, C.c_size_t, C.c_size_t, C.c_int, _vp, _vp]),
    "ppp_sor_mean_distances": (C.c_int, [_vp, C.c_int, C.c_uint, _vp, _i64p]),
    "ppp_coverage_mark": (C.c_int, [_vp, _vp, C.c_size_t, C.c_size_t, C.c_double, _vp]),
    "ppp_coverage_mark_radii": (C.c_int, [_vp, _vp, C.c_size_t, C.c_size_t, _vp, _vp]),
    "ppp_mls_smooth": (C.c_int, [_vp, C.c_double, C.c_int, _vp, C.c_size_t, _vp, _vp, _i64p]),
    "ppp_voxel_grid": (C.c_int, [_vp, _f32p, _vp, C.c_size_t, _vp, _vp, _i64p]),
    "ppp_dev_mls_smooth": (C.c_int, [_vp, C.c_double, C.c_int, _vp, C.c_size_t]),
    "ppp_dev_mls_compact": (C.c_int, [_vp, _vp, C.c_int64, _vp, C.c_size_t, C.c_int64, C.c_int64, _vp, C.c_size_t, _vp, _vp,
                                      C.c_int64, _i64p]),
    "ppp_mls_halo": (C.c_double, [C.c_double, C.c_double]),
    "ppp_dev_index": (C.c_int, [_vp, C.c_int, C.c_double]),
    "ppp_dev_normals_knn": (C.c_int, [_vp, C.c_int, _f32p, C.c_uint, C.c_int64, C.c_int64, _vp, C.c_size_t, _vp, _vp]),
    "ppp_dev_normals_radius": (C.c_int, [_vp, C.c_double, _f32p, C.c_uint, C.c_int64, C.c_int64, _vp, C.c_size_t]),
    "ppp_dev_slice_contours": (C.c_int, [_vp, _vp, C.c_int, C.c_float, C.c_int, C.c_int, C.POINTER(_vp), C.POINTER(_vp),
                                         C.POINTER(_vp), C.POINTER(_vp), _i64p, _i64p]),
    "ppp_dev_set_contour_buffers": (C.c_int, [_vp, _vp, _vp, _vp, C.c_int64]),
    "ppp_dev_set_contour_offsets_buffer": (C.c_int, [_vp, _vp, C.c_int64]),
    "ppp_dev_signal": (C.c_int, [_vp, _vp, C.c_uint32]),
    "ppp_dev_wait": (C.c_int, [_vp, _vp, C.c_uint32]),
    "ppp_dev_set_normal_row_map": (C.c_int, [_vp, _vp]),
    "ppp_peer_buffer_alloc": (C.c_int, [_vp, C.c_size_t, C.POINTER(C.c_void_p), _vp]),
    "ppp_peer_buffer_open": (C.c_int, [_vp, _vp, C.POINTER(C.c_void_p)]),
    "ppp_peer_buffer_close": (C.c_int, [_vp, _vp]),
    "ppp_peer_buffer_free": (C.c_int, [_vp, _vp]),
    "ppp_dev_download": (C.c_int, [_vp, _vp, _vp, C.c_size_t]),
    "ppp_dev_sorted_order": (_vp, [_vp]),
    "ppp_exch_create": (C.c_int, [_vp, C.c_int, C.c_int, _i64p, C.c_int64, C.c_int, C.c_int64, C.c_size_t, C.POINTER(_vp)]),
    "ppp_exch_destroy": (C.c_int, [_vp]),
    "ppp_exch_disconnect": (C.c_int, [_vp]),
    "ppp_exch_ipc_handle": (C.c_int, [_vp, _vp]),
    "ppp_exch_connect_ipc": (C.c_int, [_vp, _vp]),
    "ppp_exch_connect_local": (C.c_int, [_vp, C.POINTER(_vp)]),
    "ppp_exch_phase": (C.c_int, [_vp, C.c_int, _vp, C.c_int64, C.c_size_t, C.c_double]),
    "ppp_exch_finish": (C.c_int, [_vp, _i64p, _i64p, _f64p, _f64p]),
    "ppp_exch_slab": (_vp, [_vp]),
    "ppp_exch_row_map": (_vp, [_vp]),
    "ppp_exch_home_normals": (_vp, [_vp]),
    "ppp_exch_attach": (C.c_int, [_vp, C.c_int, C.POINTER(_vp)]),
    "ppp_exch_finish_attach": (C.c_int, [_vp, C.c_int, _i64p, _i64p, _f64p, _f64p, C.POINTER(_vp)]),
    "ppp_exch_nodes_region": (C.c_int, [_vp, C.c_int, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp)]),
    "ppp_exch_results_signal": (C.c_int, [_vp, C.c_int]),
    "ppp_exch_results_wait": (C.c_int, [_vp, C.c_int]),
    "ppp_exch_check": (C.c_int, [_vp]),
    "ppp_host_register": (C.c_int, [_vp, C.c_size_t, C.POINTER(_vp)]),
    "ppp_dev_upload": (C.c_int, [_vp, _vp, _vp, C.c_size_t]),
    "ppp_dev_download_async": (C.c_int, [_vp, _vp, _vp, C.c_size_t]),
    "ppp_host_unregister": (C.c_int, [_vp]),
}

_lib = None


class PPPError(RuntimeError):
    def __init__(self, status, msg):
        super().__init__("libppp_gpu status %d: %s" % (status, msg))
        self.status = status


def load():
    """Load libppp_gpu.so; raises if it has not been built (python -m polishpathplanning_b200.build)."""
    global _lib
    if _lib is None:
        path = os.environ.get("PPP_GPU_LIB") or LIB_PATH   # PPP_GPU_LIB: the bounds-checked build (tests/test_gpu_bounds.py)
        if not os.path.exists(path):
            raise ImportError(
                "libppp_gpu.so is missing at %s. Build it with `python -m polishpathplanning_b200.build` "
                "(nvcc, sm_100a). The hot path has no CPU / PyTorch fallback." % path)
        L = C.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(status):
    if status != PPP_OK:
        raise PPPError(status, load().ppp_last_error().decode("utf-8", "replace"))
    return status
