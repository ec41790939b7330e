"""ctypes binding of libbodyslam_b200.so (the C ABI declared in include/bodyslam_b200.h).

There is NO CPU fallback: if the shared object is missing it is built with nvcc; if that fails,
or a compute entry point is called without a CUDA device, a RuntimeError is raised.
"""
import ctypes as C
import os

from . import build as _build

_lib = None

OK, E_ARG, E_CUDA, E_CAPACITY = 0, -1, -2, -3
MAX_BATCH = 256
ZMARCH_BRICK, ZMARCH_LITERAL = 8, 0
GROW_OK, GROW_GROWN, GROW_CAP_UNITS, GROW_CAP_ROW_WORDS = 0, 1, 2, 3

_p = C.c_void_p
_SIGNATURES = {
    "bslam_last_error": (C.c_char_p, []),
    "bslam_version": (C.c_int, []),
    "bslam_device_count": (C.c_int, []),
    "bslam_invert4x4": (C.c_int, [_p, _p, C.c_int]),
    "bslam_scale_u16": (C.c_int, [_p, C.c_int64, C.c_float, _p, _p]),
    "bslam_colorize_workspace_bytes": (C.c_size_t, [C.c_int]),
    "bslam_colorize": (C.c_int, [_p, _p, C.c_int, C.c_int, C.c_int, C.c_float, _p, _p, _p, C.c_double, C.c_double,
                                 C.c_int, C.c_uint16, C.c_uint32, _p, _p, _p, _p, _p]),
    "bslam_colorize_f32_workspace_bytes": (C.c_size_t, [C.c_int]),
    "bslam_colorize_f32": (C.c_int, [_p, C.c_int, C.c_int, C.c_int, _p, _p, C.c_double, C.c_double, C.c_int, C.c_float, C.c_uint32, _p, _p, _p, _p]),
    "bslam_minmax_u8": (C.c_int, [_p, C.c_int, C.c_int, C.c_int, _p, _p, _p, _p, _p]),
    "bslam_median_u16": (C.c_int, [_p, C.c_int, C.c_int64, C.c_int, C.c_uint16, _p, _p, _p]),
    "bslam_depth_from_u16": (C.c_int, [_p, C.c_int64, C.c_float, C.c_double, _p, _p]),
    "bslam_backproject_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "bslam_backproject": (C.c_int, [_p, _p, C.c_int, C.c_int, C.c_int, C.c_int, _p, _p, C.c_int, _p, _p, C.c_int64, _p, _p, _p]),
    "bslam_tsdf_storage_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "bslam_tsdf_create": (C.c_int, [C.POINTER(_p), C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, _p,
                                    C.c_int, C.c_int, _p, _p]),
    "bslam_tsdf_destroy": (C.c_int, [_p]),
    "bslam_tsdf_reset": (C.c_int, [_p, _p]),
    "bslam_tsdf_copy": (C.c_int, [_p, _p, _p]),
    "bslam_tsdf_unit_bounds": (C.c_int, [_p, _p, C.c_int, C.c_float, C.c_double, C.c_int, C.c_int, C.c_int, C.c_int, _p, _p, _p, _p, _p]),
    "bslam_tsdf_grow_box": (C.c_int, [_p, _p, _p, _p, _p, _p]),
    "bslam_tsdf_integrate": (C.c_int, [_p, _p, _p, C.c_int, C.c_int, C.c_int, _p, _p, C.c_int, _p, C.c_int, _p]),
    "bslam_tsdf_integrate_u16": (C.c_int, [_p, _p, C.c_float, C.c_double, _p, _p, C.c_int, C.c_int, C.c_int, _p, _p, _p, _p]),
    "bslam_tsdf_prepare_u16": (C.c_int, [_p, _p, C.c_float, C.c_double, _p, C.c_int, C.c_int, C.c_int, _p, _p, _p]),
    "bslam_tsdf_integrate_prepared": (C.c_int, [_p, _p, _p, _p]),
    "bslam_tsdf_set_z_interleave": (C.c_int, [_p, C.c_int]),
    "bslam_tsdf_layout": (C.c_int, [_p, _p]),
    "bslam_tsdf_set_batch": (C.c_int, [_p, C.c_int]),
    "bslam_tsdf_set_unit_activation": (C.c_int, [_p, C.c_int, C.c_int, C.c_int]),
    "bslam_tsdf_chain_histogram": (C.c_int, [_p, _p, _p]),
    "bslam_tsdf_set_z_split": (C.c_int, [_p, C.c_int]),
    "bslam_tsdf_dry_stats": (C.c_int, [_p, _p, C.c_int, _p]),
    "bslam_selftest": (C.c_int, [C.c_ulonglong, C.c_uint, _p, _p]),
    "bslam_tsdf_profile": (C.c_int, [_p, C.c_int]),
    "bslam_tsdf_profile_read": (C.c_int, [_p, _p, _p]),
    "bslam_tsdf_profile_read_stages": (C.c_int, [_p, _p, _p]),
    "bslam_tsdf_set_clip_check": (C.c_int, [_p, C.c_int, C.c_int]),
    "bslam_tsdf_clip_stats": (C.c_int, [_p, _p, C.c_int, _p]),
    "bslam_tsdf_export": (C.c_int, [_p, _p, _p, _p, _p]),
    "bslam_tsdf_import": (C.c_int, [_p, _p, _p, _p, _p]),
    "bslam_tsdf_export_plane": (C.c_int, [_p, C.c_int, _p, _p]),
    "bslam_tsdf_export_plane_color": (C.c_int, [_p, C.c_int, _p, _p]),
    "bslam_mc_count": (C.c_int, [_p, _p, _p, _p, _p]),
    "bslam_mc_emit": (C.c_int, [_p, _p, _p, _p, _p, _p, _p, C.c_int64, _p, C.c_int64, _p]),
    "bslam_mesh_merge_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "bslam_mesh_merge": (C.c_int, [C.c_int, _p, _p, _p, C.c_int, C.c_int, _p, _p, _p, _p, _p]),
    "bslam_vbg_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "bslam_vbg_integrate": (C.c_int, [_p, _p, _p, C.c_int, C.c_int, C.c_int, _p, _p, _p, C.c_float, C.c_float, _p, _p, _p]),
    "bslam_vbg_stats": (C.c_int, [_p, _p, _p]),
    "bslam_tsdf_raycast": (C.c_int, [_p, C.c_int, C.c_int, C.c_int, _p, _p, C.c_float, C.c_float, C.c_float, C.c_float, _p, _p, _p, _p, _p]),
    "bslam_tsdf_raycast_halo_bytes": (C.c_size_t, [_p, C.c_int]),
    "bslam_tsdf_raycast_segment": (C.c_int, [_p, C.c_int, _p, C.c_int, C.c_int, C.c_int, C.c_int, _p, _p, C.c_float, C.c_float, C.c_float, _p, _p]),
    "bslam_tsdf_raycast_shade": (C.c_int, [_p, C.c_int, _p, _p, _p, C.c_int, C.c_int, C.c_int, _p, _p, C.c_float, _p, _p, _p, _p, _p, _p]),
    "bslam_vbg_raycast_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "bslam_vbg_raycast": (C.c_int, [_p, _p, C.c_int, C.c_int, _p, _p, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float,
                                    _p, _p, _p, _p, _p, _p]),
    "bslam_odom_frame_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "bslam_odom_prepare": (C.c_int, [_p, C.c_int, _p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _p, C.c_float, C.c_float, C.c_float, _p, _p]),
    "bslam_odom_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "bslam_odom_track": (C.c_int, [_p, C.c_int, _p, C.c_int, C.c_int, C.c_int, C.c_int, _p, C.c_int, _p, _p, _p, C.c_float, C.c_float,
                                   C.c_float, _p, _p, _p, _p, _p, _p, _p]),
    "bslam_odom_linearize": (C.c_int, [_p, C.c_int, _p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _p, C.c_int, C.c_float, C.c_float,
                                       C.c_float, _p, _p, _p, _p]),
    "bslam_tsdf_set_extract_flavour": (C.c_int, [_p, C.c_float, C.c_double]),
    "bslam_points_set_incremental": (C.c_int, [_p, C.c_int, C.c_int]),
    "bslam_points_last_stats": (C.c_int, [_p, _p]),
    "bslam_points_count": (C.c_int, [_p, _p, _p]),
    "bslam_points_emit": (C.c_int, [_p, _p, _p, _p, _p, C.c_int64, _p]),
    "bslam_mesh_bvh_bytes": (C.c_size_t, [C.c_int64]),
    "bslam_mesh_build_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int]),
    "bslam_mesh_build": (C.c_int, [_p, C.c_int64, _p, C.c_int64, _p, C.c_int, _p, _p, _p]),
    "bslam_mesh_cast_rays": (C.c_int, [_p, _p, C.c_int64, _p, _p, _p, _p, _p, _p]),
    "bslam_mesh_rays_pinhole": (C.c_int, [C.c_int, C.c_int, C.c_int, _p, _p, _p, _p]),
    "bslam_mesh_cast_pinhole": (C.c_int, [_p, C.c_int, C.c_int, C.c_int, _p, _p, _p, _p, _p, _p, _p, _p]),
    "bslam_mesh_closest_points": (C.c_int, [_p, _p, C.c_int64, _p, _p, _p, _p, _p, _p]),
    "bslam_mesh_distance": (C.c_int, [_p, _p, C.c_int64, _p, _p]),
    "bslam_mesh_occupancy": (C.c_int, [_p, _p, C.c_int64, C.c_int, _p, _p, _p]),
    "bslam_mesh_count_intersections": (C.c_int, [_p, _p, C.c_int64, _p, _p]),
    "bslam_mesh_test_occlusions": (C.c_int, [_p, _p, C.c_int64, C.c_float, C.c_float, _p, _p]),
    "bslam_mesh_occupancy_directions": (C.c_int, [C.c_int, _p]),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)


def lib_path() -> str:
    return _build.LIB


def load():
    """Load (building if needed) the CUDA library; raises RuntimeError when impossible."""
    global _lib
    if _lib is None:
        path = _build.LIB
        if _build.needs_build():
            try:
                _build.build()
            except Exception as e:  # stale but present .so on a box without nvcc is still usable
                if not os.path.exists(path):
                    raise RuntimeError(f"bodyslam_b200: CUDA library missing and cannot be built: {e}") from e
        try:
            L = C.CDLL(path)
        except OSError as e:
            raise RuntimeError(f"bodyslam_b200: cannot load {path}: {e} (there is no CPU fallback)") from e
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc: int) -> None:
    if rc != OK:
        msg = load().bslam_last_error().decode(errors="replace")
        raise RuntimeError(msg or f"libbodyslam_b200 error {rc}")


def require_cuda():
    """torch + a visible CUDA device, or a loud failure (the product has no CPU path)."""
    import torch

    if not torch.cuda.is_available() or load().bslam_device_count() == 0:
        raise RuntimeError("bodyslam_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    return torch


def stream_ptr(device=None):
    import torch

    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def ptr(t):
    """device/host pointer of a torch tensor or numpy array (None -> NULL)."""
    if t is None:
        return None
    if hasattr(t, "data_ptr"):
        return C.c_void_p(t.data_ptr())
    return t.ctypes.data_as(C.c_void_p)
