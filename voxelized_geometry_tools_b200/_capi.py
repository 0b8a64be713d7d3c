"""ctypes binding of libvgt_b200.so (the C-ABI declared in include/vgt_b200.h).

There is no CPU fallback anywhere in this package: if the shared library is missing, or a
compute call cannot reach a CUDA device, the call raises. Build the library with
``python -m voxelized_geometry_tools_b200.build`` (``__graft_entry__.build()`` does).
"""
from __future__ import annotations

import ctypes
from pathlib import Path

PACKAGE_DIR = Path(__file__).resolve().parent
LIBRARY_PATH = PACKAGE_DIR / "libvgt_b200.so"

OK = 0
ERR_INVALID_ARGUMENT = 1
ERR_DEVICE = 2
ERR_UNSUPPORTED = 3
ERR_NOT_CONTAINED = 4
ERR_OUT_OF_RANGE = 5
SQ_INF = 2 ** 31 - 1

_f32p = ctypes.POINTER(ctypes.c_float)
_f64p = ctypes.POINTER(ctypes.c_double)
_i32p = ctypes.POINTER(ctypes.c_int32)
_u8p = ctypes.POINTER(ctypes.c_uint8)
_i64 = ctypes.c_int64
_int = ctypes.c_int
_dbl = ctypes.c_double
_vp = ctypes.c_void_p


class Cloud(ctypes.Structure):
    """struct vgt_b200_cloud."""
    _fields_ = [("points_xyz", _f64p), ("num_points", _i64), ("x_gc", _dbl * 16),
                ("max_range", _dbl)]


class CloudF32(ctypes.Structure):
    """struct vgt_b200_cloud_f32."""
    _fields_ = [("points_xyz", _f32p), ("num_points", _i64), ("x_gc", _dbl * 16),
                ("max_range", _dbl)]


class SdfView(ctypes.Structure):
    """struct vgt_b200_sdf_view."""
    _fields_ = [("d_sdf", ctypes.c_void_p), ("nx", _i64), ("ny", _i64), ("nz", _i64),
                ("resolution", _dbl), ("origin_transform", _dbl * 16)]


class SdfViewF64(ctypes.Structure):
    """struct vgt_b200_sdf_view_f64 (the same fields; d_sdf points at doubles)."""
    _fields_ = SdfView._fields_


class FilterOptions(ctypes.Structure):
    """struct vgt_b200_filter_options."""
    _fields_ = [("percent_seen_free", _dbl), ("outlier_points_threshold", ctypes.c_int32),
                ("num_cameras_seen_free", ctypes.c_int32)]


class GridFileInfo(ctypes.Structure):
    """struct vgt_b200_grid_file_info."""
    _fields_ = [("nx", _i64), ("ny", _i64), ("nz", _i64), ("voxel_size", _dbl * 3),
                ("origin_transform", _dbl * 16), ("inverse_origin_transform", _dbl * 16),
                ("default_value", _dbl), ("oob_value", _dbl), ("initialized", ctypes.c_int32),
                ("locked", ctypes.c_int32), ("frame_length", _i64), ("payload_bytes", _i64)]


GRID_FILE_SDF_F32 = 0
GRID_FILE_SDF_F64 = 1
GRID_FILE_OCCUPANCY = 2


# name -> (restype, argtypes); must list every symbol include/vgt_b200.h declares
# (tests/test_capi_symbols.py cross-checks this table against the header).
SIGNATURES = {
    "vgt_b200_last_error": (ctypes.c_char_p, []),
    "vgt_b200_version": (ctypes.c_char_p, []),
    "vgt_b200_device_count": (_int, []),
    "vgt_b200_kernel_launch_count": (ctypes.c_uint64, []),
    "vgt_b200_reload_tuning": (None, []),
    "vgt_b200_sdf_f32": (_int, [_vp, _i64, _i64, _i64, _dbl, _int, _int, _int, _vp, _f32p, _f32p]),
    "vgt_b200_sdf_f32_multi": (_int, [_vp, _i64, _i64, _i64, _dbl, _int, _int,
                                      ctypes.POINTER(ctypes.c_int), _int, _vp, _f32p, _f32p]),
    "vgt_b200_sdf_f64": (_int, [_vp, _i64, _i64, _i64, _dbl, _int, _int, _int, _vp, _f64p, _f64p]),
    "vgt_b200_sdf_f64_multi": (_int, [_vp, _i64, _i64, _i64, _dbl, _int, _int,
                                      ctypes.POINTER(ctypes.c_int), _int, _vp, _f64p, _f64p]),
    "vgt_b200_sdf_from_mask_f32": (_int, [_vp, _i64, _i64, _i64, _dbl, _int, _int, _vp, _f32p,
                                          _f32p]),
    "vgt_b200_sdf_from_mask_f64": (_int, [_vp, _i64, _i64, _i64, _dbl, _int, _int, _vp, _f64p,
                                          _f64p]),
    "vgt_b200_sdf_from_cells_f32": (_int, [_vp, _int, _i64, _i64, _i64, _dbl, _int, _int, _vp, _i64,
                                           _int, _vp, _f32p, _f32p]),
    "vgt_b200_sdf_from_cells_f64": (_int, [_vp, _int, _i64, _i64, _i64, _dbl, _int, _int, _vp, _i64,
                                           _int, _vp, _f64p, _f64p]),
    "vgt_b200_sdf_per_object_f32": (_int, [_vp, _int, _i64, _i64, _i64, _dbl, _int, _int, _vp, _i64,
                                           _int, _vp, _vp, _vp]),
    "vgt_b200_sdf_per_object_f64": (_int, [_vp, _int, _i64, _i64, _i64, _dbl, _int, _int, _vp, _i64,
                                           _int, _vp, _vp, _vp]),
    "vgt_b200_sdf_free_and_named_f32": (_int, [_vp, _int, _i64, _i64, _i64, _dbl, _int, _int, _int,
                                               _vp, _f32p, _f32p]),
    "vgt_b200_sdf_free_and_named_f64": (_int, [_vp, _int, _i64, _i64, _i64, _dbl, _int, _int, _int,
                                               _vp, _f64p, _f64p]),
    "vgt_b200_sdf_from_cells_f32_multi": (_int, [_vp, _int, _i64, _i64, _i64, _dbl, _int, _int, _vp, _i64,
                                                 ctypes.POINTER(ctypes.c_int), _int, _vp, _f32p, _f32p]),
    "vgt_b200_sdf_from_cells_f64_multi": (_int, [_vp, _int, _i64, _i64, _i64, _dbl, _int, _int, _vp, _i64,
                                                 ctypes.POINTER(ctypes.c_int), _int, _vp, _f64p, _f64p]),
    "vgt_b200_sdf_per_object_f32_multi": (_int, [_vp, _int, _i64, _i64, _i64, _dbl, _int, _int, _vp, _i64,
                                                 ctypes.POINTER(ctypes.c_int), _int, _vp, _vp, _vp]),
    "vgt_b200_sdf_per_object_f64_multi": (_int, [_vp, _int, _i64, _i64, _i64, _dbl, _int, _int, _vp, _i64,
                                                 ctypes.POINTER(ctypes.c_int), _int, _vp, _vp, _vp]),
    "vgt_b200_sdf_free_and_named_f32_multi": (_int, [_vp, _int, _i64, _i64, _i64, _dbl, _int, _int,
                                                     ctypes.POINTER(ctypes.c_int), _int, _vp, _f32p, _f32p]),
    "vgt_b200_sdf_free_and_named_f64_multi": (_int, [_vp, _int, _i64, _i64, _i64, _dbl, _int, _int,
                                                     ctypes.POINTER(ctypes.c_int), _int, _vp, _f64p, _f64p]),
    "vgt_b200_sdf_from_cells_f32_dev": (_int, [_vp, _int, _i64, _i64, _i64, _dbl, _int, _int, _vp,
                                               _i64, _int, _vp, _vp, _vp]),
    "vgt_b200_sdf_from_cells_f64_dev": (_int, [_vp, _int, _i64, _i64, _i64, _dbl, _int, _int, _vp,
                                               _i64, _int, _vp, _vp, _vp]),
    "vgt_b200_sdf_per_object_f32_dev": (_int, [_vp, _int, _i64, _i64, _i64, _dbl, _int, _int, _vp,
                                               _i64, _int, _vp, _vp, _vp]),
    "vgt_b200_sdf_per_object_f64_dev": (_int, [_vp, _int, _i64, _i64, _i64, _dbl, _int, _int, _vp,
                                               _i64, _int, _vp, _vp, _vp]),
    "vgt_b200_sdf_free_and_named_f32_dev": (_int, [_vp, _int, _i64, _i64, _i64, _dbl, _int, _int,
                                                   _int, _vp, _vp, _vp]),
    "vgt_b200_sdf_free_and_named_f64_dev": (_int, [_vp, _int, _i64, _i64, _i64, _dbl, _int, _int,
                                                   _int, _vp, _vp, _vp]),
    "vgt_b200_edt_transform_inplace_f64": (_int, [_vp, _i64, _i64, _i64, _int]),
    "vgt_b200_edt_sq_i32": (_int, [_vp, _i64, _i64, _i64, _int, _int, _vp, _vp]),
    "vgt_b200_sdf_f32_dev": (_int, [_vp, _i64, _i64, _i64, _dbl, _int, _int, _int, _vp, _vp, _vp]),
    "vgt_b200_sdf_f32_dev_profile": (_int, [_vp, _i64, _i64, _i64, _dbl, _int, _int, _int, _vp, _vp,
                                            _vp, _f32p]),
    "vgt_b200_sdf_f64_dev": (_int, [_vp, _i64, _i64, _i64, _dbl, _int, _int, _int, _vp, _vp, _vp]),
    "vgt_b200_sdf_from_mask_f32_dev": (_int, [_vp, _i64, _i64, _i64, _dbl, _int, _int, _vp, _vp,
                                              _vp]),
    "vgt_b200_edt_local_passes_dev": (_int, [_vp, _i64, _i64, _i64, _int, _int, _int, _vp, _vp]),
    "vgt_b200_edt_local_passes_scatter_dev": (_int, [_vp, _i64, _i64, _i64, _int, _int, _int, _i64,
                                                     _i64, ctypes.POINTER(ctypes.c_uint64), _i64,
                                                     _int, _vp]),
    "vgt_b200_edt_final_pass_f32_dev": (_int, [_vp, _i64, _i64, _i64, _i64, _i64, _dbl, _int, _int,
                                               _vp, _vp, _vp]),
    "vgt_b200_sdf_estimate_distance_dev": (_int, [ctypes.POINTER(SdfView), _vp, _i64, _int, _vp,
                                                  _vp, _vp]),
    "vgt_b200_sdf_coarse_gradient_dev": (_int, [ctypes.POINTER(SdfView), _vp, _i64, _int, _int,
                                                _vp, _vp, _vp]),
    "vgt_b200_sdf_fine_gradient_dev": (_int, [ctypes.POINTER(SdfView), _vp, _i64, _dbl, _int, _vp,
                                              _vp, _vp]),
    "vgt_b200_sdf_local_extrema_map_dev": (_int, [ctypes.POINTER(SdfView), _int, _vp, _vp]),
    "vgt_b200_sdf_project_out_of_collision_dev": (_int, [ctypes.POINTER(SdfView), _vp, _i64, _dbl,
                                                         _dbl, _i64, _int, _vp, _vp, _vp]),
    "vgt_b200_sdf_estimate_distance_f64_dev": (_int, [ctypes.POINTER(SdfViewF64), _vp, _i64, _int,
                                                      _vp, _vp, _vp]),
    "vgt_b200_sdf_coarse_gradient_f64_dev": (_int, [ctypes.POINTER(SdfViewF64), _vp, _i64, _int,
                                                    _int, _vp, _vp, _vp]),
    "vgt_b200_sdf_fine_gradient_f64_dev": (_int, [ctypes.POINTER(SdfViewF64), _vp, _i64, _dbl, _int,
                                                  _vp, _vp, _vp]),
    "vgt_b200_sdf_local_extrema_map_f64_dev": (_int, [ctypes.POINTER(SdfViewF64), _int, _vp, _vp]),
    "vgt_b200_sdf_project_out_of_collision_f64_dev": (_int, [ctypes.POINTER(SdfViewF64), _vp, _i64,
                                                             _dbl, _dbl, _i64, _int, _vp, _vp,
                                                             _vp]),
    "vgt_b200_voxelize_f64": (_int, [_vp, _i64, _i64, _i64, _dbl, ctypes.POINTER(Cloud),
                                     ctypes.c_int32, ctypes.POINTER(FilterOptions), _int, _vp,
                                     _vp, _f64p]),
    "vgt_b200_voxelize_f32": (_int, [_vp, _i64, _i64, _i64, _dbl, ctypes.POINTER(CloudF32),
                                     ctypes.c_int32, ctypes.POINTER(FilterOptions), _int, _vp,
                                     _vp, _f64p]),
    "vgt_b200_raycast_f32_dev": (_int, [_vp, _i64, _f64p, _dbl, _i64, _i64, _i64, _dbl, _int, _vp,
                                        _vp]),
    "vgt_b200_raycast_f64_dev": (_int, [_vp, _i64, _f64p, _dbl, _i64, _i64, _i64, _dbl, _int, _vp,
                                        _vp]),
    "vgt_b200_filter_dev": (_int, [_vp, ctypes.c_int32, _i64, ctypes.POINTER(FilterOptions), _int,
                                   _vp, _vp]),
    "vgt_b200_rasterize_mesh_f64": (_int, [_vp, _i64, _vp, _i64, _vp, _int, _i64, _i64, _i64, _dbl,
                                           _f64p, _f64p, _int, _int]),
    "vgt_b200_rasterize_mesh_dev": (_int, [_vp, _i64, _vp, _i64, _vp, _int, _i64, _i64, _i64, _dbl,
                                           _f64p, _f64p, _int, _int, _vp, _vp]),
    "vgt_b200_rasterize_status": (_int, [_int]),
    "vgt_b200_connected_components": (_int, [_vp, _int, _i64, _i64, _i64, _int, _vp]),
    "vgt_b200_connected_components_dev": (_int, [_vp, _int, _i64, _i64, _i64, _int, _vp, _vp]),
    "vgt_b200_connected_components_multi": (_int, [_vp, _int, _i64, _i64, _i64, _vp, _int, _vp]),
    "vgt_b200_components_slab_scan_bytes": (_int, [_i64, _i64, _i64, _int,
                                                   ctypes.POINTER(ctypes.c_size_t)]),
    "vgt_b200_components_slab_local": (_int, [_vp, _int, _i64, _i64, _i64, _int, _vp, _vp, _vp,
                                              _vp, ctypes.c_size_t, _vp, _vp]),
    "vgt_b200_components_slab_face_edges": (_int, [_vp, _vp, _i64, _vp, _int, _i64, _i64, _i64,
                                                   _i64, _int, _vp, _vp, _vp, _vp]),
    "vgt_b200_components_resolve": (_int, [_vp, _i64, _i64, _i64, _i64, _int, _vp, _vp, _vp,
                                           _vp]),
    "vgt_b200_components_slab_count": (_int, [_i64, _i64, _i64, _i64, _i64, _int, _vp, _vp, _vp,
                                              _vp, _i64, _i64, _i64, _vp, _vp, _vp,
                                              ctypes.c_size_t, _vp]),
    "vgt_b200_components_slab_publish": (_int, [_i64, _i64, _i64, _i64, _i64, _i64, _int, _vp,
                                                _vp, _vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp,
                                                _vp]),
    "vgt_b200_components_slab_write": (_int, [_vp, _int, _i64, _i64, _i64, _i64, _i64, _int, _vp,
                                              _vp, _vp, _vp, _vp, _i64, _i64, _i64, _vp, _vp,
                                              _vp]),
    "vgt_b200_grid_file_save": (_int, [ctypes.c_char_p, _int, _int, _vp,
                                       ctypes.POINTER(GridFileInfo), ctypes.c_char_p]),
    "vgt_b200_grid_file_save_dev": (_int, [ctypes.c_char_p, _int, _int, _vp,
                                           ctypes.POINTER(GridFileInfo), ctypes.c_char_p, _int,
                                           _vp]),
    "vgt_b200_grid_file_probe": (_int, [ctypes.c_char_p, _int, ctypes.POINTER(GridFileInfo),
                                        ctypes.c_char_p, _i64]),
    "vgt_b200_grid_file_load": (_int, [ctypes.c_char_p, _int, _vp, _i64,
                                       ctypes.POINTER(GridFileInfo), ctypes.c_char_p, _i64]),
}

_library = None


class BackendUnavailable(RuntimeError):
    """The CUDA shared library is missing or no sm_100 device is usable."""


def library() -> ctypes.CDLL:
    global _library
    if _library is None:
        if not LIBRARY_PATH.exists():
            raise BackendUnavailable(
                f"{LIBRARY_PATH} is missing: build it with "
                "`python -m voxelized_geometry_tools_b200.build` (there is no CPU fallback)")
        handle = ctypes.CDLL(str(LIBRARY_PATH))
        for name, (restype, argtypes) in SIGNATURES.items():
            function = getattr(handle, name)  # AttributeError = stale library: fail loudly
            function.restype = restype
            function.argtypes = argtypes
        _library = handle
    return _library


def last_error() -> str:
    return library().vgt_b200_last_error().decode("utf-8", "replace")


def check(code: int) -> None:
    """Maps C-ABI codes to the exception types the reference throws for the same condition."""
    if code == OK:
        return
    message = last_error()
    if code == ERR_INVALID_ARGUMENT:
        raise ValueError(message)        # std::invalid_argument
    if code == ERR_UNSUPPORTED:
        raise NotImplementedError(message)
    if code == ERR_OUT_OF_RANGE:
        raise IndexError(message)        # std::out_of_range
    raise RuntimeError(message)          # std::runtime_error


def device_count() -> int:
    return int(library().vgt_b200_device_count())


def require_device(device: int = 0) -> None:
    count = device_count()
    if device < 0 or device >= count:
        raise BackendUnavailable(
            f"CUDA device {device} is not available ({count} usable sm_100 device(s) found); "
            "this backend has no CPU fallback")
