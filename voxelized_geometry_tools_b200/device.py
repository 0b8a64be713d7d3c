"""Device-resident entry points: torch CUDA tensors in, torch CUDA tensors out.

torch is only the owner of device memory and streams here; every kernel is launched by
libvgt_b200.so through the ``*_dev`` C-ABI functions on torch's current stream.
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _capi
from .pointcloud_voxelization import PointCloudVoxelizationFilterOptions


def _stream_handle(device: torch.device) -> int:
    return int(torch.cuda.current_stream(device).cuda_stream)


def _require_cuda(tensor: torch.Tensor, dtype: torch.dtype, what: str) -> None:
    if not tensor.is_cuda:
        raise _capi.BackendUnavailable(f"{what} must live on a CUDA device (no CPU fallback)")
    if tensor.dtype != dtype or not tensor.is_contiguous():
        raise ValueError(f"{what} must be a contiguous {dtype} tensor")


def signed_distance_field(occupancy: torch.Tensor, resolution: float,
                          unknown_is_filled: bool = True, add_virtual_border: bool = False,
                          out: torch.Tensor | None = None, min_max: torch.Tensor | None = None,
                          compute_min_max: bool = True):
    """ExtractSignedDistanceField<float> on a device-resident occupancy grid [nx, ny, nz].

    Returns (sdf float32 [nx, ny, nz], min_max float32 [2] or None). Asynchronous."""
    _require_cuda(occupancy, torch.float32, "occupancy")
    if occupancy.dim() != 3:
        raise ValueError("occupancy must be indexed [x, y, z]")
    device = occupancy.device
    if out is None:
        out = torch.empty_like(occupancy)
    _require_cuda(out, torch.float32, "out")
    if compute_min_max and min_max is None:
        min_max = torch.empty(2, dtype=torch.float32, device=device)
    nx, ny, nz = occupancy.shape
    code = _capi.library().vgt_b200_sdf_f32_dev(
        occupancy.data_ptr(), nx, ny, nz, float(resolution), int(unknown_is_filled),
        int(add_virtual_border), device.index or 0, out.data_ptr(),
        min_max.data_ptr() if compute_min_max else None, _stream_handle(device))
    _capi.check(code)
    return out, (min_max if compute_min_max else None)


def signed_distance_field_profile(occupancy: torch.Tensor, resolution: float,
                                  out: torch.Tensor, min_max: torch.Tensor | None = None,
                                  kernels: bool = False):
    """Same kernels as signed_distance_field with CUDA events between them; synchronises.
    Returns [ms z-scan, ms y-pass, ms x-pass + finalize]; kernels=True appends the durations of
    the y pass's and the x pass's main window-kernel launch alone (a pass also holds the pilot
    probe, the decision and the stack kernel over the hand-over list)."""
    _require_cuda(occupancy, torch.float32, "occupancy")
    _require_cuda(out, torch.float32, "out")
    device = occupancy.device
    nx, ny, nz = occupancy.shape
    pass_ms = (ctypes.c_float * 5)()
    code = _capi.library().vgt_b200_sdf_f32_dev_profile(
        occupancy.data_ptr(), nx, ny, nz, float(resolution), 1, 0, device.index or 0,
        out.data_ptr(), None if min_max is None else min_max.data_ptr(), _stream_handle(device),
        pass_ms)
    _capi.check(code)
    return [float(v) for v in pass_ms][:5 if kernels else 3]


def signed_distance_field_f64(occupancy: torch.Tensor, resolution: float,
                              unknown_is_filled: bool = True, add_virtual_border: bool = False):
    _require_cuda(occupancy, torch.float32, "occupancy")
    device = occupancy.device
    out = torch.empty(occupancy.shape, dtype=torch.float64, device=device)
    min_max = torch.empty(2, dtype=torch.float64, device=device)
    nx, ny, nz = occupancy.shape
    code = _capi.library().vgt_b200_sdf_f64_dev(
        occupancy.data_ptr(), nx, ny, nz, float(resolution), int(unknown_is_filled),
        int(add_virtual_border), device.index or 0, out.data_ptr(), min_max.data_ptr(),
        _stream_handle(device))
    _capi.check(code)
    return out, min_max


def signed_distance_field_from_mask(mask: torch.Tensor, resolution: float,
                                    add_virtual_border: bool = False):
    _require_cuda(mask, torch.uint8, "mask")
    device = mask.device
    out = torch.empty(mask.shape, dtype=torch.float32, device=device)
    min_max = torch.empty(2, dtype=torch.float32, device=device)
    nx, ny, nz = mask.shape
    code = _capi.library().vgt_b200_sdf_from_mask_f32_dev(
        mask.data_ptr(), nx, ny, nz, float(resolution), int(add_virtual_border),
        device.index or 0, out.data_ptr(), min_max.data_ptr(), _stream_handle(device))
    _capi.check(code)
    return out, min_max


def edt_local_passes(occupancy_slab: torch.Tensor, unknown_is_filled: bool = True,
                     out: torch.Tensor | None = None, send_parts: int = 0) -> torch.Tensor:
    """z and y passes on an x-slab [nx_local, ny, nz] -> sign-fused int32 words.

    send_parts = G > 1 writes the result in send layout (G blocks [nx_local, rows_h, nz] back to
    back, block h = the part of every y-line that rank h owns); raises NotImplementedError when the
    library cannot (ny > 1024), in which case the caller packs."""
    _require_cuda(occupancy_slab, torch.float32, "occupancy_slab")
    device = occupancy_slab.device
    if out is None:
        out = torch.empty(occupancy_slab.shape, dtype=torch.int32, device=device)
    _require_cuda(out, torch.int32, "out")
    nx, ny, nz = occupancy_slab.shape
    code = _capi.library().vgt_b200_edt_local_passes_dev(
        occupancy_slab.data_ptr(), nx, ny, nz, int(unknown_is_filled), int(send_parts),
        device.index or 0, out.data_ptr(), _stream_handle(device))
    if code == _capi.ERR_UNSUPPORTED:
        raise NotImplementedError(_capi.last_error())
    _capi.check(code)
    return out


def edt_local_passes_scatter(occupancy_slab: torch.Tensor, rank: int, x_offset: int,
                             nx_total: int, peer_buffer_ptrs, receive_capacity_words: int,
                             unknown_is_filled: bool = True) -> None:
    """z and y passes on an x-slab with the exchange fused in: the y pass stores each rank's
    part of every line straight into that rank's receive buffer (peer-mapped device pointers,
    entry h = rank h's buffer laid out [nx_total, rows_h, nz], every buffer
    ``receive_capacity_words`` int32 words long; the library refuses a layout that does not fit)."""
    _require_cuda(occupancy_slab, torch.float32, "occupancy_slab")
    device = occupancy_slab.device
    nx, ny, nz = occupancy_slab.shape
    pointers = (ctypes.c_uint64 * len(peer_buffer_ptrs))(*[int(p) for p in peer_buffer_ptrs])
    code = _capi.library().vgt_b200_edt_local_passes_scatter_dev(
        occupancy_slab.data_ptr(), nx, ny, nz, int(unknown_is_filled), len(peer_buffer_ptrs),
        int(rank), int(x_offset), int(nx_total), pointers, int(receive_capacity_words),
        device.index or 0, _stream_handle(device))
    if code == _capi.ERR_UNSUPPORTED:
        raise NotImplementedError(_capi.last_error())
    _capi.check(code)


def edt_final_pass(packed: torch.Tensor, y_offset: int, ny_total: int, resolution: float,
                   add_virtual_border: bool = False, compute_min_max: bool = True):
    """x pass + finalize on a y-slab [nx, ny_local, nz] of sign-fused words. ``packed`` is
    destroyed (the envelope stacks are built in place in it); the SDF is a new tensor."""
    _require_cuda(packed, torch.int32, "packed")
    device = packed.device
    nx, ny_local, nz = packed.shape
    out = torch.empty(packed.shape, dtype=torch.float32, device=device)
    min_max = torch.empty(2, dtype=torch.float32, device=device) if compute_min_max else None
    code = _capi.library().vgt_b200_edt_final_pass_f32_dev(
        packed.data_ptr(), nx, ny_local, nz, int(y_offset), int(ny_total), float(resolution),
        int(add_virtual_border), device.index or 0, out.data_ptr(),
        min_max.data_ptr() if compute_min_max else None, _stream_handle(device))
    _capi.check(code)
    return out, min_max


def connected_components(cells: torch.Tensor,
                         num_components: torch.Tensor | None = None) -> torch.Tensor:
    """ComputeConnectedComponents (topology_computation.hpp:138-196) on device-resident component
    map cells, in place: ``cells`` is a contiguous int32 or uint32 tensor [nx, ny, nz, words] with
    2 words per cell (OccupancyComponentCell) or 4 (TaggedObjectOccupancyComponentCell), the
    occupancy's float bits in word 0. The component word of every cell gets its component's
    number; the other words are untouched. Returns the number of components as a uint32 device
    tensor [1] (``num_components`` if given). Asynchronous."""
    if not cells.is_cuda:
        raise _capi.BackendUnavailable("cells must live on a CUDA device (no CPU fallback)")
    if cells.dtype not in (torch.int32, torch.uint32) or not cells.is_contiguous():
        raise ValueError("cells must be a contiguous int32 or uint32 tensor")
    if cells.dim() != 4 or cells.shape[3] not in (2, 4):
        raise ValueError("cells must be [nx, ny, nz, 2] or [nx, ny, nz, 4]")
    device = cells.device
    if num_components is None:
        num_components = torch.empty(1, dtype=torch.uint32, device=device)
    _require_cuda(num_components, torch.uint32, "num_components")
    nx, ny, nz, words = cells.shape
    code = _capi.library().vgt_b200_connected_components_dev(
        cells.data_ptr(), 4 * words, nx, ny, nz, device.index or 0, num_components.data_ptr(),
        _stream_handle(device))
    _capi.check(code)
    return num_components


# SDF dtype -> suffix of the cell entries' C-ABI names
_CELL_SDF_SUFFIX = {torch.float32: "f32", torch.float64: "f64"}


def _cell_entry(cells: torch.Tensor, dtype: torch.dtype, name: str):
    if not cells.is_cuda:
        raise _capi.BackendUnavailable("cells must live on a CUDA device (no CPU fallback)")
    if cells.dtype not in (torch.int32, torch.uint32) or not cells.is_contiguous():
        raise ValueError("cells must be a contiguous int32 or uint32 tensor")
    if cells.dim() != 4 or cells.shape[3] not in (2, 4):
        raise ValueError("cells must be [nx, ny, nz, 2] or [nx, ny, nz, 4]")
    if dtype not in _CELL_SDF_SUFFIX:
        raise ValueError(f"the SDF dtype must be torch.float32 or torch.float64, not {dtype}")
    return getattr(_capi.library(), f"{name}_{_CELL_SDF_SUFFIX[dtype]}_dev")


def _object_ids(object_ids) -> np.ndarray:
    return np.ascontiguousarray([int(i) for i in object_ids], dtype=np.uint32)


def signed_distance_field_from_cells(cells: torch.Tensor, resolution: float, objects_to_use=(),
                                     unknown_is_filled: bool = True,
                                     add_virtual_border: bool = False,
                                     dtype: torch.dtype = torch.float32):
    """ExtractSignedDistanceField<T> of a cell map that lives on the device
    (tagged_object_occupancy_map.hpp:199-247; with no objects listed also
    occupancy_component_map.hpp:270-306). ``cells`` has the layout of
    ``connected_components``: a contiguous int32 or uint32 tensor [nx, ny, nz, 2 | 4], the
    occupancy's float bits in word 0 and the object id in word 1. A cell is filled iff the
    occupancy rule holds and (no objects are listed or its object id is listed). Returns
    (sdf ``dtype`` [nx, ny, nz], min_max ``dtype`` [2]). Asynchronous."""
    entry = _cell_entry(cells, dtype, "vgt_b200_sdf_from_cells")
    ids = _object_ids(objects_to_use)
    device = cells.device
    nx, ny, nz, words = cells.shape
    out = torch.empty((nx, ny, nz), dtype=dtype, device=device)
    min_max = torch.empty(2, dtype=dtype, device=device)
    code = entry(cells.data_ptr(), 4 * words, nx, ny, nz, float(resolution),
                 int(unknown_is_filled), int(add_virtual_border),
                 ids.ctypes.data if ids.size else None, ids.size, device.index or 0,
                 out.data_ptr(), min_max.data_ptr(), _stream_handle(device))
    _capi.check(code)
    return out, min_max


def separate_object_sdfs(cells: torch.Tensor, resolution: float, object_ids,
                         unknown_is_filled: bool = True, add_virtual_border: bool = False,
                         dtype: torch.dtype = torch.float32):
    """MakeSeparateObjectSDFs<T> (tagged_object_occupancy_map.hpp:249-262) of a cell map that
    lives on the device (``cells`` as in ``signed_distance_field_from_cells``): SDF k is the
    field of the filled cells whose object id is ``object_ids[k]``. Repeated ids and ids absent
    from the map are allowed. The cells are read once per 255 distinct ids, not once per object.
    Returns (sdfs ``dtype`` [K, nx, ny, nz], min_max ``dtype`` [K, 2]). Asynchronous."""
    entry = _cell_entry(cells, dtype, "vgt_b200_sdf_per_object")
    ids = _object_ids(object_ids)
    device = cells.device
    nx, ny, nz, words = cells.shape
    out = torch.empty((ids.size, nx, ny, nz), dtype=dtype, device=device)
    min_max = torch.empty((ids.size, 2), dtype=dtype, device=device)
    if ids.size == 0:
        return out, min_max
    code = entry(cells.data_ptr(), 4 * words, nx, ny, nz, float(resolution),
                 int(unknown_is_filled), int(add_virtual_border), ids.ctypes.data, ids.size,
                 device.index or 0, out.data_ptr(), min_max.data_ptr(), _stream_handle(device))
    _capi.check(code)
    return out, min_max


def free_and_named_objects_sdf(cells: torch.Tensor, resolution: float,
                               unknown_is_filled: bool = True, add_virtual_border: bool = False,
                               dtype: torch.dtype = torch.float32):
    """ExtractFreeAndNamedObjectsSignedDistanceField<T> (tagged_object_occupancy_map.hpp:293-378)
    of a cell map that lives on the device (``cells`` as in
    ``signed_distance_field_from_cells``). Returns (sdf ``dtype`` [nx, ny, nz],
    min_max ``dtype`` [2]). Asynchronous."""
    entry = _cell_entry(cells, dtype, "vgt_b200_sdf_free_and_named")
    device = cells.device
    nx, ny, nz, words = cells.shape
    out = torch.empty((nx, ny, nz), dtype=dtype, device=device)
    min_max = torch.empty(2, dtype=dtype, device=device)
    code = entry(cells.data_ptr(), 4 * words, nx, ny, nz, float(resolution),
                 int(unknown_is_filled), int(add_virtual_border), device.index or 0,
                 out.data_ptr(), min_max.data_ptr(), _stream_handle(device))
    _capi.check(code)
    return out, min_max


def raycast_cloud(points_xyz: torch.Tensor, x_gc, max_range: float, counts: torch.Tensor,
                  voxel_size: float) -> torch.Tensor:
    """Accumulates one cloud (float64 or float32 [N, 3], cloud frame) into counts int32
    [nx, ny, nz, 2]; float32 points are widened on the device."""
    single = points_xyz.dtype == torch.float32
    _require_cuda(points_xyz, torch.float32 if single else torch.float64, "points_xyz")
    _require_cuda(counts, torch.int32, "counts")
    if counts.dim() != 4 or counts.shape[3] != 2:
        raise ValueError("counts must be [nx, ny, nz, 2]")
    device = counts.device
    column_major = np.ascontiguousarray(np.asarray(x_gc, dtype=np.float64).reshape(4, 4).T)
    nx, ny, nz, _ = counts.shape
    entry = _capi.library().vgt_b200_raycast_f32_dev if single \
        else _capi.library().vgt_b200_raycast_f64_dev
    code = entry(
        points_xyz.data_ptr(), points_xyz.shape[0],
        column_major.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), float(max_range), nx, ny,
        nz, float(voxel_size), device.index or 0, counts.data_ptr(), _stream_handle(device))
    _capi.check(code)
    return counts


def filter_grids(counts: torch.Tensor, occupancy: torch.Tensor,
                 filter_options: PointCloudVoxelizationFilterOptions) -> torch.Tensor:
    """counts int32 [num_grids, nx, ny, nz, 2]; occupancy float32 [nx, ny, nz] updated in place."""
    _require_cuda(counts, torch.int32, "counts")
    _require_cuda(occupancy, torch.float32, "occupancy")
    device = occupancy.device
    options = filter_options.as_struct()
    code = _capi.library().vgt_b200_filter_dev(
        counts.data_ptr(), counts.shape[0], occupancy.numel(), ctypes.byref(options),
        device.index or 0, occupancy.data_ptr(), _stream_handle(device))
    _capi.check(code)
    return occupancy


# --------------------------------------------------------------------------------------------------
# SignedDistanceField queries on a device-resident SDF (SURVEY.md section 8f, rank 2)
# --------------------------------------------------------------------------------------------------
QUERY_NO_VALUE, QUERY_VALUE, QUERY_THROWS = 0, 1, 2

# SDF dtype -> (C view struct, suffix of the C-ABI entry names)
_SDF_SCALAR_TYPES = {torch.float32: (_capi.SdfView, "_dev"),
                     torch.float64: (_capi.SdfViewF64, "_f64_dev")}


class DeviceSignedDistanceField:
    """A SignedDistanceField<float> or SignedDistanceField<double> that stays on the GPU: the
    float32 or float64 grid [nx, ny, nz] plus resolution and origin transform. The batched
    queries mirror the reference's per-point members (signed_distance_field.hpp:808-1203) for
    the grid's scalar type; points are float64 [N, 3] CUDA tensors in the WORLD frame. Every
    query returns (values, valid uint8): 1 = value, 0 = the reference returns an empty query,
    2 = the reference throws for that point."""

    def __init__(self, sdf: torch.Tensor, resolution: float, origin_transform=None):
        if sdf.dtype not in _SDF_SCALAR_TYPES:
            raise ValueError(f"sdf must be a float32 or float64 tensor, not {sdf.dtype}")
        _require_cuda(sdf, sdf.dtype, "sdf")
        if sdf.dim() != 3:
            raise ValueError("sdf must be indexed [x, y, z]")
        self.sdf = sdf
        self.resolution = float(resolution)
        self.origin_transform = np.eye(4) if origin_transform is None else \
            np.asarray(origin_transform, dtype=np.float64).reshape(4, 4)
        view_type, self._entry_suffix = _SDF_SCALAR_TYPES[sdf.dtype]
        self._view = view_type()
        self._view.d_sdf = sdf.data_ptr()
        self._view.nx, self._view.ny, self._view.nz = (int(d) for d in sdf.shape)
        self._view.resolution = self.resolution
        column_major = np.ascontiguousarray(self.origin_transform.T).reshape(-1)
        for i in range(16):
            self._view.origin_transform[i] = float(column_major[i])

    def _points(self, points: torch.Tensor) -> torch.Tensor:
        _require_cuda(points, torch.float64, "points")
        if points.dim() != 2 or points.shape[1] != 3:
            raise ValueError("points must be [N, 3]")
        if points.device != self.sdf.device:
            raise ValueError("points and sdf must live on the same device")
        return points

    def _launch(self, name, points, width, *middle):
        points = self._points(points)
        device = self.sdf.device
        count = points.shape[0]
        shape = (count,) if width == 1 else (count, width)
        values = torch.empty(shape, dtype=torch.float64, device=device)
        valid = torch.empty(count, dtype=torch.uint8, device=device)
        function = getattr(_capi.library(), name + self._entry_suffix)
        code = function(ctypes.byref(self._view), points.data_ptr(), count, *middle,
                        device.index or 0, values.data_ptr(), valid.data_ptr(),
                        _stream_handle(device))
        _capi.check(code)
        return values, valid

    def EstimateLocationDistance(self, points: torch.Tensor):
        return self._launch("vgt_b200_sdf_estimate_distance", points, 1)

    def GetLocationCoarseGradient(self, points: torch.Tensor, enable_edge_gradients=False):
        return self._launch("vgt_b200_sdf_coarse_gradient", points, 3,
                            int(bool(enable_edge_gradients)))

    def GetLocationFineGradient(self, points: torch.Tensor, nominal_window_size: float):
        return self._launch("vgt_b200_sdf_fine_gradient", points, 3,
                            float(nominal_window_size))

    def ProjectLocationOutOfCollisionToMinimumDistance(
            self, points: torch.Tensor, minimum_distance: float = 0.0,
            stepsize_multiplier: float = 1.0 / 10.0, max_steps: int = 1_000_000):
        return self._launch("vgt_b200_sdf_project_out_of_collision", points, 3,
                            float(minimum_distance), float(stepsize_multiplier), int(max_steps))

    def ProjectLocationOutOfCollision(self, points: torch.Tensor,
                                      stepsize_multiplier: float = 1.0 / 10.0):
        return self.ProjectLocationOutOfCollisionToMinimumDistance(points, 0.0,
                                                                   stepsize_multiplier)

    def ComputeLocalExtremaMap(self) -> torch.Tensor:
        """float64 [nx, ny, nz, 3]: per cell the grid-frame centre of the cell its gradient walk
        ends at, +inf when it leaves the grid (signed_distance_field.hpp:1207-1231)."""
        device = self.sdf.device
        extrema = torch.empty(tuple(self.sdf.shape) + (3,), dtype=torch.float64, device=device)
        function = getattr(_capi.library(), "vgt_b200_sdf_local_extrema_map" + self._entry_suffix)
        code = function(ctypes.byref(self._view), device.index or 0, extrema.data_ptr(),
                        _stream_handle(device))
        _capi.check(code)
        return extrema


class ComponentSlab:
    """One rank's x-slab of a component map between the phases of the per-slab connected-
    component entries (``vgt_b200_components_*``; DESIGN.md section 8): the cells [nx_r, ny, nz,
    2 | 4] (contiguous int32 or uint32, labelled in place) and every array that lives from one
    phase to the next. ``base`` is the global index of the slab's first cell. Each phase is
    asynchronous on torch's current stream; the ones that return a number read it back."""

    def __init__(self, cells: torch.Tensor, base: int):
        if not cells.is_cuda:
            raise _capi.BackendUnavailable("cells must live on a CUDA device (no CPU fallback)")
        if cells.dtype not in (torch.int32, torch.uint32) or not cells.is_contiguous():
            raise ValueError("cells must be a contiguous int32 or uint32 tensor")
        if cells.dim() != 4 or cells.shape[3] not in (2, 4):
            raise ValueError("cells must be [nx, ny, nz, 2] or [nx, ny, nz, 4]")
        self.cells = cells
        self.base = int(base)
        self.device = cells.device
        self.dims = tuple(int(d) for d in cells.shape[:3])
        self.cell_bytes = 4 * int(cells.shape[3])
        nx, ny, nz = self.dims
        count = nx * ny * nz
        root_words = (count + 31) // 32
        scan_bytes = ctypes.c_size_t()
        _capi.check(_capi.library().vgt_b200_components_slab_scan_bytes(
            nx, ny, nz, self._index(), ctypes.byref(scan_bytes)))
        self.parent = self._empty(count, torch.int32)
        self.mask = self._empty(root_words, torch.int32)
        self.word_prefix = self._empty(root_words + 1, torch.int32)
        self.scan_storage = self._empty(scan_bytes.value, torch.uint8)
        self.num_local = self.num_nodes = self.first_node = self.num_slab_nodes = 0
        self.nodes = self.node_roots = self.bits = self.bit_prefix = self.final_ids = None

    def _index(self) -> int:
        return self.device.index or 0

    def _empty(self, count: int, dtype: torch.dtype) -> torch.Tensor:
        return torch.empty(count, dtype=dtype, device=self.device)

    def _stream(self) -> int:
        return _stream_handle(self.device)

    def local(self, face_roots: bool) -> torch.Tensor | None:
        """Labels the slab on its own; returns the local roots of its last x-plane (int32
        [ny * nz]) when ``face_roots``, for the slab above."""
        nx, ny, nz = self.dims
        roots = self._empty(ny * nz, torch.int32) if face_roots else None
        _capi.check(_capi.library().vgt_b200_components_slab_local(
            self.cells.data_ptr(), self.cell_bytes, nx, ny, nz, self._index(),
            self.parent.data_ptr(), self.mask.data_ptr(), self.word_prefix.data_ptr(),
            self.scan_storage.data_ptr(), self.scan_storage.numel(),
            None if roots is None else roots.data_ptr(), self._stream()))
        return roots

    def face_edges(self, below_cells: torch.Tensor, below_roots: torch.Tensor,
                   below_base: int) -> torch.Tensor:
        """The edges (int64 [E, 2]) of the face between the last x-plane of the slab below
        (its cells [ny, nz, words] and local roots [ny * nz]) and this slab's first."""
        nx, ny, nz = self.dims
        _require_cuda(below_roots, torch.int32, "below_roots")
        if (not below_cells.is_cuda or not below_cells.is_contiguous()
                or below_cells.numel() != ny * nz * self.cell_bytes // 4
                or below_roots.numel() != ny * nz):
            raise ValueError("the face below must be one contiguous x-plane of cells and roots")
        edges = torch.empty((ny * nz, 2), dtype=torch.int64, device=self.device)
        count = self._empty(1, torch.int32)
        _capi.check(_capi.library().vgt_b200_components_slab_face_edges(
            below_cells.data_ptr(), below_roots.data_ptr(), int(below_base),
            self.cells.data_ptr(), self.cell_bytes, nx, ny, nz, self.base, self._index(),
            self.parent.data_ptr(), edges.data_ptr(), count.data_ptr(), self._stream()))
        return edges[:int(count.item())]

    def resolve(self, edges: torch.Tensor, num_cells: int) -> int:
        """The face graph of all faces' edges (int64 [E, 2], any order) of a map of ``num_cells``
        cells; returns the number of nodes (the same on every slab given the same edges)."""
        _require_cuda(edges, torch.int64, "edges")
        capacity = max(1, 2 * edges.shape[0])
        self.nodes = self._empty(capacity, torch.int64)
        self.node_roots = self._empty(capacity, torch.int32)
        node_range = self._empty(3, torch.int32)
        nx, ny, nz = self.dims
        _capi.check(_capi.library().vgt_b200_components_resolve(
            edges.data_ptr() if edges.numel() else None, edges.shape[0], int(num_cells), self.base,
            self.base + nx * ny * nz, self._index(), self.nodes.data_ptr(),
            self.node_roots.data_ptr(), node_range.data_ptr(), self._stream()))
        self.num_nodes, self.first_node, end = node_range.tolist()
        self.num_slab_nodes = end - self.first_node
        return self.num_nodes

    def _node_arguments(self):
        return (self.nodes.data_ptr(), self.num_nodes, self.first_node, self.num_slab_nodes)

    def count(self) -> int:
        """count_g: the slab's components whose smallest index lies in the slab."""
        nx, ny, nz = self.dims
        self.num_local = int(self.word_prefix[-1].item()) & 0xFFFFFFFF
        bit_words = (self.num_local + 31) // 32
        self.bits = self._empty(bit_words, torch.int32)
        self.bit_prefix = self._empty(bit_words + 1, torch.int32)
        nodes, num_nodes, first, own = self._node_arguments()
        _capi.check(_capi.library().vgt_b200_components_slab_count(
            nx, ny, nz, self.base, self.num_local, self._index(), self.mask.data_ptr(),
            self.word_prefix.data_ptr(), nodes, self.node_roots.data_ptr(), num_nodes, first, own,
            self.bits.data_ptr(), self.bit_prefix.data_ptr(), self.scan_storage.data_ptr(),
            self.scan_storage.numel(), self._stream()))
        return int(self.bit_prefix[-1].item()) & 0xFFFFFFFF

    def publish(self, offset: int) -> torch.Tensor:
        """The final ids of the slab's components numbered from ``offset`` + 1; returns the node
        ids (int32 [number of nodes] holding uint32 ids): this slab's nodes set, zero elsewhere."""
        nx, ny, nz = self.dims
        self.final_ids = self._empty(self.num_local, torch.int32)
        node_ids = torch.zeros(max(1, self.num_nodes), dtype=torch.int32, device=self.device)
        nodes, num_nodes, first, own = self._node_arguments()
        _capi.check(_capi.library().vgt_b200_components_slab_publish(
            nx, ny, nz, self.base, self.num_local, int(offset), self._index(),
            self.mask.data_ptr(), self.word_prefix.data_ptr(), nodes, num_nodes, first, own,
            self.bits.data_ptr(), self.bit_prefix.data_ptr(), self.final_ids.data_ptr(),
            node_ids.data_ptr(), self._stream()))
        return node_ids[:self.num_nodes]

    def write(self, node_ids: torch.Tensor) -> None:
        """The component word of every cell, from the node ids of every slab added up."""
        nx, ny, nz = self.dims
        if node_ids.numel() != self.num_nodes:
            raise ValueError(f"expected {self.num_nodes} node ids, got {node_ids.numel()}")
        _require_cuda(node_ids, torch.int32, "node_ids")
        nodes, num_nodes, first, own = self._node_arguments()
        _capi.check(_capi.library().vgt_b200_components_slab_write(
            self.cells.data_ptr(), self.cell_bytes, nx, ny, nz, self.base, self.num_local,
            self._index(), self.parent.data_ptr(), self.mask.data_ptr(),
            self.word_prefix.data_ptr(), nodes, self.node_roots.data_ptr(), num_nodes, first, own,
            node_ids.data_ptr() if num_nodes else None, self.final_ids.data_ptr(),
            self._stream()))
