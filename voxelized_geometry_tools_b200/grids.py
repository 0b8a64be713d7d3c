"""Host-side mirror of the grid value types on the hot path.

Names, argument meaning and error behaviour follow the reference so parity tests read like the
reference's own (paths relative to the reference checkout):

* ``OccupancyMap``                      include/voxelized_geometry_tools/occupancy_map.hpp:65-216
* ``SignedDistanceField``               include/voxelized_geometry_tools/signed_distance_field.hpp:193-211, 724-795
* ``SignedDistanceFieldGenerationParameters``  signed_distance_field.hpp:1234-1264
* ``VoxelGridSizes``                    common_robotics_utilities voxel_grid.hpp (FromGridSizes /
  FromVoxelCounts; cell count = ceil(size / voxel_size), consistent with
  test/sdf_generation_test.cpp:267-272 -> 4 x 8 x 12)

* ``OccupancyComponentMap``, ``TaggedObjectOccupancyMap``, ``TaggedObjectOccupancyComponentMap``
  (SURVEY.md section 8f, rank 1): the cell layouts and the SDF entry points of
  occupancy_component_map.hpp:270-306, tagged_object_occupancy_map.hpp:199-378 and
  tagged_object_occupancy_component_map.hpp:360-575.

Only what the occupancy -> SDF path needs is here: storage, the filled predicate's inputs, the
Extract entry points and Lock()/min-max, plus ``UpdateConnectedComponents`` of the two component
maps (topology_computation.hpp:138-196). Queries, gradients and serialization are out of scope.
"""
from __future__ import annotations

import ctypes
import math
from dataclasses import dataclass

import numpy as np

from . import _capi



def compose_rigid(a, b) -> np.ndarray:
    """a * b for rigid 4x4 transforms with ONE fixed operation order, element (r, c) =
    ((a[r,0]*b[0,c] + a[r,1]*b[1,c]) + a[r,2]*b[2,c]) + a[r,3]*b[3,c], no fused multiply-add.
    The voxelizer's counts depend on the last bits of X_GC = X_GW * X_WC
    (cpu_pointcloud_voxelization.cpp:172-176), and a BLAS matmul is free to sum in another
    order; the C++ adapter, the test suite's stand-in for Eigen (its header states the order) and
    this function all use this order (tests/test_oracle_vs_reference.py pins it)."""
    a = np.asarray(a, dtype=np.float64).reshape(4, 4)
    b = np.asarray(b, dtype=np.float64).reshape(4, 4)
    out = np.empty((4, 4), dtype=np.float64)
    for r in range(4):
        for c in range(4):
            out[r, c] = ((a[r, 0] * b[0, c] + a[r, 1] * b[1, c]) + a[r, 2] * b[2, c]) \
                + a[r, 3] * b[3, c]
    return out


def inverse_rigid(transform) -> np.ndarray:
    """Inverse of a rigid transform: R^T and -(R^T t) with t summed left to right, as the
    test suite's stand-in for Eigen::Isometry3d::inverse() does."""
    m = np.asarray(transform, dtype=np.float64).reshape(4, 4)
    inverse = np.eye(4)
    for r in range(3):
        for c in range(3):
            inverse[r, c] = m[c, r]
    for r in range(3):
        inverse[r, 3] = -((inverse[r, 0] * m[0, 3] + inverse[r, 1] * m[1, 3])
                          + inverse[r, 2] * m[2, 3])
    return inverse


@dataclass(frozen=True)
class VoxelGridSizes:
    voxel_size: float
    num_x_voxels: int
    num_y_voxels: int
    num_z_voxels: int

    @staticmethod
    def FromGridSizes(voxel_size: float, sizes) -> "VoxelGridSizes":
        if not (voxel_size > 0.0 and math.isfinite(voxel_size)):
            raise ValueError("voxel_size must be positive and finite")
        counts = [int(math.ceil(float(s) / voxel_size)) for s in sizes]
        if min(counts) < 1:
            raise ValueError("all grid sizes must be positive")
        return VoxelGridSizes(float(voxel_size), *counts)

    @staticmethod
    def FromVoxelCounts(voxel_size: float, counts) -> "VoxelGridSizes":
        if not (voxel_size > 0.0 and math.isfinite(voxel_size)):
            raise ValueError("voxel_size must be positive and finite")
        counts = [int(c) for c in counts]
        if min(counts) < 1:
            raise ValueError("all voxel counts must be positive")
        return VoxelGridSizes(float(voxel_size), *counts)

    @property
    def shape(self):
        return (self.num_x_voxels, self.num_y_voxels, self.num_z_voxels)

    def sizes(self):
        return tuple(c * self.voxel_size for c in self.shape)


class SignedDistanceFieldGenerationParameters:
    """signed_distance_field.hpp:1234-1264. ``parallelism`` is accepted and ignored on device."""

    def __init__(self, oob_value=float("inf"), parallelism=None, unknown_is_filled: bool = True,
                 add_virtual_border: bool = False):
        self._oob_value = oob_value
        self._parallelism = parallelism
        self._unknown_is_filled = bool(unknown_is_filled)
        self._add_virtual_border = bool(add_virtual_border)

    def OOBValue(self):
        return self._oob_value

    def Parallelism(self):
        return self._parallelism

    def UnknownIsFilled(self) -> bool:
        return self._unknown_is_filled

    def AddVirtualBorder(self) -> bool:
        return self._add_virtual_border


class SignedDistanceField:
    """Result container: raw [x, y, z] data, frame, lock flag and cached min/max."""

    def __init__(self, origin_transform, frame: str, sizes: VoxelGridSizes, data: np.ndarray,
                 oob_value, minimum_maximum=None):
        self._origin_transform = np.array(origin_transform, dtype=np.float64).reshape(4, 4)
        self._frame = frame
        self._sizes = sizes
        self._data = data
        self._oob_value = oob_value
        self._locked = False
        self._minimum_maximum = minimum_maximum

    # --- VoxelGridBase-like accessors -------------------------------------------------------
    def NumXVoxels(self):
        return self._sizes.num_x_voxels

    def NumYVoxels(self):
        return self._sizes.num_y_voxels

    def NumZVoxels(self):
        return self._sizes.num_z_voxels

    def Resolution(self):
        return self._sizes.voxel_size

    def Frame(self):
        return self._frame

    def ControlSizes(self):
        return self._sizes

    def OriginTransform(self):
        return self._origin_transform

    def GetImmutableRawData(self) -> np.ndarray:
        return self._data

    def GetIndexImmutable(self, x: int, y: int, z: int):
        """Value at an index; out of bounds returns the OOB value like a failed query would."""
        if (0 <= x < self.NumXVoxels() and 0 <= y < self.NumYVoxels()
                and 0 <= z < self.NumZVoxels()):
            return self._data[x, y, z]
        return self._data.dtype.type(self._oob_value)

    # --- locking + min/max (signed_distance_field.hpp:765-789) ----------------------------
    def IsLocked(self) -> bool:
        return self._locked

    def Lock(self) -> None:
        if self._minimum_maximum is None:
            self._minimum_maximum = (self._data.min(), self._data.max())
        self._locked = True
        self._data.setflags(write=False)

    def Unlock(self) -> None:
        self._locked = False
        self._data = np.array(self._data)  # writable copy
        self._minimum_maximum = None

    def GetMinimumMaximum(self):
        if not self._locked:
            raise RuntimeError("Cannot get min/max of an unlocked SDF")
        return self._minimum_maximum

    # --- files (signed_distance_field.hpp:643-722), through csrc/grid_files.cu -----------------
    @staticmethod
    def SaveToFile(sdf: "SignedDistanceField", filepath, compress: bool) -> None:
        from . import grid_files
        grid_files.SaveSignedDistanceFieldToFile(sdf, filepath, compress)

    @staticmethod
    def LoadFromFile(filepath, dtype=None) -> "SignedDistanceField":
        from . import grid_files
        return grid_files.LoadSignedDistanceFieldFromFile(filepath, dtype)


class OccupancyMap:
    """Dense occupancy grid: one float per cell, <0.5 free, 0.5 unknown, >0.5 filled
    (occupancy_map.hpp:28-58). Data is indexed [x, y, z], z contiguous."""

    def __init__(self, origin_transform, frame: str, sizes: VoxelGridSizes,
                 default_occupancy: float = 0.0, data: np.ndarray | None = None):
        self._origin_transform = np.array(origin_transform, dtype=np.float64).reshape(4, 4)
        self._frame = frame
        self._sizes = sizes
        # (the reference hands one cell to the grid as default and out-of-bounds value)
        self._default_occupancy = float(default_occupancy)
        self._oob_occupancy = float(default_occupancy)
        if data is None:
            self._data = np.full(sizes.shape, default_occupancy, dtype=np.float32)
        else:
            data = np.ascontiguousarray(data, dtype=np.float32)
            if data.shape != sizes.shape:
                raise ValueError("data shape does not match the grid sizes")
            self._data = data

    def IsInitialized(self) -> bool:
        return True

    def HasUniformVoxelSize(self) -> bool:
        return True  # VoxelGridSizes here only models cubic voxels

    def NumXVoxels(self):
        return self._sizes.num_x_voxels

    def NumYVoxels(self):
        return self._sizes.num_y_voxels

    def NumZVoxels(self):
        return self._sizes.num_z_voxels

    def NumTotalVoxels(self):
        return self._data.size

    def VoxelXSize(self):
        return self._sizes.voxel_size

    def ControlSizes(self):
        return self._sizes

    def Frame(self):
        return self._frame

    def OriginTransform(self):
        return self._origin_transform

    def InverseOriginTransform(self):
        return inverse_rigid(self._origin_transform)

    def GetMutableRawData(self) -> np.ndarray:
        return self._data

    def GetImmutableRawData(self) -> np.ndarray:
        return self._data

    def SetIndex(self, x: int, y: int, z: int, occupancy: float) -> bool:
        if (0 <= x < self.NumXVoxels() and 0 <= y < self.NumYVoxels()
                and 0 <= z < self.NumZVoxels()):
            self._data[x, y, z] = occupancy
            return True
        return False

    def copy(self) -> "OccupancyMap":
        return OccupancyMap(self._origin_transform, self._frame, self._sizes,
                            data=self._data.copy())

    # --- files (occupancy_map.cpp:116-193), through csrc/grid_files.cu -------------------------
    @staticmethod
    def SaveToFile(occupancy_map: "OccupancyMap", filepath, compress: bool) -> None:
        from . import grid_files
        grid_files.SaveOccupancyMapToFile(occupancy_map, filepath, compress)

    @staticmethod
    def LoadFromFile(filepath) -> "OccupancyMap":
        from . import grid_files
        return grid_files.LoadOccupancyMapFromFile(filepath)

    # --- the path's entry points (occupancy_map.hpp:174-216, occupancy_map.cpp:250-260) ----
    def ExtractSignedDistanceField(self, parameters: SignedDistanceFieldGenerationParameters,
                                   dtype=np.float32, device: int = 0,
                                   devices=None) -> SignedDistanceField:
        """devices: several device ordinals -> the slab-sharded multi-device call
        (vgt_b200_sdf_f32_multi / vgt_b200_sdf_f64_multi), same result bit for bit."""
        device, listed = _device_choice(device, devices)
        lib = _capi.library()
        occupancy = self._data
        nx, ny, nz = self._sizes.shape
        out = np.empty(self._sizes.shape, dtype=dtype)
        if listed is not None:
            suffix, scalar = _scalar_suffix(dtype)
            lo, hi = scalar(), scalar()
            code = getattr(lib, f"vgt_b200_sdf_{suffix}_multi")(
                occupancy.ctypes.data, nx, ny, nz, self._sizes.voxel_size,
                int(parameters.UnknownIsFilled()), int(parameters.AddVirtualBorder()), listed,
                len(listed), out.ctypes.data, ctypes.byref(lo), ctypes.byref(hi))
        elif np.dtype(dtype) == np.float32:
            lo, hi = ctypes.c_float(), ctypes.c_float()
            code = lib.vgt_b200_sdf_f32(
                occupancy.ctypes.data, nx, ny, nz, self._sizes.voxel_size,
                int(parameters.UnknownIsFilled()), int(parameters.AddVirtualBorder()), device,
                out.ctypes.data, ctypes.byref(lo), ctypes.byref(hi))
        elif np.dtype(dtype) == np.float64:
            lo, hi = ctypes.c_double(), ctypes.c_double()
            code = lib.vgt_b200_sdf_f64(
                occupancy.ctypes.data, nx, ny, nz, self._sizes.voxel_size,
                int(parameters.UnknownIsFilled()), int(parameters.AddVirtualBorder()), device,
                out.ctypes.data, ctypes.byref(lo), ctypes.byref(hi))
        else:
            raise ValueError("SDF scalar type must be float32 or float64")
        _capi.check(code)
        sdf = SignedDistanceField(
            self._origin_transform, self._frame, self._sizes, out, parameters.OOBValue(),
            minimum_maximum=(out.dtype.type(lo.value), out.dtype.type(hi.value)))
        sdf.Lock()
        return sdf

    def ExtractSignedDistanceFieldFloat(self, parameters, device: int = 0, devices=None):
        return self.ExtractSignedDistanceField(parameters, np.float32, device, devices)

    def ExtractSignedDistanceFieldDouble(self, parameters, device: int = 0, devices=None):
        return self.ExtractSignedDistanceField(parameters, np.float64, device, devices)


def _device_choice(device, devices):
    """The device arguments of the SDF members: ``devices=None`` runs on ``device``, one entry on
    that device, and two or more on the multi-device entry, which cuts the map into one x-slab per
    listed device (distinct ordinals, at most 8). Returns (device, ctypes device list or None)."""
    if not devices:
        _capi.require_device(device)
        return device, None
    ordinals = [int(d) for d in devices]
    _capi.require_device(ordinals[0])
    if len(ordinals) == 1:
        return ordinals[0], None
    return ordinals[0], (ctypes.c_int * len(ordinals))(*ordinals)


# Packed cell layouts of the other map types; the reference pins their sizes with static_asserts
# (occupancy_component_map.hpp:66-71, tagged_object_occupancy_map.hpp:66-70,
# tagged_object_occupancy_component_map.hpp:62-66).
OCCUPANCY_COMPONENT_CELL = np.dtype([("occupancy", "<f4"), ("component", "<u4")])
TAGGED_OBJECT_OCCUPANCY_CELL = np.dtype([("occupancy", "<f4"), ("object_id", "<u4")])
TAGGED_OBJECT_OCCUPANCY_COMPONENT_CELL = np.dtype(
    [("occupancy", "<f4"), ("object_id", "<u4"), ("component", "<u4"),
     ("spatial_segment", "<u4")])


class _CellGrid:
    """A dense grid of packed cells indexed [x, y, z]; what the three maps below share."""

    CELL = None

    def __init__(self, origin_transform, frame: str, sizes: VoxelGridSizes,
                 data: np.ndarray | None = None):
        self._origin_transform = np.array(origin_transform, dtype=np.float64).reshape(4, 4)
        self._frame = frame
        self._sizes = sizes
        if data is None:
            self._data = np.zeros(sizes.shape, dtype=self.CELL)
        else:
            data = np.ascontiguousarray(data, dtype=self.CELL)
            if data.shape != sizes.shape:
                raise ValueError("data shape does not match the grid sizes")
            self._data = data

    def NumXVoxels(self):
        return self._sizes.num_x_voxels

    def NumYVoxels(self):
        return self._sizes.num_y_voxels

    def NumZVoxels(self):
        return self._sizes.num_z_voxels

    def ControlSizes(self):
        return self._sizes

    def Frame(self):
        return self._frame

    def OriginTransform(self):
        return self._origin_transform

    def HasUniformVoxelSize(self) -> bool:
        return True

    def GetMutableRawData(self) -> np.ndarray:
        return self._data

    def GetImmutableRawData(self) -> np.ndarray:
        return self._data

    # ------------------------------------------------------------------ shared plumbing
    def _wrap(self, out, lo, hi, parameters):
        sdf = SignedDistanceField(self._origin_transform, self._frame, self._sizes, out,
                                  parameters.OOBValue(),
                                  minimum_maximum=(out.dtype.type(lo), out.dtype.type(hi)))
        sdf.Lock()
        return sdf

    @staticmethod
    def _cell_entry(name, suffix, device, devices):
        """The host entry vgt_b200_<name>_<suffix> and its device argument, or its multi-device
        entry and its (device list, count) arguments."""
        device, listed = _device_choice(device, devices)
        lib = _capi.library()
        if listed is None:
            return getattr(lib, f"vgt_b200_{name}_{suffix}"), (device,)
        return getattr(lib, f"vgt_b200_{name}_{suffix}_multi"), (listed, len(listed))

    def _from_cells(self, objects_to_use, parameters, dtype, device, devices=None):
        suffix, scalar = _scalar_suffix(dtype)
        function, device_arguments = self._cell_entry("sdf_from_cells", suffix, device, devices)
        ids = np.ascontiguousarray(list(objects_to_use), dtype=np.uint32)
        out = np.empty(self._sizes.shape, dtype=dtype)
        lo, hi = scalar(), scalar()
        code = function(self._data.ctypes.data, self.CELL.itemsize, *self._sizes.shape,
                        self._sizes.voxel_size, int(parameters.UnknownIsFilled()),
                        int(parameters.AddVirtualBorder()),
                        ids.ctypes.data if ids.size else None, ids.size, *device_arguments,
                        out.ctypes.data, ctypes.byref(lo), ctypes.byref(hi))
        _capi.check(code)
        return self._wrap(out, lo.value, hi.value, parameters)

    def _connected_components(self, device, devices=None):
        count = ctypes.c_uint32()
        if devices and len(devices) > 1:
            listed = [int(d) for d in devices]
            for ordinal in sorted(set(listed)):
                _capi.require_device(ordinal)
            code = _capi.library().vgt_b200_connected_components_multi(
                self._data.ctypes.data, self.CELL.itemsize, *self._sizes.shape,
                (ctypes.c_int * len(listed))(*listed), len(listed), ctypes.byref(count))
        else:
            device = int(devices[0]) if devices else device
            _capi.require_device(device)
            code = _capi.library().vgt_b200_connected_components(
                self._data.ctypes.data, self.CELL.itemsize, *self._sizes.shape, device,
                ctypes.byref(count))
        _capi.check(code)
        return int(count.value)


def _scalar_suffix(dtype):
    if np.dtype(dtype) == np.float32:
        return "f32", ctypes.c_float
    if np.dtype(dtype) == np.float64:
        return "f64", ctypes.c_double
    raise ValueError("SDF scalar type must be float32 or float64")


class OccupancyComponentMap(_CellGrid):
    """occupancy_component_map.hpp: cells {occupancy, component}; the component never enters the
    SDF predicate (occupancy_component_map.hpp:270-306)."""

    CELL = OCCUPANCY_COMPONENT_CELL

    def ExtractSignedDistanceField(self, parameters, dtype=np.float32, device: int = 0,
                                   devices=None):
        """``devices``: two or more distinct device ordinals (at most 8) cut the map into one
        x-slab per device (vgt_b200_sdf_from_cells_*_multi), for maps one device cannot hold;
        the same field and min/max as on one device."""
        return self._from_cells((), parameters, dtype, device, devices)

    def ExtractSignedDistanceFieldFloat(self, parameters, device: int = 0, devices=None):
        return self.ExtractSignedDistanceField(parameters, np.float32, device, devices)

    def ExtractSignedDistanceFieldDouble(self, parameters, device: int = 0, devices=None):
        return self.ExtractSignedDistanceField(parameters, np.float64, device, devices)

    def UpdateConnectedComponents(self, device: int = 0, devices=None) -> int:
        """Labels the connected components of the map into every cell's ``component`` and returns
        their number (ComputeConnectedComponents, topology_computation.hpp:138-196): face
        neighbours are connected iff both are filled (> 0.5) or both are not; components are
        numbered from 1 in the order of their first cell in storage order. Recomputed on every
        call (nothing is cached).
        ``devices``: two or more device ordinals (repeats allowed, at most 8, no more than the
        map's x size) label the map cut into that many x-slabs, slab g on ``devices[g]``
        (vgt_b200_connected_components_multi): the same ids and count as on one device, and
        maps of 2^32 cells or more when no slab reaches 2^32 cells."""
        return self._connected_components(device, devices)


class TaggedObjectOccupancyMap(_CellGrid):
    """tagged_object_occupancy_map.hpp: cells {occupancy, object_id}."""

    CELL = TAGGED_OBJECT_OCCUPANCY_CELL

    def ExtractSignedDistanceField(self, objects_to_use, parameters, dtype=np.float32,
                                   device: int = 0, devices=None):
        """Filled = occupancy rule and (no objects listed or object id listed)
        (tagged_object_occupancy_map.hpp:199-247).
        ``devices`` (here and on every SDF member below): two or more distinct device ordinals
        (at most 8) cut the map into one x-slab per device (the *_multi entries), for maps one
        device cannot hold; the same fields and min/max as on one device."""
        return self._from_cells(objects_to_use, parameters, dtype, device, devices)

    def ExtractSignedDistanceFieldFloat(self, objects_to_use, parameters, device: int = 0,
                                        devices=None):
        return self.ExtractSignedDistanceField(objects_to_use, parameters, np.float32, device,
                                               devices)

    def ExtractSignedDistanceFieldDouble(self, objects_to_use, parameters, device: int = 0,
                                         devices=None):
        return self.ExtractSignedDistanceField(objects_to_use, parameters, np.float64, device,
                                               devices)

    def MakeSeparateObjectSDFs(self, object_ids, parameters, dtype=np.float32, device: int = 0,
                               devices=None):
        """One SDF per object id, the cells uploaded once
        (tagged_object_occupancy_map.hpp:249-262). Returns {object_id: SignedDistanceField}."""
        suffix, _ = _scalar_suffix(dtype)
        function, device_arguments = self._cell_entry("sdf_per_object", suffix, device, devices)
        ids = np.ascontiguousarray(list(object_ids), dtype=np.uint32)
        if ids.size == 0:
            return {}
        out = np.empty((ids.size,) + self._sizes.shape, dtype=dtype)
        lows = np.empty(ids.size, dtype=dtype)
        highs = np.empty(ids.size, dtype=dtype)
        code = function(self._data.ctypes.data, self.CELL.itemsize, *self._sizes.shape,
                        self._sizes.voxel_size, int(parameters.UnknownIsFilled()),
                        int(parameters.AddVirtualBorder()), ids.ctypes.data, ids.size,
                        *device_arguments, out.ctypes.data, lows.ctypes.data, highs.ctypes.data)
        _capi.check(code)
        return {int(object_id): self._wrap(out[k], lows[k], highs[k], parameters)
                for k, object_id in enumerate(ids)}

    def MakeAllObjectSDFs(self, parameters, dtype=np.float32, device: int = 0, devices=None):
        """Every object id > 0 present in the map (tagged_object_occupancy_map.hpp:264-291)."""
        object_ids = np.unique(self._data["object_id"])
        return self.MakeSeparateObjectSDFs([i for i in object_ids.tolist() if i > 0], parameters,
                                           dtype, device, devices)

    def ExtractFreeAndNamedObjectsSignedDistanceField(self, parameters, dtype=np.float32,
                                                      device: int = 0, devices=None):
        """tagged_object_occupancy_map.hpp:293-378."""
        suffix, scalar = _scalar_suffix(dtype)
        function, device_arguments = self._cell_entry("sdf_free_and_named", suffix, device,
                                                      devices)
        out = np.empty(self._sizes.shape, dtype=dtype)
        lo, hi = scalar(), scalar()
        code = function(self._data.ctypes.data, self.CELL.itemsize, *self._sizes.shape,
                        self._sizes.voxel_size, int(parameters.UnknownIsFilled()),
                        int(parameters.AddVirtualBorder()), *device_arguments, out.ctypes.data,
                        ctypes.byref(lo), ctypes.byref(hi))
        _capi.check(code)
        return self._wrap(out, lo.value, hi.value, parameters)


class TaggedObjectOccupancyComponentMap(TaggedObjectOccupancyMap):
    """tagged_object_occupancy_component_map.hpp: 16-byte cells {occupancy, object_id, component,
    spatial_segment}; the same SDF entry points (:360-575)."""

    CELL = TAGGED_OBJECT_OCCUPANCY_COMPONENT_CELL

    def UpdateConnectedComponents(self, device: int = 0, devices=None) -> int:
        """Labels the connected components of the map into every cell's ``component`` and returns
        their number (ComputeConnectedComponents, topology_computation.hpp:138-196): face
        neighbours are connected iff both are filled (> 0.5) or both are not, and their object
        ids are equal; components are numbered from 1 in the order of their first cell in storage
        order. ``object_id`` and ``spatial_segment`` are left as they are. Recomputed on every
        call (nothing is cached).
        ``devices``: two or more device ordinals (repeats allowed, at most 8, no more than the
        map's x size) label the map cut into that many x-slabs, slab g on ``devices[g]``
        (vgt_b200_connected_components_multi): the same ids and count as on one device, and
        maps of 2^32 cells or more when no slab reaches 2^32 cells."""
        return self._connected_components(device, devices)


def ExtractSignedDistanceFieldFromMask(filled_mask: np.ndarray, origin_transform, frame: str,
                                       sizes: VoxelGridSizes,
                                       parameters: SignedDistanceFieldGenerationParameters,
                                       device: int = 0) -> SignedDistanceField:
    """internal::ExtractSignedDistanceField for an opaque predicate
    (signed_distance_field_generation.hpp:115-121): the caller evaluates it into a mask."""
    _capi.require_device(device)
    mask = np.ascontiguousarray(filled_mask, dtype=np.uint8)
    if mask.shape != sizes.shape:
        raise ValueError("mask shape does not match the grid sizes")
    out = np.empty(sizes.shape, dtype=np.float32)
    lo, hi = ctypes.c_float(), ctypes.c_float()
    code = _capi.library().vgt_b200_sdf_from_mask_f32(
        mask.ctypes.data, *sizes.shape, sizes.voxel_size, int(parameters.AddVirtualBorder()),
        device, out.ctypes.data, ctypes.byref(lo), ctypes.byref(hi))
    _capi.check(code)
    sdf = SignedDistanceField(origin_transform, frame, sizes, out, parameters.OOBValue(),
                              minimum_maximum=(np.float32(lo.value), np.float32(hi.value)))
    sdf.Lock()
    return sdf


def ComputeSquaredDistanceFields(occupancy: np.ndarray, unknown_is_filled: bool = True,
                                 device: int = 0):
    """Parity hook: (dist_to_filled_sq, dist_to_free_sq) int32, _capi.SQ_INF = the reference's +inf.
    Mirrors the two ComputeDistanceFieldTransformInPlace calls (sdfgen.hpp:76-80)."""
    _capi.require_device(device)
    occ = np.ascontiguousarray(occupancy, dtype=np.float32)
    if occ.ndim != 3:
        raise ValueError("occupancy must be indexed [x, y, z]")
    to_filled = np.empty(occ.shape, dtype=np.int32)
    to_free = np.empty(occ.shape, dtype=np.int32)
    code = _capi.library().vgt_b200_edt_sq_i32(
        occ.ctypes.data, *occ.shape, int(unknown_is_filled), device, to_filled.ctypes.data,
        to_free.ctypes.data)
    _capi.check(code)
    return to_filled, to_free


def ComputeDistanceFieldTransformInPlace(field: np.ndarray, device: int = 0) -> np.ndarray:
    """internal::ComputeDistanceFieldTransformInPlace (signed_distance_field_generation.hpp:34-37)
    on a float64 [x, y, z] field of +inf / non-negative integer samples, in place on the device
    (vgt_b200_edt_transform_inplace_f64). Raises NotImplementedError for samples the exact
    integer passes cannot take; the field is then untouched."""
    _capi.require_device(device)
    if field.dtype != np.float64 or field.ndim != 3 or not field.flags.c_contiguous:
        raise ValueError("field must be a C-contiguous float64 array indexed [x, y, z]")
    code = _capi.library().vgt_b200_edt_transform_inplace_f64(field.ctypes.data, *field.shape,
                                                              device)
    _capi.check(code)
    return field
