"""CPU: the multi-device SDF entries (vgt_b200_sdf_f64_multi, vgt_b200_sdf_from_cells_*_multi,
vgt_b200_sdf_per_object_*_multi, vgt_b200_sdf_free_and_named_*_multi) refuse bad arguments before
they touch a device, and with good arguments and no device they fail instead of computing
anything on the CPU. The Python devices= arguments raise as OccupancyMap's float path does."""
import ctypes

import numpy as np
import pytest

import voxelized_geometry_tools_b200 as vgt
from voxelized_geometry_tools_b200 import _capi, grids

IDS = np.array([3, 1, 3], dtype=np.uint32)
CELLS = np.zeros(4 * 5 * 6 * 4, dtype=np.uint32)   # big enough for 16-byte cells
OUT = np.zeros(4 * 5 * 6 * 3, dtype=np.float64)    # room for the three SDFs of IDS
MIN_MAX = np.zeros(3, dtype=np.float64)


def device_list(*ordinals):
    return (ctypes.c_int * max(len(ordinals), 1))(*ordinals)


def entries(suffix):
    lib = _capi.library()

    def occupancy(cells, cell_bytes, dims, resolution, ids, num_ids, devices, num_devices, out):
        if suffix != "f64":
            return None   # vgt_b200_sdf_f32_multi predates these entries; not covered here
        return lib.vgt_b200_sdf_f64_multi(cells, *dims, resolution, 1, 0, devices, num_devices,
                                          out, None, None)

    def from_cells(cells, cell_bytes, dims, resolution, ids, num_ids, devices, num_devices, out):
        return getattr(lib, f"vgt_b200_sdf_from_cells_{suffix}_multi")(
            cells, cell_bytes, *dims, resolution, 1, 0, ids, num_ids, devices, num_devices, out,
            None, None)

    def per_object(cells, cell_bytes, dims, resolution, ids, num_ids, devices, num_devices, out):
        return getattr(lib, f"vgt_b200_sdf_per_object_{suffix}_multi")(
            cells, cell_bytes, *dims, resolution, 1, 0, ids, num_ids, devices, num_devices, out,
            MIN_MAX.ctypes.data, MIN_MAX.ctypes.data)

    def free_and_named(cells, cell_bytes, dims, resolution, ids, num_ids, devices, num_devices,
                       out):
        return getattr(lib, f"vgt_b200_sdf_free_and_named_{suffix}_multi")(
            cells, cell_bytes, *dims, resolution, 1, 0, devices, num_devices, out, None, None)

    return {"occupancy": occupancy, "from_cells": from_cells, "per_object": per_object,
            "free_and_named": free_and_named}


GOOD = dict(cells=CELLS.ctypes.data, cell_bytes=8, dims=(4, 5, 6), resolution=0.1,
            ids=IDS.ctypes.data, num_ids=IDS.size, devices=device_list(0, 1), num_devices=2,
            out=OUT.ctypes.data)

# (what, changed arguments, message fragment, entries that take the argument)
ALL = ("occupancy", "from_cells", "per_object", "free_and_named")
CELL_ENTRIES = ("from_cells", "per_object", "free_and_named")
LISTS = ("from_cells", "per_object")
REFUSALS = [
    ("null device list", dict(devices=None), "devices are supported", ALL),
    ("no device", dict(num_devices=0), "devices are supported", ALL),
    ("nine devices", dict(devices=device_list(*range(9)), num_devices=9), "devices are supported",
     ALL),
    ("repeated device", dict(devices=device_list(1, 1)), "listed twice", ALL),
    ("negative device", dict(devices=device_list(0, -1)), "out of range", ALL),
    ("device beyond the cache", dict(devices=device_list(0, 64)), "out of range", ALL),
    ("more devices than nx", dict(dims=(2, 5, 6), devices=device_list(0, 1, 2), num_devices=3),
     "more devices than voxels", ALL),
    ("more devices than ny", dict(dims=(4, 2, 6), devices=device_list(0, 1, 2), num_devices=3),
     "more devices than voxels", ALL),
    ("null cells", dict(cells=None), "null", ALL),
    ("null output", dict(out=None), "null", ALL),
    ("cell size", dict(cell_bytes=12), "cell size", CELL_ENTRIES),
    ("cell size 4", dict(cell_bytes=4), "cell size", CELL_ENTRIES),
    ("empty axis", dict(dims=(4, 0, 6)), "out of range", ALL),
    ("long axis", dict(dims=(4, 5, 8193)), "out of range", ALL),
    ("zero resolution", dict(resolution=0.0), "resolution", ALL),
    ("nan resolution", dict(resolution=float("nan")), "resolution", ALL),
    ("negative id count", dict(num_ids=-1), "object id list", LISTS),
    ("ids missing", dict(ids=None), "object id list", LISTS),
    ("too many ids", dict(num_ids=2 ** 31), "object id list", LISTS),
]


def launch_count():
    return int(_capi.library().vgt_b200_kernel_launch_count())


@pytest.mark.parametrize("suffix", ["f32", "f64"])
@pytest.mark.parametrize("what,changed,fragment,takers", REFUSALS, ids=[r[0] for r in REFUSALS])
def test_bad_arguments_are_refused_before_any_device_call(shared_library, suffix, what, changed,
                                                          fragment, takers):
    arguments = dict(GOOD, **changed)
    before = launch_count()
    checked = 0
    for name, entry in entries(suffix).items():
        if name not in takers:
            continue
        code = entry(**arguments)
        if code is None:
            continue
        checked += 1
        assert code == _capi.ERR_INVALID_ARGUMENT, (name, code, _capi.last_error())
        assert fragment in _capi.last_error(), (name, _capi.last_error())
    assert checked > 0
    assert launch_count() == before


@pytest.mark.parametrize("suffix,scalar_bytes", [("f32", 4), ("f64", 8)])
def test_batch_refuses_a_byte_count_beyond_int64(shared_library, suffix, scalar_bytes):
    # 8192^3 voxels: the largest batch whose bytes fit int64 has (2^63 - 1) // (2^39 * T) SDFs
    per_object = entries(suffix)["per_object"]
    largest = (2 ** 63 - 1) // (2 ** 39 * scalar_bytes)
    arguments = dict(GOOD, dims=(8192, 8192, 8192))
    before = launch_count()
    assert per_object(**dict(arguments, num_ids=largest + 1)) == _capi.ERR_INVALID_ARGUMENT
    assert "overflow" in _capi.last_error()
    assert launch_count() == before
    if _capi.device_count() > 0:
        pytest.skip("a GPU is present: the batch that fits would run")
    # one SDF fewer passes every check and stops at the missing device (the ids are only read
    # after that)
    assert per_object(**dict(arguments, num_ids=largest)) == _capi.ERR_DEVICE


@pytest.mark.parametrize("suffix", ["f32", "f64"])
@pytest.mark.parametrize("num_devices", [1, 2])
def test_no_cpu_fallback_without_device(shared_library, suffix, num_devices):
    if _capi.device_count() > 0:
        pytest.skip("a GPU is present")
    arguments = dict(GOOD, devices=device_list(*range(num_devices)), num_devices=num_devices)
    for name, entry in entries(suffix).items():
        code = entry(**arguments)
        if code is None:
            continue
        assert code == _capi.ERR_DEVICE, (name, _capi.last_error())
        assert "Cuda error" in _capi.last_error(), name
    # an empty batch launches nothing, but it still needs the devices it was asked to use
    assert entries(suffix)["per_object"](**dict(arguments, ids=None, num_ids=0)) \
        == _capi.ERR_DEVICE


def maps():
    sizes = vgt.VoxelGridSizes.FromVoxelCounts(0.1, (4, 5, 6))
    return (vgt.OccupancyMap(np.eye(4), "f", sizes),
            vgt.OccupancyComponentMap(np.eye(4), "f", sizes),
            vgt.TaggedObjectOccupancyMap(np.eye(4), "f", sizes),
            vgt.TaggedObjectOccupancyComponentMap(np.eye(4), "f", sizes))


def member_calls(devices):
    parameters = vgt.SignedDistanceFieldGenerationParameters()
    occupancy_map, component_map, tagged, tagged_component = maps()
    calls = [
        lambda: occupancy_map.ExtractSignedDistanceFieldFloat(parameters, devices=devices),
        lambda: occupancy_map.ExtractSignedDistanceFieldDouble(parameters, devices=devices),
        lambda: occupancy_map.ExtractSignedDistanceField(parameters, np.float64, devices=devices),
        lambda: component_map.ExtractSignedDistanceFieldFloat(parameters, devices=devices),
        lambda: component_map.ExtractSignedDistanceFieldDouble(parameters, devices=devices),
    ]
    for grid in (tagged, tagged_component):
        calls += [
            lambda grid=grid: grid.ExtractSignedDistanceFieldFloat([1], parameters,
                                                                   devices=devices),
            lambda grid=grid: grid.ExtractSignedDistanceFieldDouble([], parameters,
                                                                    devices=devices),
            lambda grid=grid: grid.MakeSeparateObjectSDFs([1, 2], parameters, np.float64,
                                                          devices=devices),
            lambda grid=grid: grid.MakeAllObjectSDFs(parameters, devices=devices),
            lambda grid=grid: grid.ExtractFreeAndNamedObjectsSignedDistanceField(
                parameters, devices=devices),
        ]
    return calls


@pytest.mark.parametrize("devices", [[0], [0, 1], [0, 0], (0, 1, 2, 3, 4, 5, 6, 7)])
def test_python_devices_argument_raises_without_a_device(shared_library, devices):
    if _capi.device_count() > 0:
        pytest.skip("a GPU is present")
    for call in member_calls(devices):
        with pytest.raises(_capi.BackendUnavailable):
            call()


def test_python_members_take_devices():
    # every SDF member of the four map types has the devices= argument (the component map
    # inherits the tagged map's members)
    import inspect
    members = {
        vgt.OccupancyMap: ("ExtractSignedDistanceField", "ExtractSignedDistanceFieldFloat",
                           "ExtractSignedDistanceFieldDouble"),
        vgt.OccupancyComponentMap: ("ExtractSignedDistanceField",
                                    "ExtractSignedDistanceFieldFloat",
                                    "ExtractSignedDistanceFieldDouble"),
        vgt.TaggedObjectOccupancyMap: ("ExtractSignedDistanceField",
                                       "ExtractSignedDistanceFieldFloat",
                                       "ExtractSignedDistanceFieldDouble",
                                       "MakeSeparateObjectSDFs", "MakeAllObjectSDFs",
                                       "ExtractFreeAndNamedObjectsSignedDistanceField"),
    }
    members[vgt.TaggedObjectOccupancyComponentMap] = members[vgt.TaggedObjectOccupancyMap]
    for cls, names in members.items():
        for name in names:
            parameter = inspect.signature(getattr(cls, name)).parameters.get("devices")
            assert parameter is not None and parameter.default is None, (cls, name)
    assert issubclass(vgt.TaggedObjectOccupancyComponentMap, grids.TaggedObjectOccupancyMap)
