"""GPU: the multi-device SDF entries (vgt_b200_sdf_f64_multi, vgt_b200_sdf_from_cells_*_multi,
vgt_b200_sdf_per_object_*_multi, vgt_b200_sdf_free_and_named_*_multi) against their one-device
host entries, byte for byte (fields and min/max), and against the oracle on small grids.

Every comparison runs on 2 devices, on 3 when there are at least 3 (uneven slabs), and on all
visible devices. The multi-device entries need at least two devices; below that every test skips.
"""
import ctypes
import os

import numpy as np
import pytest

import voxelized_geometry_tools_b200 as vgt
from voxelized_geometry_tools_b200 import _capi, grids, synthetic

from .test_gpu_other_maps import params, random_cells, sizes_of

pytestmark = pytest.mark.gpu

RESOLUTION = 0.05
CELL_TYPES = {8: grids.TAGGED_OBJECT_OCCUPANCY_CELL,
              16: grids.TAGGED_OBJECT_OCCUPANCY_COMPONENT_CELL}
MAP_TYPES = {8: vgt.TaggedObjectOccupancyMap, 16: vgt.TaggedObjectOccupancyComponentMap}
SCALARS = {np.float32: ("f32", ctypes.c_float), np.float64: ("f64", ctypes.c_double)}
OBJECT_LISTS = {"empty": [], "listed": [1, 2], "absent": [77], "repeated": [2, 1, 2],
                "with_zero": [0, 3]}


def device_counts():
    import torch
    count = torch.cuda.device_count()
    if count < 2:
        pytest.skip("the multi-device entries need at least 2 devices")
    return sorted({2, count} | ({3} if count >= 3 else set()))


def run(member, cells, objects, unknown, border, dtype, num_devices=None):
    """One call of vgt_b200_<member>_<f32|f64>[_multi]: (fields, minima, maxima). num_devices None:
    the one-device host entry on device 0; otherwise the multi entry on devices 0..n-1."""
    suffix, scalar = SCALARS[dtype]
    lib = _capi.library()
    ids = np.ascontiguousarray(objects, dtype=np.uint32)
    results = ids.size if member == "sdf_per_object" else 1
    out = np.empty((results,) + cells.shape, dtype=dtype)
    lows = np.empty(max(results, 1), dtype=dtype)
    highs = np.empty(max(results, 1), dtype=dtype)
    arguments = [cells.ctypes.data, cells.dtype.itemsize, *cells.shape, RESOLUTION, int(unknown),
                 int(border)]
    if member != "sdf_free_and_named":
        arguments += [ids.ctypes.data if ids.size else None, ids.size]
    if num_devices is None:
        function = getattr(lib, f"vgt_b200_{member}_{suffix}")
        arguments += [0]
    else:
        function = getattr(lib, f"vgt_b200_{member}_{suffix}_multi")
        arguments += [(ctypes.c_int * num_devices)(*range(num_devices)), num_devices]
    pointer = ctypes.POINTER(scalar)
    _capi.check(function(*arguments, out.ctypes.data, lows.ctypes.data_as(pointer),
                         highs.ctypes.data_as(pointer)))
    return out, lows[:results], highs[:results]


def assert_same_bytes(got, want, what):
    for g, w, name in zip(got, want, ("fields", "minima", "maxima")):
        assert g.dtype == w.dtype and g.shape == w.shape, (what, name)
        assert g.tobytes() == w.tobytes(), (what, name)


def compare(member, cells, objects, unknown, border, dtype, oracle=None):
    counts = device_counts()
    want = run(member, cells, objects, unknown, border, dtype)
    for used in counts:
        assert_same_bytes(run(member, cells, objects, unknown, border, dtype, used), want,
                          (member, used, objects))
    if oracle is not None and cells.size < 2 ** 20:
        for k, object_id in enumerate(objects if member == "sdf_per_object" else [None]):
            if member == "sdf_free_and_named":
                field, (lo, hi) = oracle.sdf_free_and_named(cells, RESOLUTION, unknown, border,
                                                            dtype=dtype)
            else:
                listed = objects if object_id is None else [object_id]
                field, (lo, hi) = oracle.sdf_from_cells(cells, RESOLUTION, unknown, border,
                                                        listed, dtype=dtype)
            np.testing.assert_array_equal(want[0][k], field)
            assert (want[1][k], want[2][k]) == (lo, hi)
    return want


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("cell_bytes", [8, 16])
@pytest.mark.parametrize("unknown,border", [(True, False), (False, True)])
def test_single_and_free_and_named_equal_the_host_entries(shared_library, oracle, dtype,
                                                          cell_bytes, unknown, border):
    # nx, ny: multiples of neither 2 nor 3
    rng = np.random.default_rng(11 + cell_bytes)
    cells = random_cells(rng, (23, 31, 40), CELL_TYPES[cell_bytes])
    for objects in OBJECT_LISTS.values():
        compare("sdf_from_cells", cells, objects, unknown, border, dtype, oracle)
    compare("sdf_free_and_named", cells, [], unknown, border, dtype, oracle)
    compare("sdf_per_object", cells, [4, 1, 9, 4, 0, 2], unknown, border, dtype, oracle)


@pytest.mark.parametrize("nz", [127, 128, 1024, 2048])
def test_every_z_scan_route_under_the_slab_driver(shared_library, oracle, nz):
    # ny = the number of visible devices: one row per part when all of them are used
    import torch
    counts = device_counts()
    rng = np.random.default_rng(nz)
    cell_bytes = 16 if nz in (128, 2048) else 8
    dtype = np.float64 if nz == 1024 else np.float32
    cells = random_cells(rng, (9, torch.cuda.device_count(), nz), CELL_TYPES[cell_bytes])
    ids = [4, 1, 9, 4, 0, 2]   # a repeat, an id absent from the map, id 0
    assert max(counts) == cells.shape[1]
    compare("sdf_per_object", cells, ids, nz != 128, nz in (127, 2048), dtype, oracle)
    compare("sdf_from_cells", cells, [1, 4], nz == 128, nz == 1024, dtype, oracle)
    compare("sdf_free_and_named", cells, [], nz != 1024, nz == 128, dtype, oracle)


def test_batch_of_300_distinct_ids_takes_two_slot_groups(shared_library, oracle):
    rng = np.random.default_rng(300)
    shape = (12, 10, 16)
    cells = random_cells(rng, shape, CELL_TYPES[16])
    cells["occupancy"] = np.where(rng.random(shape) < 0.6, 1.0, 0.0)
    cells["object_id"] = rng.integers(0, 302, shape, dtype=np.uint32)
    ids = rng.permutation(np.arange(1, 301, dtype=np.uint32))  # 300 distinct: two slot groups
    fields, lows, highs = compare("sdf_per_object", cells, ids, True, False, np.float32)
    # sorted positions 253, 254 (the last two of group 0) and 255, 256 (the first of group 1)
    for position in (253, 254, 255, 256):
        k = int(np.flatnonzero(ids == position + 1)[0])
        field, (lo, hi) = oracle.sdf_from_cells(cells, RESOLUTION, True, False, [ids[k]])
        np.testing.assert_array_equal(fields[k], field)
        assert (lows[k], highs[k]) == (lo, hi)


def test_empty_batch(shared_library):
    rng = np.random.default_rng(5)
    cells = random_cells(rng, (8, 8, 8), CELL_TYPES[8])
    before = int(_capi.library().vgt_b200_kernel_launch_count())
    for used in device_counts():
        fields, _, _ = run("sdf_per_object", cells, [], True, False, np.float32, used)
        assert fields.shape[0] == 0
    assert int(_capi.library().vgt_b200_kernel_launch_count()) == before


def test_double_occupancy_entry_equals_one_device(shared_library, oracle):
    # the scenes of test_gpu_sharded.py::test_single_process_multi_device_entry
    counts = device_counts()
    for dims, border in (((40, 36, 44), False), ((61, 45, 130), True), ((256, 192, 160), False)):
        occupancy = synthetic.clustered_spheres_occupancy(dims)
        grid = vgt.OccupancyMap(np.eye(4), "world", vgt.VoxelGridSizes.FromVoxelCounts(0.02, dims),
                                data=occupancy)
        parameters = vgt.SignedDistanceFieldGenerationParameters(add_virtual_border=border)
        single = grid.ExtractSignedDistanceFieldDouble(parameters)
        for used in counts:
            multi = grid.ExtractSignedDistanceFieldDouble(parameters, devices=list(range(used)))
            assert multi.GetImmutableRawData().dtype == np.float64
            assert multi.GetImmutableRawData().tobytes() == single.GetImmutableRawData().tobytes()
            assert multi.GetMinimumMaximum() == single.GetMinimumMaximum()
        if np.prod(dims) < 2 ** 20:
            want, _ = oracle.sdf(occupancy, 0.02, add_virtual_border=border, dtype=np.float64)
            np.testing.assert_array_equal(multi.GetImmutableRawData(), want)
    with pytest.raises(ValueError):
        grid.ExtractSignedDistanceFieldDouble(parameters, devices=[0, 0])


def test_python_members_on_several_devices(shared_library):
    used = list(range(max(device_counts())))
    rng = np.random.default_rng(21)
    parameters = params(True, True)
    for cell_bytes, map_type in MAP_TYPES.items():
        cells = random_cells(rng, (19, 14, 33), CELL_TYPES[cell_bytes])
        grid = map_type(np.eye(4), "world", sizes_of(cells.shape, RESOLUTION), data=cells)
        pairs = [
            (grid.ExtractSignedDistanceFieldFloat([1, 3], parameters),
             grid.ExtractSignedDistanceFieldFloat([1, 3], parameters, devices=used)),
            (grid.ExtractSignedDistanceFieldDouble([], parameters),
             grid.ExtractSignedDistanceFieldDouble([], parameters, devices=used)),
            (grid.ExtractFreeAndNamedObjectsSignedDistanceField(parameters, np.float64),
             grid.ExtractFreeAndNamedObjectsSignedDistanceField(parameters, np.float64,
                                                                devices=used)),
            # one entry is that device
            (grid.ExtractSignedDistanceFieldFloat([2], parameters, device=1),
             grid.ExtractSignedDistanceFieldFloat([2], parameters, devices=[1])),
        ]
        separate = grid.MakeAllObjectSDFs(parameters)
        separate_multi = grid.MakeAllObjectSDFs(parameters, devices=used)
        assert sorted(separate) == sorted(separate_multi) and separate
        pairs += [(separate[k], separate_multi[k]) for k in separate]
        for single, multi in pairs:
            assert multi.GetImmutableRawData().tobytes() == single.GetImmutableRawData().tobytes()
            assert multi.GetMinimumMaximum() == single.GetMinimumMaximum()
        with pytest.raises(ValueError):
            grid.MakeSeparateObjectSDFs([1], parameters, devices=[0, 0])
    component = vgt.OccupancyComponentMap(
        np.eye(4), "world", sizes_of((19, 14, 33), RESOLUTION),
        data=random_cells(rng, (19, 14, 33), grids.OCCUPANCY_COMPONENT_CELL))
    single = component.ExtractSignedDistanceFieldFloat(parameters)
    multi = component.ExtractSignedDistanceFieldFloat(parameters, devices=used)
    assert multi.GetImmutableRawData().tobytes() == single.GetImmutableRawData().tobytes()
    assert multi.GetMinimumMaximum() == single.GetMinimumMaximum()
    with pytest.raises(ValueError):
        component.ExtractSignedDistanceFieldDouble(parameters, devices=[1, 1])


# ------------------------------------------------------------------------------------------------
# The case the entries exist for: a 2048^3 TaggedObjectOccupancyComponentMap on 8 devices
# ------------------------------------------------------------------------------------------------
BIG = 2048


def one_device_bytes(nx, ny, nz, cell_bytes, scalar_bytes):
    """Device memory of vgt_b200_sdf_from_cells_* on one device (SdfFromCellsHost): the cells,
    the 1-byte mask, the SDF and the 4-byte scratch of the passes."""
    voxels = nx * ny * nz
    return voxels * (cell_bytes + 1 + scalar_bytes + 4)


def host_memory_bytes():
    return os.sysconf("SC_PAGE_SIZE") * os.sysconf("SC_PHYS_PAGES")


def test_2048_cubed_component_map_on_eight_devices(shared_library):
    import torch
    if torch.cuda.device_count() < 8:
        pytest.skip("needs 8 devices")
    # the one-device call cannot run: it is not attempted
    assert one_device_bytes(BIG, BIG, BIG, 16, 4) > torch.cuda.get_device_properties(0).total_memory
    # peak: the cells (137.4 GB), the reference SDF and the cell-map SDF (34.4 each)
    needed = BIG ** 3 * (16 + 4 + 4)
    if host_memory_bytes() < needed * 1.1:
        pytest.skip(f"needs about {needed / 1e9:.0f} GB of host memory, the host has "
                    f"{host_memory_bytes() / 1e9:.0f} GB")
    devices = list(range(8))
    subset = [2, 5]
    shape = (BIG, BIG, BIG)
    sizes = sizes_of(shape, 0.01)
    parameters = params(True, False)
    step = 256

    def slab(x0):
        """occupancy and object ids of x-planes [x0, x0 + step): clustered spheres, objects in
        blocks of 256^3 with ids 0..6 (0 = unnamed)"""
        occupancy = synthetic.clustered_spheres_occupancy_torch(
            shape, "cuda:0", x_range=(x0, x0 + step)).cpu().numpy()
        y = np.arange(BIG, dtype=np.uint32)[:, None] // 256
        z = np.arange(BIG, dtype=np.uint32)[None, :] // 256
        return occupancy, ((x0 // 256) * 3 + y * 5 + z).astype(np.uint32) % 7

    # the float occupancy the predicate gives: 1.0 where filled and listed, else 0.0
    reference = np.empty(shape, dtype=np.float32)
    for x0 in range(0, BIG, step):
        occupancy, ids = slab(x0)
        filled = (occupancy >= np.float32(0.5)) & np.isin(ids, subset)[None]
        reference[x0:x0 + step] = np.where(filled, np.float32(1.0), np.float32(0.0))
    want = vgt.OccupancyMap(np.eye(4), "world", sizes, data=reference) \
        .ExtractSignedDistanceFieldFloat(parameters, devices=devices)
    del reference
    cells = np.zeros(shape, dtype=CELL_TYPES[16])
    for x0 in range(0, BIG, step):
        occupancy, ids = slab(x0)
        cells["occupancy"][x0:x0 + step] = occupancy
        cells["object_id"][x0:x0 + step] = ids[None]
    grid = vgt.TaggedObjectOccupancyComponentMap(np.eye(4), "world", sizes, data=cells)
    got = grid.ExtractSignedDistanceFieldFloat(subset, parameters, devices=devices)
    assert got.GetMinimumMaximum() == want.GetMinimumMaximum()
    for x0 in range(0, BIG, step):
        assert got.GetImmutableRawData()[x0:x0 + step].tobytes() \
            == want.GetImmutableRawData()[x0:x0 + step].tobytes(), x0
