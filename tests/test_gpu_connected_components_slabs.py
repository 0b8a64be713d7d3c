"""GPU: connected components of the component maps cut into x-slabs
(vgt_b200_connected_components_multi, UpdateConnectedComponents(devices=...)) against the
one-device entry, byte for byte: one device listed several times, distinct devices, and a map of
more than 2^32 cells checked plane by plane against its closed-form labelling."""
import ctypes
import os
import zlib

import numpy as np
import pytest

from tests import components, slab_scenes
from tests.conftest import random_occupancy

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def vgt(shared_library):
    import voxelized_geometry_tools_b200 as module
    return module


def make_map(vgt, cells):
    sizes = vgt.VoxelGridSizes.FromVoxelCounts(0.1, cells.shape)
    cls = vgt.OccupancyComponentMap if cells.dtype.itemsize == 8 \
        else vgt.TaggedObjectOccupancyComponentMap
    return cls(np.eye(4), "world", sizes, data=cells.copy())


def label(vgt, cells, devices=None):
    grid = make_map(vgt, cells)
    count = grid.UpdateConnectedComponents() if devices is None \
        else grid.UpdateConnectedComponents(devices=devices)
    return grid.GetImmutableRawData(), count


def check_equals_one_device(vgt, cells, devices):
    want, want_count = label(vgt, cells)
    got, count = label(vgt, cells, devices)
    assert count == want_count, devices
    assert got.tobytes() == want.tobytes(), devices
    return got, count


def scene(name, shape, rng):
    if name == "free":
        return np.zeros(shape, dtype=np.float32)
    if name == "checkerboard":
        return components.checkerboard(shape)
    if name == "noise30":
        return random_occupancy(rng, shape, 0.3)
    if name == "noise50":
        return random_occupancy(rng, shape, 0.5)
    if name == "blobs":
        return random_occupancy(rng, shape, 0.4, blobs=True)
    if name == "serpentine":
        return components.serpentine(shape)
    if name == "x_serpentine":
        return slab_scenes.x_serpentine(shape)
    if name == "shells":
        return components.nested_shells(shape)
    return components.special_values(rng, shape)


SCENES = ["free", "checkerboard", "noise30", "noise50", "blobs", "serpentine", "x_serpentine",
          "shells", "special"]


def shapes_for(slabs):
    # nx = slabs (one-plane slabs), nx = slabs + 1, ny = 1, nz = 1, odd sizes
    return [(slabs, 5, 7), (slabs + 1, 3, 9), (2 * slabs + 1, 1, 13), (3 * slabs, 11, 1),
            (17, 13, 11), (33, 9, 65)]


@pytest.mark.parametrize("tagged", [False, True], ids=["8B", "16B"])
@pytest.mark.parametrize("name", SCENES)
@pytest.mark.parametrize("slabs", [2, 3, 4, 8])
def test_one_device_listed_repeatedly_equals_one_device(vgt, slabs, name, tagged):
    for shape in shapes_for(slabs):
        rng = np.random.default_rng(zlib.crc32(repr((slabs, shape, name, tagged)).encode()))
        object_id = rng.integers(0, 3, shape, dtype=np.uint32) if tagged else None
        cells = components.make_cells(scene(name, shape, rng), object_id, rng)
        got, count = check_equals_one_device(vgt, cells, [0] * slabs)
        if name == "free" and not tagged:
            assert count == 1
        if name == "checkerboard" and not tagged:
            assert count == cells.size


@pytest.mark.parametrize("slabs", [2, 3, 8])
@pytest.mark.parametrize("tagged", [False, True], ids=["8B", "16B"])
def test_512_cubed_on_one_device_listed_repeatedly(vgt, slabs, tagged):
    rng = np.random.default_rng(512 + slabs + 16 * tagged)
    shape = (512, 512, 512)
    object_id = (rng.random(shape) < 0.2).astype(np.uint32) if tagged else None
    cells = components.make_cells(random_occupancy(rng, shape, 0.3), object_id, rng)
    check_equals_one_device(vgt, cells, [0] * slabs)


def test_ring_whose_halves_in_slab_0_meet_only_in_slab_2(vgt):
    shape = (9, 8, 6)
    occupancy = slab_scenes.ring_closed_in_slab(shape, 7)  # slabs [0, 3) [3, 6) [6, 9)
    cells = components.make_cells(occupancy, None, np.random.default_rng(1))
    got, count = check_equals_one_device(vgt, cells, [0, 0, 0])
    assert count == 2
    assert got["component"][0, 0, 1] == got["component"][0, 7, 1] == 2
    want, want_count = components.scipy_components(cells)
    np.testing.assert_array_equal(got["component"], want)


def test_components_whose_smallest_index_lies_in_the_last_slab(vgt):
    shape = (12, 9, 10)
    cells = components.make_cells(slab_scenes.last_slab_components(shape, 9), None,
                                  np.random.default_rng(2))
    for slabs in (2, 3, 4):
        got, count = check_equals_one_device(vgt, cells, [0] * slabs)
        want, want_count = components.scipy_components(cells)
        assert count == want_count
        np.testing.assert_array_equal(got["component"], want)


def test_serpentine_crossing_every_face(vgt):
    shape = (40, 63, 5)
    cells = components.make_cells(slab_scenes.x_serpentine(shape), np.zeros(shape, np.uint32),
                                  np.random.default_rng(3))
    for slabs in (2, 5, 8):
        got, count = check_equals_one_device(vgt, cells, [0] * slabs)
        assert count == 2


# ---- distinct devices ---------------------------------------------------------------------------
def device_lists(count):
    lists = [[0, 1], list(range(count)), [0, 1, 0, 1]]
    return [devices for k, devices in enumerate(lists) if devices not in lists[:k]]


@pytest.mark.parametrize("n", [512, 1024])
def test_distinct_devices_equal_one_device(vgt, n):
    from voxelized_geometry_tools_b200 import _capi, synthetic
    count = _capi.device_count()
    if count < 2:
        pytest.skip(f"{count} device(s): distinct devices need 2 or more")
    cells = components.make_cells(synthetic.clustered_spheres_occupancy((n, n, n)))
    want, want_count = label(vgt, cells)
    for devices in device_lists(min(count, 8)):
        got, got_count = label(vgt, cells, devices)
        assert got_count == want_count, devices
        assert got.tobytes() == want.tobytes(), devices
        del got


# ---- more than 2^32 cells -----------------------------------------------------------------------
BIG = (4096, 1024, 1025)  # 4 299 161 600 cells, 2 149 580 800 per slab of two
WALLS = (300, 700)
BAR = dict(y=10, x=(2040, 2056))      # joins the two walls, across the slab face at x = 2048
U = dict(z=900, y=(100, 200), x=(100, 3000))  # two arms from slab 0 closed at x = 3000


def require_big_memory():
    host = os.sysconf("SC_PAGE_SIZE") * os.sysconf("SC_PHYS_PAGES")
    if host < 100e9:
        pytest.skip(f"host RAM {host / 1e9:.0f} GB < 100 GB (the map alone is 34 GB)")
    import torch
    device = torch.cuda.get_device_properties(0).total_memory
    if device < 100e9:
        pytest.skip(f"device memory {device / 1e9:.0f} GB < 100 GB (two 2^31-cell slabs)")


def big_scene_plane(x):
    """The occupancy of plane x and its closed-form labelling: free z < 300 (1), the walls
    z = 300 / 700 and the bar (2), free between the walls (3), free above (4), the U (5)."""
    nx, ny, nz = BIG
    z = np.arange(nz)
    ids = np.where(z < WALLS[0], 1, np.where(z < WALLS[1], 3, 4)).astype(np.uint32)
    ids[list(WALLS)] = 2
    ids = np.broadcast_to(ids, (ny, nz)).copy()
    if BAR["x"][0] <= x < BAR["x"][1]:
        ids[BAR["y"], WALLS[0]:WALLS[1] + 1] = 2
    y0, y1 = U["y"]
    x0, x1 = U["x"]
    if x0 <= x <= x1:
        ids[[y0, y1], U["z"]] = 5
    if x == x1:
        ids[y0:y1 + 1, U["z"]] = 5
    occupancy = np.isin(ids, (2, 5)).astype(np.float32)
    return occupancy, ids


def multi(cells, devices):
    from voxelized_geometry_tools_b200 import _capi
    count = ctypes.c_uint32(0)
    listed = (ctypes.c_int * len(devices))(*devices)
    code = _capi.library().vgt_b200_connected_components_multi(
        cells.ctypes.data, cells.dtype.itemsize, *cells.shape, listed, len(devices),
        ctypes.byref(count))
    return code, int(count.value)


def test_more_than_2_32_cells(vgt):
    require_big_memory()
    from voxelized_geometry_tools_b200 import _capi
    cells = np.empty(BIG, dtype=components.OCCUPANCY_COMPONENT_CELL)
    sentinel = np.uint32(0xDEADBEEF)
    for x in range(BIG[0]):
        cells["occupancy"][x] = big_scene_plane(x)[0]
        cells["component"][x] = sentinel

    # the one-device entry refuses it and leaves the cells as they were
    count = ctypes.c_uint32(0)
    code = _capi.library().vgt_b200_connected_components(
        cells.ctypes.data, 8, *BIG, 0, ctypes.byref(count))
    assert code == _capi.ERR_UNSUPPORTED
    assert "2^32" in _capi.last_error()
    assert all((cells["component"][x] == sentinel).all() for x in range(0, BIG[0], 64))

    lists = [[0, 0]] + ([[0, 1]] if _capi.device_count() >= 2 else [])
    for devices in lists:
        cells["component"] = sentinel
        code, count = multi(cells, devices)
        assert code == _capi.OK, _capi.last_error()
        assert count == 5, devices
        for x in range(BIG[0]):
            occupancy, ids = big_scene_plane(x)
            np.testing.assert_array_equal(cells["component"][x], ids, err_msg=f"{devices} x={x}")
            np.testing.assert_array_equal(cells["occupancy"][x], occupancy)


def test_more_than_0xffffffff_components_are_refused(vgt):
    require_big_memory()
    from voxelized_geometry_tools_b200 import _capi
    cells = np.empty(BIG, dtype=components.OCCUPANCY_COMPONENT_CELL)
    y, z = np.indices(BIG[1:])
    sentinel = np.uint32(0x12345678)
    for x in range(BIG[0]):
        cells["occupancy"][x] = ((x + y + z) % 2).astype(np.float32)
        cells["component"][x] = sentinel
    code, _ = multi(cells, [0, 0])
    assert code == _capi.ERR_UNSUPPORTED
    assert "0xFFFFFFFF" in _capi.last_error() or "32-bit" in _capi.last_error()
    for x in range(BIG[0]):
        assert (cells["component"][x] == sentinel).all(), x
