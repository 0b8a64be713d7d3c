"""CPU: the connected-component labelling of the component maps (ComputeConnectedComponents,
topology_computation.hpp:138-196). Three independent statements of it agree: the reference's scan
and breadth-first fill restated in oracle/components_oracle.cpp, a numpy model of the device's
union-find (run-start init, min-linking unions in a shuffled order, flatten, rank of the roots) and
scipy.ndimage.label renumbered by first occurrence; plus hand cases and the C-ABI's refusals."""
import ctypes

import numpy as np
import pytest

from tests import components
from tests.conftest import random_occupancy


@pytest.fixture(scope="module")
def cc_oracle():
    """The restated reference (oracle/components_oracle.py), built for this host if needed."""
    from oracle import components_oracle
    components_oracle.build()
    return components_oracle


def random_cells(rng, shape, tagged):
    scene = rng.integers(0, 4)
    if scene == 0:
        occupancy = random_occupancy(rng, shape, rng.choice([0.2, 0.5, 0.8]))
    elif scene == 1:
        occupancy = random_occupancy(rng, shape, 0.4, blobs=True)
    elif scene == 2:
        occupancy = components.special_values(rng, shape)
    else:
        occupancy = components.checkerboard(shape) if rng.random() < 0.5 \
            else components.serpentine(shape)
    object_id = rng.integers(0, 3, shape, dtype=np.uint32) if tagged else None
    return components.make_cells(occupancy, object_id, rng)


SHAPES = [(1, 1, 1), (1, 1, 9), (1, 7, 1), (6, 1, 1), (3, 4, 5), (5, 5, 5), (2, 9, 13),
          (7, 3, 33), (4, 6, 17)]


@pytest.mark.parametrize("tagged", [False, True])
@pytest.mark.parametrize("seed", range(6))
def test_model_equals_the_restated_reference_and_scipy(cc_oracle, tagged, seed):
    rng = np.random.default_rng(1000 * seed + tagged)
    for shape in SHAPES:
        cells = random_cells(rng, shape, tagged)
        want, want_count = cc_oracle.connected_components(cells)
        for tile in (4, 8, 32):
            ids, count = components.model_components(cells, rng, tile)
            assert count == want_count, (shape, tile)
            np.testing.assert_array_equal(ids, want["component"], err_msg=f"{shape} {tile}")
        ids, count = components.scipy_components(cells)
        assert count == want_count, shape
        np.testing.assert_array_equal(ids, want["component"])
        # the oracle writes only the component word
        for name in cells.dtype.names:
            if name != "component":
                np.testing.assert_array_equal(want[name].view(np.uint32),
                                              cells[name].view(np.uint32))


def test_hand_case_a_row(cc_oracle):
    cells = components.make_cells(np.array([1.0, 0.0, 0.5, 1.0], dtype=np.float32).reshape(1, 1, 4))
    labelled, count = cc_oracle.connected_components(cells)
    assert count == 3
    assert labelled["component"].reshape(-1).tolist() == [1, 2, 2, 3]
    ids, count = components.model_components(cells, np.random.default_rng(0), 2)
    assert count == 3 and ids.reshape(-1).tolist() == [1, 2, 2, 3]


def test_hand_case_shell_cavity_core(cc_oracle):
    occupancy = np.ones((7, 7, 7), dtype=np.float32)
    occupancy[1:6, 1:6, 1:6] = 0.0
    occupancy[3, 3, 3] = 1.0
    labelled, count = cc_oracle.connected_components(components.make_cells(occupancy))
    assert count == 3
    component = labelled["component"]
    assert component[0, 0, 0] == 1 and component[6, 6, 6] == 1
    assert component[1, 1, 1] == 2 and component[5, 5, 5] == 2
    assert component[3, 3, 3] == 3
    assert np.unique(component).tolist() == [1, 2, 3]


def test_hand_case_special_occupancies(cc_oracle):
    # 0.5, NaN and -0.0 join the free cells; the float after 0.5 and +inf are filled
    row = np.array([0.5, np.nan, -0.0, 0.0, np.nextafter(np.float32(0.5), np.float32(1)), np.inf,
                    -np.inf, 0.75], dtype=np.float32)
    labelled, count = cc_oracle.connected_components(components.make_cells(row.reshape(1, 1, -1)))
    assert labelled["component"].reshape(-1).tolist() == [1, 1, 1, 1, 2, 2, 3, 4]
    assert count == 4


def test_hand_case_object_ids(cc_oracle):
    occupancy = np.array([1.0, 1.0, 1.0, 0.0, 0.0], dtype=np.float32).reshape(1, 1, 5)
    object_id = np.array([4, 4, 5, 5, 5], dtype=np.uint32).reshape(1, 1, 5)
    labelled, count = cc_oracle.connected_components(components.make_cells(occupancy, object_id))
    # equal ids across the 0.5 boundary are not connected; neither are different ids
    assert labelled["component"].reshape(-1).tolist() == [1, 1, 2, 3, 3]
    assert count == 3


def test_renumbering_helper():
    labels = np.array([7, 7, 3, 9, 3, 7, 1]).reshape(1, 1, 7)
    ids, count = components.renumber_by_first_occurrence(labels)
    assert count == 4
    assert ids.reshape(-1).tolist() == [1, 1, 2, 3, 2, 1, 4]


# ---- the product surface without a device -----------------------------------------------------
def test_methods_exist_only_on_the_component_maps():
    import voxelized_geometry_tools_b200 as vgt
    assert hasattr(vgt.OccupancyComponentMap, "UpdateConnectedComponents")
    assert hasattr(vgt.TaggedObjectOccupancyComponentMap, "UpdateConnectedComponents")
    assert not hasattr(vgt.TaggedObjectOccupancyMap, "UpdateConnectedComponents")
    assert not hasattr(vgt.OccupancyMap, "UpdateConnectedComponents")


def test_no_cpu_fallback_without_device(shared_library):
    import voxelized_geometry_tools_b200 as vgt
    from voxelized_geometry_tools_b200 import _capi
    if _capi.device_count() > 0:
        pytest.skip("a GPU is present")
    sizes = vgt.VoxelGridSizes.FromVoxelCounts(0.1, (3, 4, 5))
    for cls in (vgt.OccupancyComponentMap, vgt.TaggedObjectOccupancyComponentMap):
        grid = cls(np.eye(4), "world", sizes)
        before = grid.GetImmutableRawData().copy()
        with pytest.raises(vgt.BackendUnavailable):
            grid.UpdateConnectedComponents()
        np.testing.assert_array_equal(grid.GetImmutableRawData(), before)
        count = ctypes.c_uint32(7)
        code = _capi.library().vgt_b200_connected_components(
            grid.GetMutableRawData().ctypes.data, grid.CELL.itemsize, 3, 4, 5, 0,
            ctypes.byref(count))
        assert code == _capi.ERR_DEVICE
        assert "Cuda error" in _capi.last_error()


def test_the_c_abi_refuses_bad_arguments(shared_library):
    from voxelized_geometry_tools_b200 import _capi
    lib = _capi.library()
    cells = np.zeros((2, 2, 2, 4), dtype=np.uint32)
    count = ctypes.c_uint32()
    for entry, extra in ((lib.vgt_b200_connected_components, ()),
                         (lib.vgt_b200_connected_components_dev, (None,))):
        def call(pointer, cell_bytes, dims, out):
            return entry(pointer, cell_bytes, *dims, 0, out, *extra)
        for cell_bytes in (4, 12, 0, 32):
            assert call(cells.ctypes.data, cell_bytes, (2, 2, 2),
                        ctypes.byref(count)) == _capi.ERR_INVALID_ARGUMENT
        assert "cell size" in _capi.last_error()
        assert call(None, 8, (2, 2, 2), ctypes.byref(count)) == _capi.ERR_INVALID_ARGUMENT
        assert call(cells.ctypes.data, 8, (2, 2, 2), None) == _capi.ERR_INVALID_ARGUMENT
        for dims in ((0, 2, 2), (2, -1, 2), (2, 2, 8193)):
            assert call(cells.ctypes.data, 8, dims,
                        ctypes.byref(count)) == _capi.ERR_INVALID_ARGUMENT
        # 2^32 cells or more: refused before anything is read
        for dims in ((4096, 1024, 1024), (8192, 8192, 8192)):
            assert call(cells.ctypes.data, 16, dims,
                        ctypes.byref(count)) == _capi.ERR_UNSUPPORTED
            assert "2^32" in _capi.last_error()
