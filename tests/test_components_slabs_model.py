"""CPU: the x-slab labelling of the component maps (vgt_b200_connected_components_multi,
csrc/connected_components.cu) as a numpy model, step by step: per-slab labels renumbered to their
local roots (the smallest local index of each local set), face edges between the last plane of
one slab and the first of the next with the implied-edge skip, the face graph resolved by
union-find over the sorted unique endpoints, the global roots counted and numbered per slab. It
reproduces the whole-grid labelling (scipy, renumbered by first occurrence) for every slab count;
plus the C-ABI's refusals, made before any device call."""
import ctypes
import zlib

import numpy as np
import pytest

from tests import components, slab_scenes
from tests.conftest import random_occupancy
from voxelized_geometry_tools_b200.sharded import split_range


def local_roots(key):
    """The local root (smallest linear index of its set) of every cell of one slab."""
    from scipy import ndimage
    flat_roots = np.empty(key.size, dtype=np.int64)
    index = np.arange(key.size, dtype=np.int64).reshape(key.shape)
    for value in np.unique(key):
        mask = key == value
        labelled, count = ndimage.label(mask)
        smallest = np.full(count + 1, np.iinfo(np.int64).max, dtype=np.int64)
        np.minimum.at(smallest, labelled[mask], index[mask])
        flat_roots[index[mask]] = smallest[labelled[mask]]
    return flat_roots


def slab_model(cells, num_slabs, rng):
    """Returns (ids, count, number of face edges)."""
    nx, ny, nz = cells.shape
    plane = ny * nz
    key = components.keys(cells)
    slabs = []
    for g in range(num_slabs):
        x0, x1 = split_range(nx, num_slabs, g)
        roots = local_roots(key[x0:x1])
        unique_roots = np.unique(roots)
        slabs.append(dict(x0=x0, x1=x1, base=x0 * plane, roots=roots,
                          unique_roots=unique_roots))

    # face edges: (global root below, global root above) where the keys are equal and the
    # (y, z - 1) pair does not already imply the edge
    edges = []
    z = np.arange(plane) % nz
    for g in range(1, num_slabs):
        below, above = slabs[g - 1], slabs[g]
        below_key = key[above["x0"] - 1].reshape(-1)
        above_key = key[above["x0"]].reshape(-1)
        equal = below_key == above_key
        implied = np.zeros(plane, dtype=bool)
        implied[1:] = (z[1:] > 0) & (above_key[:-1] == above_key[1:]) \
            & (below_key[:-1] == above_key[1:])
        emit = np.flatnonzero(equal & ~implied)
        below_roots = below["roots"][(below["x1"] - below["x0"] - 1) * plane + emit]
        above_roots = above["roots"][emit]
        assert np.all(np.isin(below_roots, below["unique_roots"]))
        edges.append(np.stack([below["base"] + below_roots, above["base"] + above_roots], axis=1))
    edges = np.concatenate(edges) if edges else np.zeros((0, 2), dtype=np.int64)

    # the face graph: nodes = sorted unique endpoints, union-find with parent <= self
    nodes = np.unique(edges.reshape(-1))
    compact = np.searchsorted(nodes, edges)
    parent = np.arange(nodes.size)

    def find(i):
        while parent[i] != i:
            parent[i] = parent[parent[i]]
            i = parent[i]
        return i

    for e in rng.permutation(len(compact)):
        a, b = find(compact[e, 0]), find(compact[e, 1])
        if a != b:
            parent[max(a, b)] = min(a, b)
    node_roots = np.array([find(k) for k in range(nodes.size)], dtype=np.int64)
    assert np.all(node_roots <= np.arange(nodes.size))

    # numbering: per slab, the local sets that are not merged into another node are the global
    # roots; ids = offset_g + 1 + rank among them
    slab_first = np.searchsorted(nodes, [s["base"] for s in slabs] + [nx * plane])
    counts = []
    for g, s in enumerate(slabs):
        first, last = slab_first[g], slab_first[g + 1]
        s["nodes"] = np.arange(first, last)
        s["node_ranks"] = np.searchsorted(s["unique_roots"], nodes[first:last] - s["base"])
        bits = np.ones(s["unique_roots"].size, dtype=bool)
        merged = node_roots[first:last] != s["nodes"]
        bits[s["node_ranks"][merged]] = False
        s["bits"] = bits
        counts.append(int(bits.sum()))
    offsets = np.concatenate([[0], np.cumsum(counts)])
    node_ids = np.zeros(nodes.size, dtype=np.int64)
    for g, s in enumerate(slabs):
        final = np.zeros(s["bits"].size, dtype=np.int64)
        final[s["bits"]] = offsets[g] + 1 + np.arange(counts[g])
        s["final"] = final
        node_ids[s["nodes"]] = final[s["node_ranks"]]  # published by the root nodes
    node_ids = node_ids[node_roots]
    ids = np.empty(cells.size, dtype=np.uint32)
    for g, s in enumerate(slabs):
        s["final"][s["node_ranks"]] = node_ids[s["nodes"]]
        assert np.all(s["final"] > 0)
        ranks = np.searchsorted(s["unique_roots"], s["roots"])
        ids[s["base"]:s["base"] + s["roots"].size] = s["final"][ranks]
    return ids.reshape(cells.shape), int(offsets[-1]), len(edges)


def spheres(rng, shape, count=6):
    index = np.indices(shape).reshape(3, -1).T
    occupancy = np.zeros(int(np.prod(shape)), dtype=np.float32)
    for _ in range(count):
        centre = rng.uniform(0, shape)
        radius = rng.uniform(1.0, max(1.5, min(shape) / 2.5))
        occupancy[((index - centre) ** 2).sum(axis=1) <= radius ** 2] = 1.0
    return occupancy.reshape(shape)


def scene(name, shape, rng):
    if name == "noise":
        return random_occupancy(rng, shape, rng.choice([0.3, 0.5, 0.7]))
    if name == "spheres":
        return spheres(rng, shape)
    if name == "serpentine":
        return components.serpentine(shape)
    if name == "x_serpentine":
        return slab_scenes.x_serpentine(shape)
    if name == "ring":
        return slab_scenes.ring_closed_in_slab(shape, shape[0] - 1)
    return slab_scenes.last_slab_components(shape, shape[0] - 1)


SHAPES = [(8, 5, 6), (9, 4, 7), (13, 1, 11), (12, 9, 1), (17, 6, 5), (24, 7, 3)]
SCENES = ["noise", "spheres", "serpentine", "x_serpentine", "ring", "last_slab"]


@pytest.mark.parametrize("tagged", [False, True], ids=["8B", "16B"])
@pytest.mark.parametrize("name", SCENES)
def test_slab_model_equals_the_whole_grid_labelling(name, tagged):
    rng = np.random.default_rng(zlib.crc32(repr((name, tagged)).encode()))
    for shape in SHAPES:
        object_id = rng.integers(0, 3, shape, dtype=np.uint32) if tagged else None
        cells = components.make_cells(scene(name, shape, rng), object_id, rng)
        want, want_count = components.scipy_components(cells)
        for num_slabs in range(1, min(8, shape[0]) + 1):  # one-plane slabs at nx == 8
            ids, count, _ = slab_model(cells, num_slabs, rng)
            assert count == want_count, (shape, num_slabs)
            np.testing.assert_array_equal(ids, want, err_msg=f"{shape} {num_slabs}")


def test_u_closed_only_in_a_later_slab():
    shape = (9, 8, 6)
    cells = components.make_cells(slab_scenes.ring_closed_in_slab(shape, 7))
    ids, count, edges = slab_model(cells, 3, np.random.default_rng(0))
    assert count == 2
    assert ids[0, 0, 1] == ids[0, 7, 1] == 2
    np.testing.assert_array_equal(ids, components.scipy_components(cells)[0])


def test_chain_crossing_every_face_many_times():
    shape = (16, 41, 3)
    cells = components.make_cells(slab_scenes.x_serpentine(shape))
    rows = (shape[1] + 1) // 2
    for num_slabs in (2, 4, 8):
        ids, count, edges = slab_model(cells, num_slabs, np.random.default_rng(num_slabs))
        assert count == 2
        # each face: one edge per filled row, one per free run of the face plane's y-z rows
        assert edges >= (num_slabs - 1) * rows


def test_implied_edges_are_skipped():
    # free space: every face has exactly one edge per y row (z = 0); the others are implied
    cells = components.make_cells(np.zeros((6, 5, 7), dtype=np.float32))
    ids, count, edges = slab_model(cells, 3, np.random.default_rng(0))
    assert count == 1 and edges == 2 * 5


# ---- the C-ABI without a device --------------------------------------------------------------
def call_multi(cells, cell_bytes, dims, devices, num_slabs, out):
    from voxelized_geometry_tools_b200 import _capi
    listed = None if devices is None else (ctypes.c_int * len(devices))(*devices)
    return _capi.library().vgt_b200_connected_components_multi(
        None if cells is None else cells.ctypes.data, cell_bytes, *dims, listed, num_slabs, out)


def test_the_multi_entry_refuses_bad_arguments(shared_library):
    from voxelized_geometry_tools_b200 import _capi
    cells = np.zeros((4, 2, 2, 4), dtype=np.uint32)
    count = ctypes.c_uint32()
    ok = dict(cells=cells, cell_bytes=8, dims=(4, 2, 2), devices=[0, 0], num_slabs=2,
              out=ctypes.byref(count))

    def refused(code_wanted, text, **changes):
        arguments = dict(ok, **changes)
        assert call_multi(**arguments) == code_wanted, changes
        assert text in _capi.last_error(), (changes, _capi.last_error())

    invalid = _capi.ERR_INVALID_ARGUMENT
    refused(invalid, "null cell array", cells=None)
    refused(invalid, "null device list", devices=None)
    refused(invalid, "null component count", out=None)
    for num_slabs in (0, 9, -1):
        refused(invalid, "slabs", num_slabs=num_slabs, devices=[0] * max(num_slabs, 1))
    refused(invalid, "more slabs", dims=(3, 2, 2), devices=[0] * 4, num_slabs=4)
    for cell_bytes in (4, 12, 0, 32):
        refused(invalid, "cell size", cell_bytes=cell_bytes)
    for dims in ((0, 2, 2), (2, -1, 2), (2, 2, 8193), (8193, 2, 2)):
        refused(invalid, "out of range", dims=dims)
    refused(invalid, "device ordinal", devices=[0, -1])
    # slabs of 2^32 cells or more: refused before anything is read
    refused(_capi.ERR_UNSUPPORTED, "2^32", dims=(4096, 1024, 1024), devices=[0], num_slabs=1)
    refused(_capi.ERR_UNSUPPORTED, "2^32", dims=(8192, 8192, 8192), devices=[0] * 8, num_slabs=8)
    refused(_capi.ERR_UNSUPPORTED, "2^32", dims=(8192, 1024, 1025), devices=[0, 0], num_slabs=2)


def test_no_cpu_fallback_without_device(shared_library):
    import voxelized_geometry_tools_b200 as vgt
    from voxelized_geometry_tools_b200 import _capi
    if _capi.device_count() > 0:
        pytest.skip("a GPU is present")
    cells = components.make_cells(np.zeros((4, 3, 5), dtype=np.float32))
    before = cells.copy()
    for num_slabs in (1, 2, 4):
        count = ctypes.c_uint32(7)
        code = call_multi(cells, 8, cells.shape, [0] * num_slabs, num_slabs, ctypes.byref(count))
        assert code == _capi.ERR_DEVICE
        assert "Cuda error" in _capi.last_error()
        assert count.value == 7
    assert cells.tobytes() == before.tobytes()
    sizes = vgt.VoxelGridSizes.FromVoxelCounts(0.1, (4, 3, 5))
    for cls in (vgt.OccupancyComponentMap, vgt.TaggedObjectOccupancyComponentMap):
        with pytest.raises(vgt.BackendUnavailable):
            cls(np.eye(4), "world", sizes).UpdateConnectedComponents(devices=[0, 0])
