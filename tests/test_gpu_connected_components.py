"""GPU: connected components of the component maps through the C-ABI (host entry via
UpdateConnectedComponents, device entry via device.connected_components) against the reference's
scan and breadth-first fill restated in oracle/components_oracle.cpp (small grids) or
scipy.ndimage.label renumbered by first occurrence (large grids): the same ids and count, every
other cell byte unchanged, host and device entries equal, repeated calls identical, and
concurrent callers on different maps each right."""
import threading
import zlib

import numpy as np
import pytest

from tests import components
from tests.conftest import random_occupancy

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def cc_oracle():
    """The restated reference (oracle/components_oracle.py), built for this host if needed."""
    from oracle import components_oracle
    components_oracle.build()
    return components_oracle


@pytest.fixture(scope="module")
def vgt(shared_library):
    import voxelized_geometry_tools_b200 as module
    return module


def make_map(vgt, cells):
    sizes = vgt.VoxelGridSizes.FromVoxelCounts(0.1, cells.shape)
    cls = vgt.OccupancyComponentMap if cells.dtype.itemsize == 8 \
        else vgt.TaggedObjectOccupancyComponentMap
    return cls(np.eye(4), "world", sizes, data=cells.copy())


def run_host(vgt, cells):
    grid = make_map(vgt, cells)
    count = grid.UpdateConnectedComponents()
    return grid.GetImmutableRawData(), count


def run_device(cells):
    import torch
    from voxelized_geometry_tools_b200 import device
    words = cells.dtype.itemsize // 4
    raw = np.ascontiguousarray(cells).view(np.uint32).reshape(cells.shape + (words,))
    tensor = torch.from_numpy(raw.view(np.int32).copy()).cuda()
    count = device.connected_components(tensor)
    torch.cuda.synchronize()
    out = tensor.cpu().numpy().view(np.uint32).reshape(-1).view(cells.dtype).reshape(cells.shape)
    return out, int(count.item())


def check(vgt, cells, want_ids, want_count, device_entry=True, repeat=True):
    got, count = run_host(vgt, cells)
    assert count == want_count
    np.testing.assert_array_equal(got["component"], want_ids)
    for name in cells.dtype.names:
        if name != "component":
            np.testing.assert_array_equal(got[name].view(np.uint32), cells[name].view(np.uint32),
                                          err_msg=name)
    if repeat:
        again, count_again = run_host(vgt, cells)
        assert count_again == count
        assert again.tobytes() == got.tobytes()
    if device_entry:
        on_device, device_count = run_device(cells)
        assert device_count == count
        assert on_device.tobytes() == got.tobytes()
    return got


SHAPES = [(1, 1, 1), (1, 1, 37), (1, 29, 1), (31, 1, 1), (5, 7, 9), (13, 11, 3), (3, 4, 33),
          (2, 3, 65), (2, 2, 1025), (3, 5, 257), (9, 17, 31)]
SCENES = ["free", "filled", "checkerboard", "noise30", "noise50", "blobs", "serpentine", "shells",
          "special"]


def scene(name, shape, rng):
    if name == "free":
        return np.zeros(shape, dtype=np.float32)
    if name == "filled":
        return np.ones(shape, dtype=np.float32)
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
    if name == "shells":
        return components.nested_shells(shape)
    return components.special_values(rng, shape)


@pytest.mark.parametrize("tagged", [False, True], ids=["8B", "16B"])
@pytest.mark.parametrize("name", SCENES)
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_equals_the_restated_reference(cc_oracle, vgt, shape, name, tagged):
    rng = np.random.default_rng(zlib.crc32(repr((shape, name, tagged)).encode()))
    occupancy = scene(name, shape, rng)
    object_id = None
    if tagged:
        uniform = name in ("free", "filled", "checkerboard")
        object_id = np.full(shape, 3, np.uint32) if uniform \
            else rng.integers(0, 3, shape, dtype=np.uint32)
    cells = components.make_cells(occupancy, object_id, rng)  # garbage component words
    want, want_count = cc_oracle.connected_components(cells)
    volume = int(np.prod(shape))
    if name in ("free", "filled"):
        assert want_count == 1
    if name == "checkerboard":
        assert want_count == volume
    check(vgt, cells, want["component"], want_count)


def test_object_ids_split_and_the_boundary_splits(cc_oracle, vgt):
    rng = np.random.default_rng(5)
    shape = (6, 10, 70)
    occupancy = np.ones(shape, dtype=np.float32)
    occupancy[:, :, 35:] = 0.0                     # free half with the same ids as the filled
    object_id = np.zeros(shape, dtype=np.uint32)
    object_id[:, ::2, :] = 1                       # neighbours along y differ only in the id
    object_id[3:, :, :] += 7
    cells = components.make_cells(occupancy, object_id, rng)
    want, want_count = cc_oracle.connected_components(cells)
    # every (x half, y row, z half) is its own component: rows alternate ids along y
    assert want_count == 2 * shape[1] * 2
    check(vgt, cells, want["component"], want_count)


def test_large_8_byte_map_equals_scipy(vgt):
    rng = np.random.default_rng(512)
    shape = (512, 512, 512)
    cells = components.make_cells(random_occupancy(rng, shape, 0.3, unknown=0.0),
                                  None, rng)
    want, want_count = components.scipy_components(cells)
    check(vgt, cells, want, want_count, repeat=False)


def test_large_16_byte_map_equals_scipy(vgt):
    rng = np.random.default_rng(256)
    shape = (256, 256, 256)
    occupancy = random_occupancy(rng, shape, 0.5)
    object_id = (rng.random(shape) < 0.2).astype(np.uint32)
    cells = components.make_cells(occupancy, object_id, rng)
    want, want_count = components.scipy_components(cells)
    check(vgt, cells, want, want_count)


def test_large_serpentine_equals_scipy(vgt):
    rng = np.random.default_rng(3)
    cells = components.make_cells(components.serpentine((96, 128, 160)), None, rng)
    want, want_count = components.scipy_components(cells)
    assert want_count == 2
    check(vgt, cells, want, want_count)


def test_two_host_threads_on_different_maps(cc_oracle, vgt):
    rng = np.random.default_rng(11)
    jobs = [components.make_cells(random_occupancy(rng, (40, 50, 70), 0.3), None, rng),
            components.make_cells(random_occupancy(rng, (33, 65, 48), 0.5, blobs=True),
                                  rng.integers(0, 2, (33, 65, 48), dtype=np.uint32), rng)]
    wants = [cc_oracle.connected_components(cells) for cells in jobs]
    results = [None, None]
    errors = []

    def work(k):
        try:
            for _ in range(4):
                got, count = run_host(vgt, jobs[k])
                if results[k] is not None:
                    assert got.tobytes() == results[k][0].tobytes()
                results[k] = (got, count)
        except Exception as error:  # reported on the main thread
            errors.append(error)

    threads = [threading.Thread(target=work, args=(k,)) for k in range(2)]
    for thread in threads:
        thread.start()
    for thread in threads:
        thread.join()
    assert errors == []
    for (got, count), (want, want_count) in zip(results, wants):
        assert count == want_count
        np.testing.assert_array_equal(got["component"], want["component"])


def test_device_entry_restores_the_current_device_and_uses_the_stream(vgt):
    import torch
    from voxelized_geometry_tools_b200 import device
    rng = np.random.default_rng(8)
    cells = components.make_cells(random_occupancy(rng, (64, 64, 64), 0.4), None, rng)
    want, want_count = components.scipy_components(cells)
    raw = cells.view(np.int32).reshape(cells.shape + (2,))
    tensor = torch.from_numpy(raw.copy()).cuda()
    before = torch.cuda.current_device()
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        count = device.connected_components(tensor)
    stream.synchronize()
    assert torch.cuda.current_device() == before
    assert int(count.item()) == want_count
    np.testing.assert_array_equal(tensor[..., 1].cpu().numpy().view(np.uint32), want)
