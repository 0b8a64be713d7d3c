"""GPU: the cell maps' SDF entries on device-resident cells (vgt_b200_sdf_from_cells_*_dev,
vgt_b200_sdf_per_object_*_dev, vgt_b200_sdf_free_and_named_*_dev and their device.py functions)
against the host entries, byte for byte, and against the oracle.

The single SDF classifies the cells into a mask (CellsToMaskKernel), as the host entry does; the
batch classifies them once per group of 255 distinct ids into a slot map
(CellsToObjectSlotsKernel) and runs each SDF on "slot == key". torch.profiler checks which of the
two ran and which z-scan instantiation read the slot map.

The profiled calls run in a child process of their own (`launched_kernels`). A torch.profiler
session tears CUPTI down when it ends, and a later session in the same process can then miss the
first activities it should record. tests/test_gpu_sdf_thresholds.py counts kernels the same way,
so the test process must not have held a profiler session before it."""
import collections
import contextlib
import ctypes
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

import voxelized_geometry_tools_b200 as vgt
from voxelized_geometry_tools_b200 import _capi, grids

from .test_gpu_other_maps import params, random_cells, sizes_of

pytestmark = pytest.mark.gpu

REPO = Path(__file__).resolve().parents[1]
IDENTITY = np.eye(4)
CELL_TYPES = {8: grids.TAGGED_OBJECT_OCCUPANCY_CELL,
              16: grids.TAGGED_OBJECT_OCCUPANCY_COMPONENT_CELL}
MAP_TYPES = {8: vgt.TaggedObjectOccupancyMap, 16: vgt.TaggedObjectOccupancyComponentMap}
SCALARS = {np.float32: ("f32", ctypes.c_float), np.float64: ("f64", ctypes.c_double)}
SCAN_OF_LENGTH = {
    127: "ScanContiguousAxisKernel<ObjectSlot>",
    128: "ScanContiguousAxisRegistersKernel<SlotEquals4Source, 1>",
    1024: "ScanContiguousAxisRegistersKernel<SlotEquals4Source, 8>",
    2048: "ScanContiguousAxisRegistersKernel<SlotEquals4Source, 16>",
    4096: "ScanContiguousAxisVec4Kernel<SlotEquals4Source>",
}


def torch_dtype(dtype):
    import torch
    return {np.float32: torch.float32, np.float64: torch.float64}[dtype]


def device_cells(cells):
    """A structured cell array as the [nx, ny, nz, words] uint32 CUDA tensor device.py takes."""
    import torch
    words = cells.dtype.itemsize // 4
    raw = np.ascontiguousarray(cells).view(np.uint32).reshape(cells.shape + (words,))
    return torch.from_numpy(raw.copy()).to("cuda:0")


def launch_count():
    return int(_capi.library().vgt_b200_kernel_launch_count())


# ------------------------------------------------------------------------------------------------
# Kernel witness
# ------------------------------------------------------------------------------------------------
def short_kernel_name(name):
    name = name.replace("vgt_b200::edt::(anonymous namespace)::", "")
    if name.startswith("void "):
        name = name[len("void "):]
    return name.split("(")[0]


@contextlib.contextmanager
def _profiled():
    import torch
    kernels = collections.Counter()
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as profile:
        yield kernels
        torch.cuda.synchronize()
    for event in profile.events():
        if event.device_type == torch.autograd.DeviceType.CUDA:
            kernels[short_kernel_name(event.name)] += 1
    assert any(n.startswith("Scan") for n in kernels), sorted(kernels)


# The cases whose kernels are counted; each returns (cells, ids or objects, unknown_is_filled,
# add_virtual_border, dtype). The tests below check the results of the same cases.
def single_case(dtype, cell_bytes):
    rng = np.random.default_rng(70 + cell_bytes)
    return random_cells(rng, (23, 31, 40), CELL_TYPES[cell_bytes]), [1, 2], True, False, dtype


def route_case(nz):
    rng = np.random.default_rng(nz)
    cell_bytes = 16 if nz in (128, 2048) else 8
    dtype = np.float64 if nz in (1024, 4096) else np.float32
    cells = random_cells(rng, (4, 6, nz), CELL_TYPES[cell_bytes])
    ids = [4, 1, 9, 4, 0, 2]  # a repeat, an id absent from the map, id 0
    return cells, ids, nz != 128, nz in (127, 2048), dtype


def two_group_case():
    rng = np.random.default_rng(300)
    shape = (12, 10, 16)
    cells = random_cells(rng, shape, CELL_TYPES[16])
    cells["occupancy"] = np.where(rng.random(shape) < 0.6, 1.0, 0.0)
    cells["object_id"] = rng.integers(0, 302, shape, dtype=np.uint32)
    ids = rng.permutation(np.arange(1, 301, dtype=np.uint32))  # 300 distinct: two slot groups
    return cells, ids, True, False, np.float32


def profiled_cases():
    """{case: {kernel: launches}} of every profiled call; runs in the child process."""
    from voxelized_geometry_tools_b200 import device as vdev
    cases = {}
    for dtype in (np.float32, np.float64):
        for cell_bytes in (8, 16):
            cells, objects, unknown, border, _ = single_case(dtype, cell_bytes)
            cells_dev = device_cells(cells)
            with _profiled() as kernels:
                vdev.signed_distance_field_from_cells(cells_dev, 0.04, objects, unknown, border,
                                                      torch_dtype(dtype))
            cases[f"single {np.dtype(dtype).name} {cell_bytes}"] = dict(kernels)
    for name, (cells, ids, unknown, border, dtype) in (
            [(f"batch {nz}", route_case(nz)) for nz in sorted(SCAN_OF_LENGTH)]
            + [("two groups", two_group_case())]):
        cells_dev = device_cells(cells)
        with _profiled() as kernels:
            vdev.separate_object_sdfs(cells_dev, 0.05, ids, unknown, border, torch_dtype(dtype))
        cases[name] = dict(kernels)
    return cases


@pytest.fixture(scope="module")
def launched_kernels(shared_library):
    """The kernel counts of `profiled_cases`, taken in a child process (see the module text)."""
    script = ("import json, sys; sys.path.insert(0, %r); "
              "from tests.test_gpu_other_maps_dev import profiled_cases; "
              "print(json.dumps(profiled_cases()))" % str(REPO))
    command = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", script]
    result = subprocess.run(command, cwd=REPO, capture_output=True, text=True, timeout=1800)
    assert result.returncode == 0, result.stdout[-2000:] + result.stderr[-4000:]
    cases = json.loads(result.stdout.strip().splitlines()[-1])
    return {case: collections.Counter(kernels) for case, kernels in cases.items()}


def count(kernels, prefix):
    return sum(c for name, c in kernels.items() if name.startswith(prefix))


# ------------------------------------------------------------------------------------------------
# Host references
# ------------------------------------------------------------------------------------------------
def host_from_cells(cells, resolution, objects, unknown, border, dtype):
    tagged = MAP_TYPES[cells.dtype.itemsize](IDENTITY, "f", sizes_of(cells.shape, resolution),
                                             cells)
    sdf = tagged.ExtractSignedDistanceField(list(objects), params(unknown, border), dtype)
    return sdf.GetImmutableRawData(), sdf.GetMinimumMaximum()


def host_per_object(cells, resolution, ids, unknown, border, dtype):
    """vgt_b200_sdf_per_object_* called directly: one output per listed id, repeats included."""
    suffix, _ = SCALARS[dtype]
    ids = np.ascontiguousarray(ids, dtype=np.uint32)
    out = np.empty((ids.size,) + cells.shape, dtype=dtype)
    lows = np.empty(ids.size, dtype=dtype)
    highs = np.empty(ids.size, dtype=dtype)
    code = getattr(_capi.library(), "vgt_b200_sdf_per_object_" + suffix)(
        cells.ctypes.data, cells.dtype.itemsize, *cells.shape, resolution, int(unknown),
        int(border), ids.ctypes.data, ids.size, 0, out.ctypes.data, lows.ctypes.data,
        highs.ctypes.data)
    _capi.check(code)
    return out, lows, highs


def host_free_and_named(cells, resolution, unknown, border, dtype):
    tagged = MAP_TYPES[cells.dtype.itemsize](IDENTITY, "f", sizes_of(cells.shape, resolution),
                                             cells)
    sdf = tagged.ExtractFreeAndNamedObjectsSignedDistanceField(params(unknown, border), dtype)
    return sdf.GetImmutableRawData(), sdf.GetMinimumMaximum()


def assert_same_bytes(got, want):
    assert got.dtype == want.dtype and got.shape == want.shape
    assert got.tobytes() == want.tobytes()


# ------------------------------------------------------------------------------------------------
# One SDF
# ------------------------------------------------------------------------------------------------
OBJECT_LISTS = [(), (3,), (77,), (1, 4, 4, 1), (0, 2)]


@pytest.mark.parametrize("cell_bytes", [8, 16])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_single_sdf_equals_host_entry_and_oracle(shared_library, oracle, launched_kernels,
                                                 cell_bytes, dtype):
    from voxelized_geometry_tools_b200 import device as vdev
    cells = single_case(dtype, cell_bytes)[0]
    cells_dev = device_cells(cells)
    # the mask route, as in the host entry
    kernels = launched_kernels[f"single {np.dtype(dtype).name} {cell_bytes}"]
    assert kernels["CellsToMaskKernel"] == 1, sorted(kernels)
    assert kernels["ScanContiguousAxisRegistersKernel<Uchar4Source, 1>"] == 1, sorted(kernels)
    assert "CellsToObjectSlotsKernel" not in kernels, sorted(kernels)
    for objects in OBJECT_LISTS:
        for unknown in (True, False):
            for border in (False, True):
                sdf, min_max = vdev.signed_distance_field_from_cells(
                    cells_dev, 0.04, objects, unknown, border, torch_dtype(dtype))
                got = sdf.cpu().numpy()
                lo, hi = min_max.cpu().numpy().tolist()
                want, extrema = host_from_cells(cells, 0.04, objects, unknown, border, dtype)
                assert_same_bytes(got, want)
                assert (lo, hi) == tuple(extrema)
                oracle_sdf, oracle_extrema = oracle.sdf_from_cells(
                    cells, 0.04, unknown, border, list(objects), dtype=dtype)
                np.testing.assert_array_equal(got, oracle_sdf)
                assert (lo, hi) == tuple(oracle_extrema)


# ------------------------------------------------------------------------------------------------
# The batch
# ------------------------------------------------------------------------------------------------
def check_batch(oracle, cells, resolution, ids, unknown, border, dtype, sdfs, min_max,
                oracle_positions=None):
    got = sdfs.cpu().numpy()
    got_min_max = min_max.cpu().numpy()
    assert got.shape == (len(ids),) + cells.shape and got_min_max.shape == (len(ids), 2)
    want, lows, highs = host_per_object(cells, resolution, ids, unknown, border, dtype)
    assert_same_bytes(got, want)
    assert_same_bytes(got_min_max[:, 0].copy(), lows)
    assert_same_bytes(got_min_max[:, 1].copy(), highs)
    for k in (range(len(ids)) if oracle_positions is None else oracle_positions):
        oracle_sdf, (lo, hi) = oracle.sdf_from_cells(cells, resolution, unknown, border,
                                                     [int(ids[k])], dtype=dtype)
        np.testing.assert_array_equal(got[k], oracle_sdf)
        assert tuple(got_min_max[k].tolist()) == (lo, hi)


@pytest.mark.parametrize("nz", sorted(SCAN_OF_LENGTH))
def test_batch_on_every_scan_route(shared_library, oracle, launched_kernels, nz):
    from voxelized_geometry_tools_b200 import device as vdev
    cells, ids, unknown, border, dtype = route_case(nz)
    sdfs, min_max = vdev.separate_object_sdfs(device_cells(cells), 0.05, ids, unknown, border,
                                              torch_dtype(dtype))
    kernels = launched_kernels[f"batch {nz}"]
    assert kernels["CellsToObjectSlotsKernel"] == 1, sorted(kernels)
    assert "CellsToMaskKernel" not in kernels, sorted(kernels)
    assert kernels[SCAN_OF_LENGTH[nz]] == len(ids), sorted(kernels)
    assert count(kernels, "ScanContiguousAxis") == len(ids), sorted(kernels)
    check_batch(oracle, cells, 0.05, ids, unknown, border, dtype, sdfs, min_max)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_batch_slices_off_sixteen_byte_boundaries(shared_library, oracle, dtype):
    # V = 105: SDF k > 0 starts 4k or 8k bytes past a 16-byte boundary (nz % 4 != 0, so the
    # scalar z scan reads these grids anyway)
    from voxelized_geometry_tools_b200 import device as vdev
    rng = np.random.default_rng(9)
    shape = (3, 5, 7)
    cells = random_cells(rng, shape, CELL_TYPES[8], num_objects=4)
    ids = [1, 3, 2]
    sdfs, min_max = vdev.separate_object_sdfs(device_cells(cells), 0.1, ids, True, False,
                                              torch_dtype(dtype))
    check_batch(oracle, cells, 0.1, ids, True, False, dtype, sdfs, min_max)


def test_batch_of_two_slot_groups(shared_library, oracle, launched_kernels):
    from voxelized_geometry_tools_b200 import device as vdev
    cells, ids, unknown, border, dtype = two_group_case()
    sdfs, min_max = vdev.separate_object_sdfs(device_cells(cells), 0.05, ids, unknown, border,
                                              torch_dtype(dtype))
    kernels = launched_kernels["two groups"]
    assert kernels["CellsToObjectSlotsKernel"] == 2, sorted(kernels)
    assert "CellsToMaskKernel" not in kernels, sorted(kernels)
    assert count(kernels, "ScanContiguousAxisRegistersKernel<SlotEquals4Source, 1>") == 300
    # positions in the sorted ids: both ends, the last two of the first group of 255 (253, 254) and
    # the first two of the second (255, 256)
    distinct = np.sort(ids)
    edges = [int(np.flatnonzero(ids == distinct[p])[0]) for p in (0, 253, 254, 255, 256, 299)]
    check_batch(oracle, cells, 0.05, ids, unknown, border, dtype, sdfs, min_max,
                oracle_positions=edges)


# ------------------------------------------------------------------------------------------------
# Free and named
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cell_bytes", [8, 16])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_free_and_named_equals_host_entry(shared_library, oracle, cell_bytes, dtype):
    from voxelized_geometry_tools_b200 import device as vdev
    rng = np.random.default_rng(90 + cell_bytes)
    shape = (26, 22, 34)
    cells = random_cells(rng, shape, CELL_TYPES[cell_bytes], num_objects=3)
    cells_dev = device_cells(cells)
    for unknown, border in ((True, False), (False, True)):
        sdf, min_max = vdev.free_and_named_objects_sdf(cells_dev, 0.05, unknown, border,
                                                       torch_dtype(dtype))
        got = sdf.cpu().numpy()
        lo, hi = min_max.cpu().numpy().tolist()
        want, extrema = host_free_and_named(cells, 0.05, unknown, border, dtype)
        assert_same_bytes(got, want)
        assert (lo, hi) == tuple(extrema)
        oracle_sdf, oracle_extrema = oracle.sdf_free_and_named(cells, 0.05, unknown, border,
                                                               dtype)
        np.testing.assert_array_equal(got, oracle_sdf)
        assert (lo, hi) == tuple(oracle_extrema)


# ------------------------------------------------------------------------------------------------
# Streams, empty batches and refused arguments
# ------------------------------------------------------------------------------------------------
def test_entries_run_on_a_side_stream(shared_library, oracle):
    import torch
    from voxelized_geometry_tools_b200 import device as vdev
    rng = np.random.default_rng(11)
    shape = (40, 36, 64)
    cells = random_cells(rng, shape, CELL_TYPES[8], num_objects=4)
    cells_dev = device_cells(cells)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        single, single_min_max = vdev.signed_distance_field_from_cells(cells_dev, 0.03, [2])
        batch, batch_min_max = vdev.separate_object_sdfs(cells_dev, 0.03, [3, 1])
        merged, merged_min_max = vdev.free_and_named_objects_sdf(cells_dev, 0.03)
    side.synchronize()
    want, extrema = host_from_cells(cells, 0.03, [2], True, False, np.float32)
    assert_same_bytes(single.cpu().numpy(), want)
    assert tuple(single_min_max.cpu().numpy().tolist()) == tuple(extrema)
    check_batch(oracle, cells, 0.03, [3, 1], True, False, np.float32, batch, batch_min_max)
    want, extrema = host_free_and_named(cells, 0.03, True, False, np.float32)
    assert_same_bytes(merged.cpu().numpy(), want)
    assert tuple(merged_min_max.cpu().numpy().tolist()) == tuple(extrema)


def test_empty_batch_and_refusals_launch_nothing(shared_library):
    import torch
    from voxelized_geometry_tools_b200 import device as vdev
    lib = _capi.library()
    cells = torch.zeros((4, 4, 4, 2), dtype=torch.int32, device="cuda:0")
    out = torch.empty((4, 4, 4), dtype=torch.float32, device="cuda:0")
    out64 = torch.empty((4, 4, 4), dtype=torch.float64, device="cuda:0")
    min_max = torch.empty(2, dtype=torch.float32, device="cuda:0")
    ids = np.array([1, 2], dtype=np.uint32)
    stream = torch.cuda.current_stream().cuda_stream
    torch.cuda.synchronize()
    before = launch_count()

    sdfs, extrema = vdev.separate_object_sdfs(cells, 0.1, [])
    assert sdfs.shape == (0, 4, 4, 4) and extrema.shape == (0, 2)
    for suffix, target in (("f32", out), ("f64", out64)):
        entry = getattr(lib, f"vgt_b200_sdf_per_object_{suffix}_dev")
        assert entry(cells.data_ptr(), 8, 4, 4, 4, 0.1, 1, 0, None, 0, 0, target.data_ptr(),
                     None, stream) == _capi.OK

    base, c, o, m = cells.data_ptr(), cells.data_ptr(), out.data_ptr(), min_max.data_ptr()
    refusals = {
        "null cells": (0, 8, 4, 4, 4, 0.1, ids, 2, o, m),
        "null output": (c, 8, 4, 4, 4, 0.1, ids, 2, 0, m),
        "cell size": (c, 12, 4, 4, 4, 0.1, ids, 2, o, m),
        "empty axis": (c, 8, 0, 4, 4, 0.1, ids, 2, o, m),
        "long axis": (c, 8, 8193, 4, 4, 0.1, ids, 2, o, m),
        "resolution": (c, 8, 4, 4, 4, 0.0, ids, 2, o, m),
        "infinite resolution": (c, 8, 4, 4, 4, float("inf"), ids, 2, o, m),
        "negative id count": (c, 8, 4, 4, 4, 0.1, ids, -1, o, m),
        "ids missing": (c, 8, 4, 4, 4, 0.1, None, 2, o, m),
        "too many ids": (c, 8, 4, 4, 4, 0.1, ids, 2 ** 31, o, m),
        "unaligned cells": (base + 2, 8, 4, 4, 4, 0.1, ids, 2, o, m),
        "unaligned output": (c, 8, 4, 4, 4, 0.1, ids, 2, o + 2, m),
        "unaligned min/max": (c, 8, 4, 4, 4, 0.1, ids, 2, o, m + 1),
    }
    for what, (cp, size, nx, ny, nz, res, id_array, num, op, mp) in refusals.items():
        id_pointer = None if id_array is None else id_array.ctypes.data
        for name in ("vgt_b200_sdf_from_cells_f32_dev", "vgt_b200_sdf_per_object_f32_dev"):
            code = getattr(lib, name)(cp, size, nx, ny, nz, res, 1, 0, id_pointer, num, 0, op,
                                      mp, stream)
            assert code == _capi.ERR_INVALID_ARGUMENT, (what, name, _capi.last_error())
        if id_array is not None and num == 2:
            code = lib.vgt_b200_sdf_free_and_named_f32_dev(cp, size, nx, ny, nz, res, 1, 0, 0,
                                                            op, mp, stream)
            assert code == _capi.ERR_INVALID_ARGUMENT, (what, _capi.last_error())
    # 2^21 SDFs of 8192^3 doubles are 2^63 bytes
    assert lib.vgt_b200_sdf_per_object_f64_dev(c, 8, 8192, 8192, 8192, 0.1, 1, 0,
                                               ids.ctypes.data, 2 ** 21, 0, out64.data_ptr(),
                                               None, stream) == _capi.ERR_INVALID_ARGUMENT
    assert "overflow" in _capi.last_error()
    torch.cuda.synchronize()
    assert launch_count() == before


def test_python_argument_errors(shared_library):
    import torch
    from voxelized_geometry_tools_b200 import device as vdev
    good = torch.zeros((4, 4, 4, 2), dtype=torch.int32, device="cuda:0")
    functions = [lambda cells, **kw: vdev.signed_distance_field_from_cells(cells, 0.1, **kw),
                 lambda cells, **kw: vdev.separate_object_sdfs(cells, 0.1, [1], **kw),
                 lambda cells, **kw: vdev.free_and_named_objects_sdf(cells, 0.1, **kw)]
    for function in functions:
        for bad in (good.float(), good[..., :1].contiguous().expand(4, 4, 4, 2),
                    torch.zeros((4, 4, 4, 3), dtype=torch.int32, device="cuda:0"),
                    torch.zeros((4, 4, 8), dtype=torch.int32, device="cuda:0")):
            with pytest.raises(ValueError):
                function(bad)
        with pytest.raises(ValueError):
            function(good, dtype=torch.float16)
        with pytest.raises(_capi.BackendUnavailable):
            function(good.cpu())
        function(good.view(torch.uint32))
