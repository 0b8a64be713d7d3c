"""GPU: the occupancy -> SDF path on both sides of every kernel-selection and value-range threshold,
for every input type, bit for bit against the oracle (and the reference's own code where
oracle/_ref is built).

Every call picks among about twenty kernel instantiations by line length, pointer alignment, input
type and the largest partial distance it can see, and inside the kernels fixed ranges decide what
is computed in 16 bits, in 32 bits, from a table or by another kernel. Each case here states the
route it targets and checks, with torch.profiler, that the targeted kernel really ran: when a
threshold moves, a case that drifted off its route fails instead of passing without checking
anything. The rules the cases restate (and assert their shapes against) are:

* z scan (LaunchScan, csrc/edt_kernels.cu): register kernel <Source, 1/2/4/8/16> for aligned lines
  of <= 128/256/512/1024/2048 voxels, the Vec4 kernel for longer aligned lines, the scalar kernel
  otherwise. Aligned: length % 4 == 0, input aligned to the source vector (16 B float4, 4 B
  uchar4), output aligned to 16 B.
* stack kernel entries (LaunchEnvelope): packed (f << 10) | v entries when the line has <= 1024
  voxels and the largest input is <= 2^21 - 1, else split entries; the 32-bit pop test when
  (max_input + (L - 1)^2) * L < 2^31, else 64-bit.
* window kernel (csrc/edt_envelope_window.cuh): certify below (R + 1)^2, values clamped at
  kSaturated = 0x7800, joint search capped at 168 rows.
* finalize magnitude table: 2^20 entries, larger squared distances take the direct fp64 path.
* axes of up to VGT_B200_MAX_AXIS = 8192 voxels.
* the transform's range: integer samples, max sample + 1 + sum (n - 1)^2 <= 2^29 - 1.
* the pipelined host entry: >= 2^24 voxels and nx > 1; min(nx, 8) slabs in, min(ny, 8) slabs out.
"""
import collections
import contextlib
import ctypes
import os
import re

import numpy as np
import pytest

import voxelized_geometry_tools_b200 as vgt
from voxelized_geometry_tools_b200 import _capi

from .conftest import random_occupancy
from .test_gpu_sdf import IDENTITY, assert_matches_oracle, make_map, params, squared_to_int

pytestmark = pytest.mark.gpu

# profiles/kernel_coverage.py runs the suite inside one profiler session of its own and sets this;
# a second session cannot start inside it, so the route checks stand down there (the values are
# still checked). Everywhere else every route check is active.
COVERAGE_RUN = os.environ.get("VGT_B200_KERNEL_COVERAGE") == "1"

MAX_AXIS = 8192
PACKED_MAX_LENGTH = 1024
PACKED_MAX_INPUT = 2 ** 21 - 1
TRANSFORM_MAX_INPUT = 2 ** 29 - 1
PIPELINE_MIN_VOXELS = 2 ** 24
PIPELINE_CHUNKS = 8
MAGNITUDE_TABLE_ENTRIES = 2 ** 20
SATURATED = 0x7800
WINDOW_RADIUS_PACKED = 12
JOINT_SEARCH_CAP = 168


# ------------------------------------------------------------------------------------------------
# Route witness
# ------------------------------------------------------------------------------------------------
def short_kernel_name(name: str) -> str:
    """'void vgt_b200::edt::(anonymous namespace)::K<vgt_b200::edt::(anonymous namespace)::S, 2>(...)'
    -> 'K<S, 2>'."""
    name = name.replace("vgt_b200::edt::(anonymous namespace)::", "")
    if name.startswith("void "):
        name = name[len("void "):]
    return name.split("(")[0]


class Launched(collections.Counter):
    """Launch count of every kernel (short name) that ran inside the `launched()` block."""

    recorded = False

    def assert_ran(self, name: str) -> None:
        if self.recorded:
            assert self[name] > 0, f"{name} did not run; launched: {sorted(self)}"

    def assert_not_ran(self, prefix: str) -> None:
        if self.recorded:
            assert not any(n.startswith(prefix) for n in self), (prefix, sorted(self))

    def count(self, prefix: str) -> int:
        return sum(c for n, c in self.items() if n.startswith(prefix))

    def lean_routes(self, mode: int) -> set:
        """(narrow, split) of every EnvelopeAxisLeanKernel<mode, ...> that ran."""
        routes = set()
        for n in self:
            m = re.fullmatch(r"EnvelopeAxisLeanKernel<(\d), (true|false), (?:true|false), "
                             r"(?:true|false), (true|false), \d+>", n)
            if m and int(m.group(1)) == mode:
                routes.add((m.group(2) == "true", m.group(3) == "true"))
        return routes

    def assert_lean_routes(self, mode: int, expected: set) -> None:
        if self.recorded:
            assert self.lean_routes(mode) == expected, sorted(self)


@contextlib.contextmanager
def _launched_kernels():
    import torch
    launched = Launched()
    if COVERAGE_RUN:
        yield launched
        return
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as profile:
        yield launched
        torch.cuda.synchronize()
    for event in profile.events():
        if event.device_type == torch.autograd.DeviceType.CUDA:
            launched[short_kernel_name(event.name)] += 1
    launched.recorded = True
    # the library's kernels must be visible at all, or every route check would be vacuous
    assert any(n.startswith(("Scan", "Envelope", "Ingest", "CellsToMask")) for n in launched), \
        sorted(launched)


@pytest.fixture
def launched():
    """`with launched() as kernels:` runs the block under torch.profiler (CUDA activities) and
    fills `kernels` with the launch count of every kernel that ran."""
    return _launched_kernels


TUNING_SWITCHES = ("VGT_B200_WINDOW_BUDGET", "VGT_B200_ENVELOPE", "VGT_B200_WINDOW_PILOT",
                   "VGT_B200_WINDOW_STAGE", "VGT_B200_WINDOW_RADIUS_Y")
ROUTES = [{}, {"VGT_B200_ENVELOPE": "lean"}, {"VGT_B200_WINDOW_BUDGET": "100000"},
          {"VGT_B200_WINDOW_PILOT": "0"}]


@contextlib.contextmanager
def tuning(switches):
    """The library's A/B switches (read once per process; vgt_b200_reload_tuning re-reads)."""
    saved = {key: os.environ.get(key) for key in TUNING_SWITCHES}
    for key in saved:
        os.environ.pop(key, None)
    os.environ.update(switches)
    _capi.library().vgt_b200_reload_tuning()
    try:
        yield
    finally:
        for key, value in saved.items():
            os.environ.pop(key, None)
            if value is not None:
                os.environ[key] = value
        _capi.library().vgt_b200_reload_tuning()


def assert_envelope_route(kernels, switches):
    if switches.get("VGT_B200_ENVELOPE") == "lean":
        kernels.assert_not_ran("EnvelopeAxisWindowKernel")
    else:
        assert not kernels.recorded or kernels.count("EnvelopeAxisWindowKernel") > 0, sorted(kernels)
    if switches.get("VGT_B200_WINDOW_PILOT") == "0":
        kernels.assert_not_ran("DecideWindowModeKernel")


# ------------------------------------------------------------------------------------------------
# The dispatch rules, restated
# ------------------------------------------------------------------------------------------------
def scan_kernel(length: int, source: str, aligned: bool = True) -> str:
    if aligned and length % 4 == 0:
        if length <= 2048:
            iterations = next(i for i in (1, 2, 4, 8, 16) if length <= 128 * i)
            return f"ScanContiguousAxisRegistersKernel<{source}, {iterations}>"
        return f"ScanContiguousAxisVec4Kernel<{source}>"
    return "ScanContiguousAxisKernel<{}>".format(
        "float" if source == "Float4Source" else "unsigned char")


def lean_route(length: int, max_input: int):
    """(narrow, split) of the stack kernel for one pass."""
    packed = length <= PACKED_MAX_LENGTH and max_input <= PACKED_MAX_INPUT
    narrow = packed and (max_input + (length - 1) ** 2) * length < 2 ** 31
    return narrow, not packed


def occupancy_lean_routes(shape):
    """{mode 0 (y pass): routes, 1 (x pass + finalize): routes} of an occupancy -> SDF call."""
    nx, ny, nz = shape
    y_pass = {lean_route(ny, (nz - 1) ** 2)} if ny > 1 else set()
    return y_pass, {lean_route(nx, (nz - 1) ** 2 + (ny - 1) ** 2)}


def transform_lean_routes(shape, largest_sample):
    """Routes of the transform's passes (x, y, z; an axis of one voxel is skipped)."""
    routes = set()
    max_input = largest_sample + 1
    for n in shape:
        if n > 1:
            routes.add(lean_route(n, max_input))
            max_input += (n - 1) ** 2
    return routes


def transform_checker(oracle):
    from oracle import reference_oracle
    return reference_oracle.transform_inplace if reference_oracle.available() \
        else oracle.transform_inplace


def test_restated_rules_on_both_sides_of_each_edge():
    # the two sides of each edge the cases below rely on
    assert lean_route(64, 2_097_151) == (True, False)          # sample 2 097 150: packed
    assert lean_route(64, 2_097_152) == (False, True)          # sample 2 097 151: split
    assert (1_050_622 + 1023 ** 2) * 1024 == 2 ** 31 - 1024
    assert lean_route(1024, 1_050_622) == (True, False)        # sample 1 050 621: 32-bit pops
    assert lean_route(1024, 1_050_623) == (False, False)       # sample 1 050 622: 64-bit pops
    assert lean_route(1024, 1024 ** 2) == (True, False)        # occupancy (1, 1024, 1025)
    assert lean_route(1024, 1025 ** 2) == (False, False)       # occupancy (1, 1024, 1026)
    assert lean_route(1025, 4) == (False, True)
    assert scan_kernel(2048, "Uchar4Source") == "ScanContiguousAxisRegistersKernel<Uchar4Source, 16>"
    assert scan_kernel(2052, "Uchar4Source") == "ScanContiguousAxisVec4Kernel<Uchar4Source>"
    assert scan_kernel(128, "Float4Source", aligned=False) == "ScanContiguousAxisKernel<float>"


# ------------------------------------------------------------------------------------------------
# b. z scan x input type x alignment
# ------------------------------------------------------------------------------------------------
ALIGNED_LENGTHS = [124, 128, 132, 252, 256, 260, 508, 512, 516, 1020, 1024, 1028, 2044, 2048, 2052,
                   4096, 8192]
SCALAR_LENGTHS = [127, 1025, 2047, 2049, 8191]
LINE_MARKS = (0, 31, 32, 127, 128, 1023, 1024, 2047, 2048)
RESOLUTION = 0.05


def line_grid(rng, length):
    """[3, ny, length]: x = 0 lines hold one filled voxel at each mark (a warp word, a 128-voxel
    iteration, a register half apart), x = 1 the same with one free voxel in a filled line, two
    lines of each of those planes are all free / all filled, the rest are blobs."""
    marks = sorted({m for m in LINE_MARKS if m < length} | {length - 1})
    ny = len(marks) + 4
    occupancy = random_occupancy(rng, (3, ny, length), 0.1, blobs=True)
    for k, mark in enumerate(marks):
        occupancy[0, k, :] = 0.0
        occupancy[0, k, mark] = 1.0
        occupancy[1, k, :] = 1.0
        occupancy[1, k, mark] = 0.0
    occupancy[0:2, -4, :] = 0.0
    occupancy[0:2, -3, :] = 1.0
    return occupancy


def mask_values(rng, filled):
    """uint8 mask: every non-zero value counts as filled; 2, 128 and 255 as well as 1."""
    values = rng.choice(np.array([1, 2, 128, 255], dtype=np.uint8), size=filled.shape)
    return np.where(filled, values, 0).astype(np.uint8)


def cells_from(occupancy, rng, cell_dtype):
    cells = np.zeros(occupancy.shape, dtype=cell_dtype)
    cells["occupancy"] = occupancy
    if "object_id" in cell_dtype.names:
        cells["object_id"] = rng.integers(0, 4, occupancy.shape)
    if "component" in cell_dtype.names:
        cells["component"] = rng.integers(0, 1000, occupancy.shape)
    return cells


def offset_view(tensor, elements):
    """A contiguous copy of `tensor` that starts `elements` elements into a larger buffer."""
    import torch
    buffer = torch.empty(tensor.numel() + elements, dtype=tensor.dtype, device=tensor.device)
    view = buffer[elements:].view(tensor.shape)
    view.copy_(tensor)
    return view


def assert_device_sdf(got, min_max, want, lo, hi):
    np.testing.assert_array_equal(got.cpu().numpy(), want)
    assert tuple(min_max.cpu().numpy().tolist()) == (lo, hi)


@pytest.mark.parametrize("length", ALIGNED_LENGTHS + SCALAR_LENGTHS)
def test_z_scan_routes_for_every_input_type(shared_library, oracle, launched, length):
    import torch
    from voxelized_geometry_tools_b200 import device as vdev
    from voxelized_geometry_tools_b200.grids import (OCCUPANCY_COMPONENT_CELL,
                                                     TAGGED_OBJECT_OCCUPANCY_CELL,
                                                     TAGGED_OBJECT_OCCUPANCY_COMPONENT_CELL)
    rng = np.random.default_rng(length)
    occupancy = line_grid(rng, length)
    float_scan = scan_kernel(length, "Float4Source")
    mask_scan = scan_kernel(length, "Uchar4Source")
    cuda = torch.device("cuda", 0)

    # float occupancy, host entry
    with launched() as kernels:
        assert_matches_oracle(oracle, occupancy, RESOLUTION)
    kernels.assert_ran(float_scan)
    # float occupancy, device entries (aligned buffers), float and double
    want, (lo, hi) = oracle.sdf(occupancy, RESOLUTION)
    occupancy_dev = torch.from_numpy(occupancy).to(cuda)
    with launched() as kernels:
        aligned_out, aligned_min_max = vdev.signed_distance_field(occupancy_dev, RESOLUTION)
        assert_device_sdf(aligned_out, aligned_min_max, want, lo, hi)
    kernels.assert_ran(float_scan)
    want64, (lo64, hi64) = oracle.sdf(occupancy, RESOLUTION, False, True, dtype=np.float64)
    with launched() as kernels:
        out64, min_max64 = vdev.signed_distance_field_f64(occupancy_dev, RESOLUTION, False, True)
        assert_device_sdf(out64, min_max64, want64, lo64, hi64)
    kernels.assert_ran(float_scan)

    # uint8 mask, host and device entries; 2, 128 and 255 are filled like 1
    mask = mask_values(rng, occupancy > 0.5)
    want_mask, (lo_mask, hi_mask) = oracle.sdf_from_mask(mask != 0, RESOLUTION)
    sizes = vgt.VoxelGridSizes.FromVoxelCounts(RESOLUTION, mask.shape)
    with launched() as kernels:
        sdf = vgt.ExtractSignedDistanceFieldFromMask(mask, IDENTITY, "f", sizes, params())
    np.testing.assert_array_equal(sdf.GetImmutableRawData(), want_mask)
    assert sdf.GetMinimumMaximum() == (lo_mask, hi_mask)
    kernels.assert_ran(mask_scan)
    mask_dev = torch.from_numpy(mask).to(cuda)
    with launched() as kernels:
        mask_out, mask_min_max = vdev.signed_distance_field_from_mask(mask_dev, RESOLUTION)
        assert_device_sdf(mask_out, mask_min_max, want_mask, lo_mask, hi_mask)
    kernels.assert_ran(mask_scan)

    # unaligned device buffers: the scalar kernels, the same bytes
    if length % 4 == 0:
        with launched() as kernels:
            out, min_max = vdev.signed_distance_field(offset_view(occupancy_dev, 1), RESOLUTION)
            assert torch.equal(out, aligned_out) and torch.equal(min_max, aligned_min_max)
        kernels.assert_ran("ScanContiguousAxisKernel<float>")
        with launched() as kernels:
            out = offset_view(torch.zeros_like(occupancy_dev), 1)
            out, min_max = vdev.signed_distance_field(occupancy_dev, RESOLUTION, out=out)
            assert torch.equal(out, aligned_out) and torch.equal(min_max, aligned_min_max)
        kernels.assert_ran("ScanContiguousAxisKernel<float>")
        with launched() as kernels:
            out, min_max = vdev.signed_distance_field_from_mask(offset_view(mask_dev, 1),
                                                                RESOLUTION)
            assert torch.equal(out, mask_out) and torch.equal(min_max, mask_min_max)
        kernels.assert_ran("ScanContiguousAxisKernel<unsigned char>")

    # 8- and 16-byte cells, with and without an object list (the cells become a device mask)
    from oracle import reference_oracle
    for cell_dtype, objects in ((OCCUPANCY_COMPONENT_CELL, ()),
                                (TAGGED_OBJECT_OCCUPANCY_CELL, ()),
                                (TAGGED_OBJECT_OCCUPANCY_CELL, (1, 3)),
                                (TAGGED_OBJECT_OCCUPANCY_COMPONENT_CELL, ()),
                                (TAGGED_OBJECT_OCCUPANCY_COMPONENT_CELL, (2,))):
        cells = cells_from(occupancy, rng, cell_dtype)
        sizes = vgt.VoxelGridSizes.FromVoxelCounts(RESOLUTION, cells.shape)
        if cell_dtype is OCCUPANCY_COMPONENT_CELL:
            grid = vgt.OccupancyComponentMap(IDENTITY, "f", sizes, data=cells)
            call = lambda: grid.ExtractSignedDistanceField(params())  # noqa: E731
        elif cell_dtype is TAGGED_OBJECT_OCCUPANCY_CELL:
            grid = vgt.TaggedObjectOccupancyMap(IDENTITY, "f", sizes, data=cells)
            call = lambda: grid.ExtractSignedDistanceField(objects, params())  # noqa: E731
        else:
            grid = vgt.TaggedObjectOccupancyComponentMap(IDENTITY, "f", sizes, data=cells)
            call = lambda: grid.ExtractSignedDistanceField(objects, params())  # noqa: E731
        with launched() as kernels:
            sdf = call()
        kernels.assert_ran(mask_scan)
        want_cells, (lo_cells, hi_cells) = oracle.sdf_from_cells(cells, RESOLUTION,
                                                                 objects_to_use=objects)
        np.testing.assert_array_equal(sdf.GetImmutableRawData(), want_cells)
        assert sdf.GetMinimumMaximum() == (lo_cells, hi_cells)
        if reference_oracle.maps_available():
            if cell_dtype is TAGGED_OBJECT_OCCUPANCY_CELL:
                ref, ref_min_max = reference_oracle.tagged_map_sdf(cells, RESOLUTION, objects)
            else:
                ref, ref_min_max = reference_oracle.component_map_sdf(cells, RESOLUTION, objects)
            np.testing.assert_array_equal(sdf.GetImmutableRawData(), ref)
            assert sdf.GetMinimumMaximum() == ref_min_max


@pytest.mark.parametrize("length", [127, 128, 1028])
def test_special_occupancy_values(shared_library, oracle, launched, length):
    # NaN, +-inf, -0.0, 0.5 and the floats right next to 0.5, under both unknown_is_filled rules
    import torch
    from voxelized_geometry_tools_b200 import device as vdev
    from voxelized_geometry_tools_b200.grids import TAGGED_OBJECT_OCCUPANCY_CELL
    from oracle import reference_oracle
    rng = np.random.default_rng(length + 7)
    specials = np.array([np.nan, np.inf, -np.inf, -0.0, 0.0, 0.5,
                         np.nextafter(np.float32(0.5), np.float32(1)),
                         np.nextafter(np.float32(0.5), np.float32(0)), 1.0], dtype=np.float32)
    occupancy = line_grid(rng, length)
    pick = rng.random(occupancy.shape) < 0.3
    occupancy[pick] = rng.choice(specials, size=int(pick.sum()))
    occupancy[2, 0, :] = specials[np.arange(length) % len(specials)]
    occupancy_dev = torch.from_numpy(occupancy).to(torch.device("cuda", 0))
    for unknown_is_filled in (True, False):
        with launched() as kernels:
            assert_matches_oracle(oracle, occupancy, RESOLUTION, unknown_is_filled)
        kernels.assert_ran(scan_kernel(length, "Float4Source"))
        assert_matches_oracle(oracle, occupancy, RESOLUTION, unknown_is_filled, True, np.float64)
        want, (lo, hi) = oracle.sdf(occupancy, RESOLUTION, unknown_is_filled)
        out, min_max = vdev.signed_distance_field(occupancy_dev, RESOLUTION, unknown_is_filled)
        assert_device_sdf(out, min_max, want, lo, hi)
        got_filled, got_free = vgt.ComputeSquaredDistanceFields(occupancy, unknown_is_filled)
        want_filled, want_free = oracle.edt_squared(occupancy, unknown_is_filled)
        np.testing.assert_array_equal(got_filled, squared_to_int(want_filled))
        np.testing.assert_array_equal(got_free, squared_to_int(want_free))
        cells = cells_from(occupancy, rng, TAGGED_OBJECT_OCCUPANCY_CELL)
        grid = vgt.TaggedObjectOccupancyMap(
            IDENTITY, "f", vgt.VoxelGridSizes.FromVoxelCounts(RESOLUTION, cells.shape), data=cells)
        sdf = grid.ExtractSignedDistanceField((), params(unknown_is_filled))
        want_cells, _ = oracle.sdf_from_cells(cells, RESOLUTION, unknown_is_filled)
        np.testing.assert_array_equal(sdf.GetImmutableRawData(), want_cells)
        if reference_oracle.maps_available():
            ref, ref_min_max = reference_oracle.occupancy_map_sdf(occupancy, RESOLUTION,
                                                                  unknown_is_filled)
            np.testing.assert_array_equal(out.cpu().numpy(), ref)
            assert (lo, hi) == ref_min_max


# ------------------------------------------------------------------------------------------------
# c. window and stack kernel ranges, on occupancy
# ------------------------------------------------------------------------------------------------
def single_site(shape, site, filled=True):
    """Grid with one filled voxel at `site` (or one free voxel in a filled grid), and the exact
    squared distance of every other voxel to it."""
    occupancy = np.zeros(shape, dtype=np.float32)
    occupancy[site] = 1.0
    axes = np.ogrid[tuple(slice(0, n) for n in shape)]
    sq = sum((a - s).astype(np.int64) ** 2 for a, s in zip(axes, site))
    return (occupancy if filled else 1.0 - occupancy), sq


def sdf_host(occupancy, resolution, border=False, dtype=np.float32):
    sdf = make_map(occupancy, resolution).ExtractSignedDistanceField(params(True, border), dtype)
    return sdf.GetImmutableRawData(), sdf.GetMinimumMaximum()


def transposed(array, long_axis):
    # the long axis of the base [400, 48, 48] layout moves to x, y or z
    order = {0: (0, 1, 2), 1: (1, 0, 2), 2: (1, 2, 0)}[long_axis]
    return np.ascontiguousarray(array.transpose(order)), order


@pytest.mark.parametrize("long_axis", [0, 1, 2])
@pytest.mark.parametrize("corner", [True, False])
def test_window_ranges_on_a_single_site(shared_library, oracle, launched, long_axis, corner):
    base_site = (0, 0, 0) if corner else (200, 24, 24)
    occupancy, sq = single_site((400, 48, 48), base_site)
    values = np.unique(sq)
    # the exact results cross every range edge of the window kernel: (R + 1)^2 for R = 8, 10, 12,
    # and kSaturated (0x7800 itself is no sum of three squares that fits this grid)
    for edge in (81, 121, 169):
        assert {edge - 1, edge, edge + 1} <= set(values.tolist()), edge
    assert np.any((values >= SATURATED - 4) & (values < SATURATED))
    assert np.any((values >= SATURATED) & (values <= SATURATED + 4))
    # lines whose site is 160 - 185 rows away: the joint search cap (168 rows) lies in between
    offsets = np.abs(np.arange(400) - base_site[0])
    assert np.any(offsets == JOINT_SEARCH_CAP - 8) and np.any(offsets == 185)
    occupancy, order = transposed(occupancy, long_axis)
    sq = np.ascontiguousarray(sq.transpose(order))
    for filled in (True, False):
        grid = occupancy if filled else 1.0 - occupancy
        got_filled, got_free = vgt.ComputeSquaredDistanceFields(grid)
        np.testing.assert_array_equal(got_filled if filled else got_free, sq)
        want, want_min_max = oracle.sdf(grid, 0.02)
        for switches in ROUTES:
            with tuning(switches), launched() as kernels:
                got, got_min_max = sdf_host(grid, 0.02)
            np.testing.assert_array_equal(got, want)
            assert got_min_max == want_min_max
            assert_envelope_route(kernels, switches)
            y_routes, x_routes = occupancy_lean_routes(grid.shape)
            kernels.assert_lean_routes(0, y_routes)
            kernels.assert_lean_routes(1, x_routes)
        assert_matches_oracle(oracle, grid, 0.02, add_virtual_border=True)
        assert_matches_oracle(oracle, grid, 0.037, dtype=np.float64)


@pytest.mark.parametrize("resolution", [0.02, 0.037, 1.0 / 3.0])
def test_magnitude_table_edge(shared_library, oracle, launched, resolution):
    # squared distances just below, at and above 2^20, the size of the finalize table; above it the
    # kernel computes the magnitude in fp64 directly. 2^20 - 1 is 7 mod 8, never a sum of three
    # squares, so 2^20 - 2 is the largest value that can come from the table's last entries.
    occupancy, sq = single_site((1100, 20, 48), (0, 0, 0))
    largest = int(sq.max())
    assert largest + 1 > MAGNITUDE_TABLE_ENTRIES
    for value in (MAGNITUDE_TABLE_ENTRIES - 2, MAGNITUDE_TABLE_ENTRIES,
                  MAGNITUDE_TABLE_ENTRIES + 1):
        assert np.any(sq == value), value
    for grid in (occupancy, 1.0 - occupancy):
        for dtype in (np.float32, np.float64):
            for border in (False, True):
                want, want_min_max = oracle.sdf(grid, resolution, True, border, dtype=dtype)
                with launched() as kernels:
                    got, got_min_max = sdf_host(grid, resolution, border, dtype)
                np.testing.assert_array_equal(got, want)
                assert got_min_max == want_min_max
                kernels.assert_ran("BuildMagnitudeTableKernel<{}>".format(
                    "float" if dtype == np.float32 else "double"))
                kernels.assert_lean_routes(1 if dtype == np.float32 else 2,
                                           {lean_route(1100, 47 ** 2 + 19 ** 2)})
        want, want_min_max = oracle.sdf(grid, resolution)
        for switches in ROUTES[1:]:
            with tuning(switches), launched() as kernels:
                got, got_min_max = sdf_host(grid, resolution)
            np.testing.assert_array_equal(got, want)
            assert got_min_max == want_min_max
            assert_envelope_route(kernels, switches)


# ------------------------------------------------------------------------------------------------
# d. stack kernel and transform ranges, on sampled fields
# ------------------------------------------------------------------------------------------------
WINDOW_SAMPLES = [167, 168, 169, 0x77FE, 0x77FF, 0x7800]     # the kernels see sample + 1
WINDOW_DISTANCES = [0, 1, WINDOW_RADIUS_PACKED, WINDOW_RADIUS_PACKED + 1, JOINT_SEARCH_CAP,
                    JOINT_SEARCH_CAP + 1]


def window_sample_lines(rng, length, columns):
    """[length, columns] lines of +inf with sites whose values straddle (R + 1)^2 and kSaturated.
    Two equal sites 2 d + 1 rows apart make the minimum of the row d past the first come from the
    site exactly d rows away (0, 1, R, R + 1, 168, 169), the other site one row further."""
    lines = np.full((length, columns), np.inf)
    for c in range(columns):
        value = WINDOW_SAMPLES[c % len(WINDOW_SAMPLES)]
        d = WINDOW_DISTANCES[(c // len(WINDOW_SAMPLES)) % len(WINDOW_DISTANCES)]
        first = int(rng.integers(0, max(1, length - 2 * d - 1)))
        lines[first, c] = value
        if first + 2 * d + 1 < length:
            lines[first + 2 * d + 1, c] = value
        if c % 5 == 4:       # a smaller site elsewhere competes from further away
            lines[int(rng.integers(0, length)), c] = rng.choice(WINDOW_SAMPLES[:3])
    return lines


@pytest.mark.parametrize("switches", ROUTES, ids=lambda s: ",".join(f"{k}={v}" for k, v in
                                                                     s.items()) or "default")
def test_transform_window_thresholds(shared_library, oracle, launched, switches):
    checker = transform_checker(oracle)
    rng = np.random.default_rng(41)
    lines = window_sample_lines(rng, 400, 72)
    for field in (np.ascontiguousarray(lines.reshape(1, 400, 72)),      # y pass first
                  np.ascontiguousarray(lines[:, :36].reshape(400, 1, 36)),   # x pass first
                  np.ascontiguousarray(lines.T.reshape(2, 36, 400))):    # long z
        want = checker(field.copy())
        with tuning(switches), launched() as kernels:
            got = vgt.ComputeDistanceFieldTransformInPlace(field.copy())
        np.testing.assert_array_equal(got, want)
        assert_envelope_route(kernels, switches)
        kernels.assert_lean_routes(0, transform_lean_routes(field.shape, 0x7800))


@pytest.mark.parametrize("largest", [2_097_150, 2_097_151])
def test_transform_packed_against_split_entries(shared_library, oracle, launched, largest):
    # nx = 1: the y pass runs first and sees largest + 1 = 2^21 - 1 (packed) or 2^21 (split)
    checker = transform_checker(oracle)
    rng = np.random.default_rng(largest)
    shape = (1, 64, 33)
    field = rng.integers(0, 1000, size=shape).astype(np.float64)
    field[rng.random(shape) < 0.5] = np.inf
    field[0, rng.integers(0, 64, 8), rng.integers(0, 33, 8)] = largest
    field[0, 5, 7] = largest
    first_pass = lean_route(64, largest + 1)
    assert first_pass == ((True, False) if largest == 2_097_150 else (False, True))
    for switches in ({}, {"VGT_B200_ENVELOPE": "lean"}):
        with tuning(switches), launched() as kernels:
            got = vgt.ComputeDistanceFieldTransformInPlace(field.copy())
        np.testing.assert_array_equal(got, checker(field.copy()))
        kernels.assert_lean_routes(0, transform_lean_routes(shape, largest))
        assert not kernels.recorded or first_pass in kernels.lean_routes(0)


@pytest.mark.parametrize("largest", [1_050_621, 1_050_622])
def test_transform_pop_test_at_its_overflow_edge(shared_library, oracle, launched, largest):
    # L = 1024: (largest + 1 + 1023^2) * 1024 is 2^31 - 1024 (32-bit pops) or 2^31 (64-bit)
    checker = transform_checker(oracle)
    rng = np.random.default_rng(largest)
    shape = (1, 1024, 24)
    rows = np.arange(1024)
    field = np.full(shape, np.inf)
    field[0, :, 0] = np.where(rows % 2 == 0, 0, largest)            # alternating small, maximal
    field[0, :, 1] = np.where(rows % 2 == 1, 0, largest)
    field[0, :, 2] = largest
    field[0, 0, 2] = 0
    field[0, :, 3] = largest
    field[0, 1023, 3] = 0
    field[0, [0, 1023], 4] = largest
    field[0, 511, 4] = 3
    field[0, :, 5] = np.where(rng.random(1024) < 0.5, largest, np.inf)
    field[0, :, 6:] = np.where(rng.random((1024, 18)) < 0.3, largest,
                               rng.integers(0, 50, (1024, 18)))
    narrow = largest == 1_050_621
    assert lean_route(1024, largest + 1) == (narrow, False)
    with tuning({"VGT_B200_ENVELOPE": "lean"}), launched() as kernels:
        got = vgt.ComputeDistanceFieldTransformInPlace(field.copy())
    np.testing.assert_array_equal(got, checker(field.copy()))
    kernels.assert_lean_routes(0, transform_lean_routes(shape, largest))
    assert not kernels.recorded or (narrow, False) in kernels.lean_routes(0)


@pytest.mark.parametrize("nz", [1025, 1026])
def test_occupancy_pop_test_at_its_overflow_edge(shared_library, oracle, launched, nz):
    # y lines of 1024 voxels with inputs up to (nz - 1)^2: 32-bit pops for nz = 1025, 64-bit for
    # nz = 1026; z lines with their filled voxel at z = 0 or z = nz - 1, some lines empty
    shape = (1, 1024, nz)
    occupancy = np.zeros(shape, dtype=np.float32)
    occupancy[0, 0::2, 0] = 1.0
    occupancy[0, 1::2, nz - 1] = 1.0
    occupancy[0, 300:340, :] = 0.0
    occupancy[0, 700, :] = 0.0
    assert lean_route(1024, (nz - 1) ** 2) == (nz == 1025, False)
    y_routes, x_routes = occupancy_lean_routes(shape)
    for switches in ({"VGT_B200_ENVELOPE": "lean"}, {}):
        with tuning(switches), launched() as kernels:
            assert_matches_oracle(oracle, occupancy, 0.02)
        kernels.assert_lean_routes(0, y_routes)
        kernels.assert_lean_routes(1, x_routes)
    got_filled, got_free = vgt.ComputeSquaredDistanceFields(occupancy)
    want_filled, want_free = oracle.edt_squared(occupancy)
    np.testing.assert_array_equal(got_free, squared_to_int(want_free))
    np.testing.assert_array_equal(got_filled, squared_to_int(want_filled))


@pytest.mark.parametrize("shape", [(3, 4, 5), (2, 9, 40), (1, 1, 7)])
def test_transform_range_edge(shared_library, oracle, shape):
    # the last accepted sample is exact, the first refused one raises and leaves the field as it was
    checker = transform_checker(oracle)
    spread = sum((n - 1) ** 2 for n in shape)
    last = TRANSFORM_MAX_INPUT - 1 - spread
    rng = np.random.default_rng(sum(shape))
    field = rng.integers(0, 100, size=shape).astype(np.float64)
    field[rng.random(shape) < 0.3] = np.inf
    field.flat[len(field.flat) // 2] = last
    want = checker(field.copy())
    np.testing.assert_array_equal(vgt.ComputeDistanceFieldTransformInPlace(field.copy()), want)
    field.flat[len(field.flat) // 2] = last + 1
    before = field.copy()
    with pytest.raises(NotImplementedError):
        vgt.ComputeDistanceFieldTransformInPlace(field)
    np.testing.assert_array_equal(field, before)


# ------------------------------------------------------------------------------------------------
# e. axis limit
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("long_axis", [0, 1, 2])
def test_longest_axis(shared_library, oracle, launched, long_axis):
    import torch
    from voxelized_geometry_tools_b200 import device as vdev
    rng = np.random.default_rng(long_axis)
    base = random_occupancy(rng, (MAX_AXIS, 2, 3), 0.2, blobs=True)
    base[MAX_AXIS // 4:] = 0.0                      # blobs in the first quarter ...
    base[MAX_AXIS - 1, 1, 2] = 1.0                  # ... and one site at the far end
    order = {0: (0, 1, 2), 1: (2, 0, 1), 2: (1, 2, 0)}[long_axis]
    occupancy = np.ascontiguousarray(base.transpose(order))
    assert occupancy.shape[long_axis] == MAX_AXIS
    with launched() as kernels:
        assert_matches_oracle(oracle, occupancy, 0.01)
    y_routes, x_routes = occupancy_lean_routes(occupancy.shape)
    kernels.assert_lean_routes(0, y_routes)
    kernels.assert_lean_routes(1, x_routes)
    kernels.assert_ran(scan_kernel(occupancy.shape[2], "Float4Source"))
    assert_matches_oracle(oracle, occupancy, 0.01, False, True, np.float64)
    mask = occupancy > 0.5
    sizes = vgt.VoxelGridSizes.FromVoxelCounts(0.01, mask.shape)
    sdf = vgt.ExtractSignedDistanceFieldFromMask(mask, IDENTITY, "f", sizes, params())
    np.testing.assert_array_equal(sdf.GetImmutableRawData(), oracle.sdf_from_mask(mask, 0.01)[0])

    # one voxel more is refused before anything is launched
    lib = _capi.library()
    shape = list(occupancy.shape)
    shape[long_axis] = MAX_AXIS + 1
    too_long = np.zeros(shape, dtype=np.float32)
    out = np.empty(shape, dtype=np.float32)
    lo, hi = ctypes.c_float(), ctypes.c_float()
    launches = lib.vgt_b200_kernel_launch_count()
    assert lib.vgt_b200_sdf_f32(too_long.ctypes.data, *shape, 0.01, 1, 0, 0, out.ctypes.data,
                                ctypes.byref(lo), ctypes.byref(hi)) == _capi.ERR_INVALID_ARGUMENT
    with pytest.raises(ValueError):
        make_map(too_long, 0.01).ExtractSignedDistanceField(params())
    with pytest.raises(ValueError):
        vgt.ExtractSignedDistanceFieldFromMask(
            too_long > 0, IDENTITY, "f", vgt.VoxelGridSizes.FromVoxelCounts(0.01, shape), params())
    with pytest.raises(ValueError):
        vgt.ComputeSquaredDistanceFields(too_long)
    with pytest.raises(ValueError):
        vdev.signed_distance_field(torch.from_numpy(too_long).to(torch.device("cuda", 0)), 0.01)
    torch.cuda.synchronize()
    assert lib.vgt_b200_kernel_launch_count() == launches


# ------------------------------------------------------------------------------------------------
# f. pipelined host entry
# ------------------------------------------------------------------------------------------------
def boxes(rng, shape, count=40):
    """Filled boxes of random extent plus sparse noise; cheap to build at 2^24 voxels."""
    occupancy = np.zeros(shape, dtype=np.float32)
    for _ in range(count):
        low = [int(rng.integers(0, n)) for n in shape]
        high = [min(n, lo + int(rng.integers(1, max(2, n // 6)))) for lo, n in zip(low, shape)]
        occupancy[low[0]:high[0], low[1]:high[1], low[2]:high[2]] = 1.0
    flat = occupancy.reshape(-1)
    flat[rng.integers(0, flat.size, flat.size // 5000)] = 0.5
    return occupancy


def expected_pipeline_launches(shape):
    nx, ny, nz = shape
    pipelined = nx * ny * nz >= PIPELINE_MIN_VOXELS and nx > 1
    slabs_in = min(nx, PIPELINE_CHUNKS) if pipelined else 1
    slabs_out = min(ny, PIPELINE_CHUNKS) if pipelined else 1
    return pipelined, slabs_in, (slabs_in if ny > 1 else 0), slabs_out


@pytest.mark.parametrize("shape,dtypes", [
    ((256, 256, 256), (np.float32,)),             # 2^24 voxels: pipelined
    ((255, 241, 273), (np.float32,)),             # 2^24 - 1: the one-shot host path
    ((2, 4096, 2048), (np.float32, np.float64)),  # two x-slabs in
    ((7, 2400, 1000), (np.float32,)),             # seven x-slabs in
    ((2048, 3, 2731), (np.float32,)),             # three y-slabs out, scalar z scan
    ((4096, 1, 4096), (np.float32, np.float64)),  # no y axis: the z scan writes the packed field
])
def test_pipelined_host_entry_edges(shared_library, oracle, launched, shape, dtypes):
    rng = np.random.default_rng(sum(shape))
    occupancy = boxes(rng, shape)
    assert (int(np.prod(shape)) >= PIPELINE_MIN_VOXELS) == (shape != (255, 241, 273))
    pipelined, scans, y_passes, x_passes = expected_pipeline_launches(shape)
    for dtype in dtypes:
        border = dtype == np.float64
        with launched() as kernels:
            assert_matches_oracle(oracle, occupancy, 0.03, add_virtual_border=border, dtype=dtype)
        if kernels.recorded:
            mode = 1 if dtype == np.float32 else 2
            assert kernels.count("ScanContiguousAxis") == scans, sorted(kernels.items())
            assert kernels.count("EnvelopeAxisLeanKernel<0,") == y_passes, sorted(kernels.items())
            assert kernels.count(f"EnvelopeAxisLeanKernel<{mode},") == x_passes, \
                sorted(kernels.items())


def test_pipelined_mask_host_entry(shared_library, oracle, launched):
    rng = np.random.default_rng(3)
    shape = (256, 256, 256)
    mask = mask_values(rng, boxes(rng, shape) > 0.5)
    sizes = vgt.VoxelGridSizes.FromVoxelCounts(0.03, shape)
    _, scans, y_passes, x_passes = expected_pipeline_launches(shape)
    for border in (False, True):
        with launched() as kernels:
            sdf = vgt.ExtractSignedDistanceFieldFromMask(mask, IDENTITY, "f", sizes,
                                                         params(add_virtual_border=border))
        want, (lo, hi) = oracle.sdf_from_mask(mask != 0, 0.03, border)
        np.testing.assert_array_equal(sdf.GetImmutableRawData(), want)
        assert sdf.GetMinimumMaximum() == (lo, hi)
        if kernels.recorded:
            assert kernels.count("ScanContiguousAxisRegistersKernel<Uchar4Source, 2>") == scans
            assert kernels.count("EnvelopeAxisLeanKernel<0,") == y_passes
            assert kernels.count("EnvelopeAxisLeanKernel<1,") == x_passes
