"""GPU: the CUDA SDF path, called through the C-ABI, against the oracle and the reference goldens.

Bar: squared voxel distances bit-exact; float / double SDF bit-exact (0 ulp; the north star allows
1 ulp), min/max exact."""
import itertools

import numpy as np
import pytest

import voxelized_geometry_tools_b200 as vgt
from voxelized_geometry_tools_b200 import _capi

from .conftest import occupancy_from_golden_case, random_occupancy

pytestmark = pytest.mark.gpu

IDENTITY = np.eye(4)


def make_map(occupancy, resolution):
    sizes = vgt.VoxelGridSizes.FromVoxelCounts(resolution, occupancy.shape)
    return vgt.OccupancyMap(IDENTITY, "test_frame", sizes, data=occupancy)


def params(unknown_is_filled=True, add_virtual_border=False):
    return vgt.SignedDistanceFieldGenerationParameters(
        float("inf"), None, unknown_is_filled, add_virtual_border)


def squared_to_int(field):
    out = np.where(np.isinf(field), float(_capi.SQ_INF), field)
    return out.astype(np.int64)


def assert_matches_oracle(oracle, occupancy, resolution, unknown_is_filled=True,
                          add_virtual_border=False, dtype=np.float32):
    sdf = make_map(occupancy, resolution).ExtractSignedDistanceField(
        params(unknown_is_filled, add_virtual_border), dtype)
    want, (lo, hi) = oracle.sdf(occupancy, resolution, unknown_is_filled, add_virtual_border,
                                dtype=dtype)
    got = sdf.GetImmutableRawData()
    assert got.dtype == np.dtype(dtype)
    np.testing.assert_array_equal(got, want)
    assert sdf.IsLocked()
    got_lo, got_hi = sdf.GetMinimumMaximum()
    assert got_lo == lo and got_hi == hi


def test_reference_known_answers(shared_library, sdf_goldens, oracle):
    # Every case of test/sdf_generation_test.cpp, through the drop-in entry point.
    tolerance = sdf_goldens["extrema_tolerance"]
    for case in sdf_goldens["cases"]:
        occupancy, resolution = occupancy_from_golden_case(case)
        for dtype in (np.float32, np.float64):
            sdf = make_map(occupancy, resolution).ExtractSignedDistanceField(params(), dtype)
            data = sdf.GetImmutableRawData()
            if "expected_min_max" in case and case["expected_min_max"]:
                for got, want in zip(sdf.GetMinimumMaximum(), case["expected_min_max"]):
                    want = float(want)
                    assert got == want or abs(got - want) <= tolerance, case["name"]
                assert np.all(data[occupancy >= 0.5] < 0)
                assert np.all(data[occupancy < 0.5] > 0)
            for cell in case["expected_cells"]:
                x, y, z = cell["index"]
                if dtype == np.float32:
                    assert data[x, y, z] == np.float32(cell["value"]), (case["name"], cell)
        assert_matches_oracle(oracle, occupancy, resolution)


SHAPES = [(1, 1, 1), (1, 1, 2), (1, 1, 9), (1, 9, 1), (9, 1, 1), (2, 2, 2), (3, 1, 4), (1, 6, 6),
          (5, 7, 9), (8, 8, 8), (9, 10, 11), (4, 8, 12), (33, 31, 35), (64, 3, 70), (2, 100, 40),
          (130, 5, 33)]


@pytest.mark.parametrize("shape", SHAPES)
def test_squared_fields_bit_exact(shared_library, oracle, shape):
    rng = np.random.default_rng(abs(hash(shape)) % 2 ** 32)
    for fill, unknown_is_filled in itertools.product((0.0, 0.02, 0.3, 0.97, 1.0), (True, False)):
        occupancy = random_occupancy(rng, shape, fill)
        got_filled, got_free = vgt.ComputeSquaredDistanceFields(occupancy, unknown_is_filled)
        want_filled, want_free = oracle.edt_squared(occupancy, unknown_is_filled)
        np.testing.assert_array_equal(got_filled, squared_to_int(want_filled))
        np.testing.assert_array_equal(got_free, squared_to_int(want_free))


@pytest.mark.parametrize("shape", SHAPES)
def test_sdf_bit_exact_small(shared_library, oracle, shape):
    rng = np.random.default_rng(abs(hash(shape)) % 2 ** 32 + 1)
    for fill in (0.0, 0.1, 0.6, 1.0):
        occupancy = random_occupancy(rng, shape, fill)
        for border in (False, True):
            assert_matches_oracle(oracle, occupancy, 0.25, True, border)
        assert_matches_oracle(oracle, occupancy, 0.02, False, False)
        assert_matches_oracle(oracle, occupancy, 0.037, True, True, np.float64)


def test_single_voxel_and_single_hole(shared_library, oracle):
    occupancy = np.zeros((21, 17, 40), dtype=np.float32)
    occupancy[10, 8, 20] = 1.0
    assert_matches_oracle(oracle, occupancy, 0.1)
    assert_matches_oracle(oracle, 1.0 - occupancy, 0.1)
    assert_matches_oracle(oracle, 1.0 - occupancy, 0.1, add_virtual_border=True)


@pytest.mark.parametrize("shape,fill", [((128, 128, 128), 0.1), ((96, 160, 200), 0.02),
                                        ((256, 64, 300), 0.5)])
def test_sdf_bit_exact_medium(shared_library, oracle, shape, fill):
    rng = np.random.default_rng(17)
    occupancy = random_occupancy(rng, shape, fill, blobs=True)
    assert_matches_oracle(oracle, occupancy, 0.02)
    assert_matches_oracle(oracle, occupancy, 0.02, add_virtual_border=True)


def test_config1_box_scene(shared_library, oracle):
    from voxelized_geometry_tools_b200 import synthetic
    assert_matches_oracle(oracle, synthetic.box_scene(128), 0.02)


def test_long_axis_uses_wide_entries(shared_library, oracle):
    # > 1024 voxels along y and x forces the 8-byte stack entries and narrower tiles.
    rng = np.random.default_rng(23)
    occupancy = random_occupancy(rng, (6, 1500, 40), 0.05, blobs=True)
    assert_matches_oracle(oracle, occupancy, 0.01)
    assert_matches_oracle(oracle, np.ascontiguousarray(occupancy.transpose(1, 0, 2)), 0.01)
    assert_matches_oracle(oracle, np.ascontiguousarray(occupancy.transpose(0, 2, 1)), 0.01)


def test_mask_entry_point(shared_library, oracle):
    rng = np.random.default_rng(29)
    occupancy = random_occupancy(rng, (20, 30, 40), 0.2, blobs=True)
    mask = occupancy > 0.5
    sizes = vgt.VoxelGridSizes.FromVoxelCounts(0.05, mask.shape)
    for border in (False, True):
        sdf = vgt.ExtractSignedDistanceFieldFromMask(mask, IDENTITY, "f", sizes,
                                                     params(add_virtual_border=border))
        want, (lo, hi) = oracle.sdf_from_mask(mask, 0.05, border)
        np.testing.assert_array_equal(sdf.GetImmutableRawData(), want)
        assert sdf.GetMinimumMaximum() == (lo, hi)


def test_invalid_arguments_raise_value_error(shared_library):
    lib = _capi.library()
    occupancy = np.zeros((2, 2, 2), dtype=np.float32)
    out = np.zeros((2, 2, 2), dtype=np.float32)
    assert lib.vgt_b200_sdf_f32(occupancy.ctypes.data, 2, 2, 2, -1.0, 1, 0, 0, out.ctypes.data,
                                None, None) == _capi.ERR_INVALID_ARGUMENT
    assert "resolution" in _capi.last_error()
    assert lib.vgt_b200_sdf_f32(occupancy.ctypes.data, 0, 2, 2, 1.0, 1, 0, 0, out.ctypes.data,
                                None, None) == _capi.ERR_INVALID_ARGUMENT
    assert lib.vgt_b200_sdf_f32(None, 2, 2, 2, 1.0, 1, 0, 0, out.ctypes.data,
                                None, None) == _capi.ERR_INVALID_ARGUMENT
    assert lib.vgt_b200_sdf_f32(occupancy.ctypes.data, 2, 2, 2, 1.0, 1, 0, 99, out.ctypes.data,
                                None, None) == _capi.ERR_DEVICE


def test_full_size_512_properties_and_parity(shared_library, oracle):
    """BASELINE config 2 at full size: size-independent properties first, then full parity."""
    from voxelized_geometry_tools_b200 import synthetic
    occupancy = synthetic.clustered_spheres_occupancy((512, 512, 512))
    resolution = 0.02
    sdf = make_map(occupancy, resolution).ExtractSignedDistanceFieldFloat(params())
    data = sdf.GetImmutableRawData()
    filled = occupancy >= 0.5
    # sign == class, |d| >= one voxel, 1-Lipschitz along every axis (in voxel units)
    assert np.all(data[filled] < 0) and np.all(data[~filled] > 0)
    assert np.abs(data).min() == np.float32(resolution)
    for axis in range(3):
        step = np.abs(np.diff(data.astype(np.float64), axis=axis))
        same = np.diff(filled.astype(np.int8), axis=axis) == 0
        # float32 rounding of two values near 17 m: 2 * spacing(16) on top of one voxel
        assert step[same].max() <= resolution + 4e-6
    # idempotence: re-running the SDF on the sign of the SDF gives the same field
    again = make_map((data < 0).astype(np.float32), resolution).ExtractSignedDistanceFieldFloat(
        params())
    np.testing.assert_array_equal(again.GetImmutableRawData(), data)
    # and the full-size oracle comparison (tens of seconds of CPU)
    want, (lo, hi) = oracle.sdf(occupancy, resolution)
    np.testing.assert_array_equal(data, want)
    assert sdf.GetMinimumMaximum() == (lo, hi)


@pytest.mark.parametrize("shape", [(5, 9, 128), (4, 7, 132), (6, 5, 256), (3, 11, 640),
                                   (2, 6, 1024), (3, 5, 1028), (4, 6, 98)])
def test_z_scan_variants(shared_library, oracle, shape):
    # z lengths that select each z-scan kernel: 1, 2, 4 and 8 register iterations (<= 1024
    # voxels, multiple of 4), the shared-memory 128-bit kernel (> 1024) and the scalar one
    # (length not a multiple of 4).
    rng = np.random.default_rng(shape[2])
    for fill in (0.02, 0.4):
        occupancy = random_occupancy(rng, shape, fill, blobs=True)
        assert_matches_oracle(oracle, occupancy, 0.05)
    empty = np.zeros(shape, dtype=np.float32)
    assert_matches_oracle(oracle, empty, 0.05)
    empty[0, 0, shape[2] - 1] = 1.0
    assert_matches_oracle(oracle, empty, 0.05)


def test_long_axes_through_the_lean_kernel(shared_library, oracle):
    # y and x lines of 2048+ voxels: split stack entries (f in the row, position in the side
    # array), 64-bit pop test, class words for 64+ words per line.
    rng = np.random.default_rng(43)
    base = random_occupancy(rng, (3, 2300, 36), 0.04, blobs=True)
    assert_matches_oracle(oracle, base, 0.02)
    assert_matches_oracle(oracle, np.ascontiguousarray(base.transpose(1, 0, 2)), 0.02,
                          add_virtual_border=True)


def test_pipelined_host_entry_odd_shape(shared_library, oracle):
    # >= 2^24 voxels: the host entry overlaps the slab copies with the passes (x-slabs in,
    # y-slabs out as strided 2-D copies). Odd extents so that no slab boundary is aligned.
    rng = np.random.default_rng(37)
    occupancy = random_occupancy(rng, (70, 515, 470), 0.05, blobs=True)
    assert occupancy.size >= 2 ** 24
    assert_matches_oracle(oracle, occupancy, 0.03)
    assert_matches_oracle(oracle, occupancy, 0.03, add_virtual_border=True, dtype=np.float64)


def test_axes_longer_than_1024_and_large_distances(shared_library, oracle):
    # > 1024 voxels along an axis (or partial distances >= 2^21) switches the envelope kernel to
    # split stack entries (value in place, position in a uint16 side array).
    rng = np.random.default_rng(31)
    base = random_occupancy(rng, (5, 1100, 37), 0.03, blobs=True)
    assert_matches_oracle(oracle, base, 0.01)                                           # y long
    assert_matches_oracle(oracle, np.ascontiguousarray(base.transpose(1, 0, 2)), 0.01)  # x long
    assert_matches_oracle(oracle, np.ascontiguousarray(base.transpose(0, 2, 1)), 0.01,
                          add_virtual_border=True)                                      # z long
    sparse = np.zeros((3, 40, 2100), dtype=np.float32)   # z distances up to 2099 -> sq > 2^21
    sparse[1, 20, 0] = 1.0
    assert_matches_oracle(oracle, sparse, 0.5)


def test_drop_in_equals_the_references_own_occupancy_map_member(shared_library):
    # OccupancyMap::ExtractSignedDistanceField<T> on the reference's own class (its
    # occupancy_map.hpp / .cpp compiled unmodified into oracle/_ref/libvgt_ref_maps.so) against
    # the same call on the device: values, extrema, both scalar types, both predicates, border.
    from oracle import reference_oracle
    if not reference_oracle.maps_available():
        pytest.skip("oracle/_ref/libvgt_ref_maps.so not built")
    rng = np.random.default_rng(77)
    for shape in ((40, 36, 70), (7, 130, 33)):
        occupancy = random_occupancy(rng, shape, 0.08, unknown=0.1, blobs=True)
        for unknown_is_filled, border, dtype in ((True, False, np.float32),
                                                 (False, True, np.float32),
                                                 (True, True, np.float64)):
            want, (lo, hi) = reference_oracle.occupancy_map_sdf(
                occupancy, 0.05, unknown_is_filled, border, dtype=dtype)
            sdf = make_map(occupancy, 0.05).ExtractSignedDistanceField(
                params(unknown_is_filled, border), dtype)
            np.testing.assert_array_equal(sdf.GetImmutableRawData(), want)
            assert sdf.GetMinimumMaximum() == (lo, hi)


@pytest.mark.parametrize("nz", [1028, 1536, 2044, 2048])
def test_register_z_scan_with_two_words_per_lane(shared_library, oracle, nz):
    # z lines of 1025 .. 2048 voxels: the register scan keeps two words per lane ("halves");
    # the last voxel of a class in the first half precedes every word of the second and the
    # first one of the second half follows every word of the first. Lines whose only
    # opposite-class voxel sits right at the boundary (voxels 1023 / 1024), at the ends, or
    # nowhere; plus random lines.
    rng = np.random.default_rng(nz)
    occupancy = random_occupancy(rng, (3, 9, nz), 0.02, blobs=True)
    occupancy[0, 0, :] = 0.0
    occupancy[0, 0, 1023] = 1.0
    occupancy[0, 1, :] = 0.0
    occupancy[0, 1, 1024] = 1.0
    occupancy[0, 2, :] = 1.0
    occupancy[0, 2, 1024] = 0.0
    occupancy[0, 3, :] = 0.0
    occupancy[0, 3, 0] = 1.0
    occupancy[0, 4, :] = 0.0
    occupancy[0, 4, nz - 1] = 1.0
    occupancy[0, 5, :] = 1.0
    occupancy[0, 6, :] = 0.0
    occupancy[0, 7, :1024] = 1.0
    occupancy[0, 7, 1024:] = 0.0
    got_filled, got_free = vgt.ComputeSquaredDistanceFields(occupancy, True)
    want_filled, want_free = oracle.edt_squared(occupancy, True)
    np.testing.assert_array_equal(got_filled, squared_to_int(want_filled))
    np.testing.assert_array_equal(got_free, squared_to_int(want_free))
    assert_matches_oracle(oracle, occupancy, 0.02)


@pytest.mark.parametrize("shape", [(1, 1, 1), (1, 1, 40), (9, 1, 7), (1, 33, 5), (11, 14, 9),
                                   (40, 36, 70), (3, 130, 33), (64, 64, 64)])
def test_transform_in_place_on_sampled_functions(shared_library, oracle, shape):
    # vgt_b200_edt_transform_inplace_f64 == ComputeDistanceFieldTransformInPlace
    # (sdfgen.hpp:34-37) on arbitrary integer / +inf samples, against the reference's own code
    # where oracle/_ref is there, else the restatement.
    from oracle import reference_oracle
    checker = reference_oracle.transform_inplace if reference_oracle.available() \
        else oracle.transform_inplace
    rng = np.random.default_rng(sum(shape))
    for scale, inf_rate in ((1, 0.0), (400, 0.3), (50000, 0.9), (7, 1.0), (3, 0.97)):
        field = rng.integers(0, scale + 1, size=shape).astype(np.float64)
        field[rng.random(shape) < inf_rate] = np.inf
        want = checker(field.copy())
        got = vgt.ComputeDistanceFieldTransformInPlace(field.copy())
        np.testing.assert_array_equal(got, want)
    # the binary 0 / inf marks of the SDF path
    marks = np.where(rng.random(shape) < 0.05, 0.0, np.inf)
    np.testing.assert_array_equal(vgt.ComputeDistanceFieldTransformInPlace(marks.copy()),
                                  checker(marks.copy()))


def test_transform_in_place_rejects_what_it_cannot_do_exactly(shared_library):
    field = np.full((4, 4, 4), 2.5)
    before = field.copy()
    with pytest.raises(NotImplementedError):
        vgt.ComputeDistanceFieldTransformInPlace(field)
    np.testing.assert_array_equal(field, before)
    with pytest.raises(NotImplementedError):
        vgt.ComputeDistanceFieldTransformInPlace(np.full((4, 4, 4), -1.0))
    with pytest.raises(NotImplementedError):
        vgt.ComputeDistanceFieldTransformInPlace(np.full((4, 4, 4), 2.0 ** 30))
    with pytest.raises(ValueError):
        vgt.ComputeDistanceFieldTransformInPlace(np.zeros((4, 4), dtype=np.float64))


def test_bench_dumps_the_sdf_of_its_last_timed_step(shared_library, oracle, tmp_path):
    # bench.py --dump-outputs end to end: the sampled SDF and its min/max equal the oracle's SDF
    # of the bench grid at the sampled positions
    import subprocess
    import sys
    from pathlib import Path

    import torch
    from voxelized_geometry_tools_b200 import synthetic
    repo = Path(__file__).resolve().parents[1]
    result = subprocess.run(
        [sys.executable, str(repo / "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
         "--skip-cpu", "--skip-voxelizer", "--skip-strong", "--dump-outputs", str(tmp_path)],
        capture_output=True, text=True, timeout=1200)
    assert result.returncode == 0, result.stderr[-3000:]
    dims = (512, 512, 512)
    occupancy = synthetic.clustered_spheres_occupancy_torch(dims, torch.device("cuda", 0)).cpu()
    want, (lo, hi) = oracle.sdf(occupancy.numpy(), 0.02)
    index = np.load(tmp_path / "sdf_sample_index.npy").astype(np.int64)
    assert len(index) > 3_000_000
    np.testing.assert_array_equal(np.load(tmp_path / "sdf_sample.npy"), want.reshape(-1)[index])
    np.testing.assert_array_equal(np.load(tmp_path / "sdf_min_max.npy"),
                                  np.array([lo, hi], dtype=np.float32))
