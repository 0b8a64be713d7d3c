"""CPU: the SignedDistanceField<double> query restatement (oracle/sdf_queries_oracle_f64.py) and
the argument checks of the query entries, which refuse a bad call before any device call.

The double restatement differs from the float one in two statements only (the interior
gradient's subtraction and the sign test of the extrema walk). So on a field of
float32-representable values whose neighbour differences are exact it must give the float
results; on a general double field its interior gradient must be the plain double expression."""
import ctypes

import numpy as np
import pytest

from oracle import sdf_queries_oracle
from oracle.sdf_queries_oracle_f64 import SdfOracle
from tests.test_gpu_sdf_queries import _posed, _world_points
from voxelized_geometry_tools_b200 import _capi


def exact_field(rng, dims):
    """Multiples of 1/256 below 4 in magnitude (at most 10 significant bits), so every value
    and every difference of two values is exact in float32; about 10 % exact zeros."""
    field = np.round(rng.normal(size=dims) * 0.3 * 256) / 256
    field[rng.random(dims) < 0.1] = 0.0
    return field


def sphere_field(dims, res):
    """A sphere's signed distance rounded to multiples of 1/1024 (exact in float32)."""
    index = np.indices(dims).transpose(1, 2, 3, 0)
    centre = (np.array(dims) * res) / 2.0
    distance = np.linalg.norm((index + 0.5) * res - centre, axis=-1) - 0.25 * min(dims) * res
    return np.round(distance * 1024) / 1024


def all_queries(checker, points):
    return {
        "distance": [checker.estimate_distance(p) for p in points],
        "coarse": [checker.coarse_gradient(p, False) for p in points],
        "coarse_edge": [checker.coarse_gradient(p, True) for p in points],
        "fine": [checker.fine_gradient(p, 0.04) for p in points],
        "fine_too_large": [checker.fine_gradient(p, 0.5) for p in points[:50]],
        "project": [checker.project_out_of_collision(p, 0.02, 0.25, 500) for p in points[:150]],
    }


def test_double_oracle_equals_float_oracle_on_exact_values():
    rng = np.random.default_rng(4)
    dims, res = (12, 10, 11), 0.1
    pose = _posed(rng)
    field = sphere_field(dims, res)
    assert np.array_equal(field.astype(np.float32).astype(np.float64), field)
    points = _world_points(rng, pose, dims, res, 400)
    single = sdf_queries_oracle.SdfOracle(field, res, pose)
    double = SdfOracle(field, res, pose, dtype=np.float64)
    assert double.sdf.dtype == np.float64
    want, got = all_queries(single, points), all_queries(double, points)
    for name in want:
        assert got[name] == want[name], name
    assert any(status == 1 for status, _ in want["project"])
    np.testing.assert_array_equal(double.local_extrema_map(), single.local_extrema_map())


@pytest.mark.parametrize("seed", [0, 1])
def test_double_extrema_map_equals_float_on_exact_values(seed):
    rng = np.random.default_rng(seed)
    field = exact_field(rng, (9, 8, 10))
    pose = _posed(rng)
    single = sdf_queries_oracle.SdfOracle(field, 0.1, pose)
    double = SdfOracle(field, 0.1, pose, dtype=np.float64)
    np.testing.assert_array_equal(double.local_extrema_map(), single.local_extrema_map())


def test_interior_coarse_gradient_is_the_double_expression():
    rng = np.random.default_rng(7)
    dims, res = (9, 10, 8), 0.05
    field = rng.normal(size=dims)
    field[4, 5, 3], field[6, 5, 3] = 1.0 - 1e-9, 1.0          # equal after rounding to float
    pose = _posed(rng)
    double = SdfOracle(field, res, pose, dtype=np.float64)
    single = SdfOracle(field, res, pose)
    scale = 1.0 / (2.0 * res)
    inner = (slice(1, -1),) * 3
    aligned = [(field[2:, 1:-1, 1:-1] - field[:-2, 1:-1, 1:-1]) * scale,
               (field[1:-1, 2:, 1:-1] - field[1:-1, :-2, 1:-1]) * scale,
               (field[1:-1, 1:-1, 2:] - field[1:-1, 1:-1, :-2]) * scale]
    want = np.stack([((pose[r, 0] * aligned[0] + pose[r, 1] * aligned[1]) + pose[r, 2] * aligned[2])
                     + pose[r, 3] * 0.0 for r in range(3)], axis=-1)
    differs = 0
    for x, y, z in np.ndindex(*field[inner].shape):
        status, got = double.coarse_gradient_at_index(x + 1, y + 1, z + 1, False)
        assert status == 1
        assert got == want[x, y, z].tolist(), (x, y, z)
        differs += got != single.coarse_gradient_at_index(x + 1, y + 1, z + 1, False)[1]
    assert differs > 0.9 * want[..., 0].size
    # the cell between the two values that float cannot tell apart: float sees a 0 difference
    x_axis = np.linalg.solve(pose[:3, :3], np.array(double.coarse_gradient_at_index(5, 5, 3,
                                                                                   False)[1]))
    assert abs(x_axis[0] - (1e-9 * scale)) < 1e-15
    single_x = np.linalg.solve(pose[:3, :3], np.array(single.coarse_gradient_at_index(5, 5, 3,
                                                                                     False)[1]))
    assert abs(single_x[0]) < 1e-15


def test_tiny_negative_values_keep_their_sign():
    # -1e-300 is negative in double (the walk goes downhill, the half cell is added) and -0.0 in
    # float (uphill, the half cell subtracted)
    field = np.zeros((5, 5, 5))
    field[:, :, :] = np.arange(5, dtype=np.float64)[:, None, None] * 0.5
    field[2, 2, 2] = -1e-300
    double = SdfOracle(field, 0.1, np.eye(4), dtype=np.float64)
    single = SdfOracle(field, 0.1, np.eye(4))
    g = double.coarse_gradient_at_index(2, 2, 2, True)[1]
    assert g[0] > 0
    assert double._next_from_gradient((2, 2, 2), g) == (1, 2, 2)
    assert single._next_from_gradient((2, 2, 2), g) == (3, 2, 2)
    assert double._corrected(2, 2, 2) == 0.05
    assert single._corrected(2, 2, 2) == -0.05


def test_default_scalar_type_is_float32():
    rng = np.random.default_rng(3)
    field = rng.normal(size=(6, 5, 4))
    checker = SdfOracle(field, 0.1)
    assert checker.sdf.dtype == np.float32
    np.testing.assert_array_equal(checker.sdf, sdf_queries_oracle.SdfOracle(field, 0.1).sdf)
    assert SdfOracle(field, 0.1, dtype="float64").sdf.dtype == np.float64
    for dtype in (np.float16, np.int32):
        with pytest.raises(ValueError):
            SdfOracle(field, 0.1, dtype=dtype)


# ---- argument checks of the C-ABI entries (no device is touched by a refused call)

SCALAR_TYPES = {"f32": (_capi.SdfView, "_dev"), "f64": (_capi.SdfViewF64, "_f64_dev")}
FAKE_DEVICE_POINTER = 0x10000          # never dereferenced: every call below is refused first


def _view(view_type, dims=(4, 5, 6), resolution=0.1, d_sdf=FAKE_DEVICE_POINTER):
    view = view_type()
    view.d_sdf = d_sdf
    view.nx, view.ny, view.nz = dims
    view.resolution = resolution
    view.origin_transform[0] = view.origin_transform[5] = view.origin_transform[10] = 1.0
    view.origin_transform[15] = 1.0
    return view


def _queries(lib, suffix, view, count=8, points=FAKE_DEVICE_POINTER):
    """Each query entry called with `view` (a ctypes view, or None); returns their codes."""
    out = valid = FAKE_DEVICE_POINTER
    reference = None if view is None else ctypes.byref(view)
    return [
        getattr(lib, "vgt_b200_sdf_estimate_distance" + suffix)(
            reference, points, count, 0, out, valid, None),
        getattr(lib, "vgt_b200_sdf_coarse_gradient" + suffix)(
            reference, points, count, 1, 0, out, valid, None),
        getattr(lib, "vgt_b200_sdf_fine_gradient" + suffix)(
            reference, points, count, 0.1, 0, out, valid, None),
        getattr(lib, "vgt_b200_sdf_project_out_of_collision" + suffix)(
            reference, points, count, 0.0, 0.1, 100, 0, out, valid, None),
    ]


def _extrema(lib, suffix, view, out=FAKE_DEVICE_POINTER):
    return getattr(lib, "vgt_b200_sdf_local_extrema_map" + suffix)(
        None if view is None else ctypes.byref(view), 0, out, None)


def _refused(code, message):
    assert code == _capi.ERR_INVALID_ARGUMENT
    assert message in _capi.last_error()


@pytest.mark.parametrize("scalar", sorted(SCALAR_TYPES))
def test_bad_views_are_refused(shared_library, scalar):
    lib = _capi.library()
    view_type, suffix = SCALAR_TYPES[scalar]
    bad = [(None, "null SDF view"), (_view(view_type, d_sdf=None), "null SDF view")]
    for dims in ((0, 5, 6), (4, -1, 6), (4, 5, 8193), (8193, 1, 1)):
        bad.append((_view(view_type, dims=dims), "dimensions out of range"))
    for resolution in (0.0, -0.1, float("nan"), float("inf"), -float("inf")):
        bad.append((_view(view_type, resolution=resolution), "positive and finite"))
    for view, message in bad:
        for code in _queries(lib, suffix, view):
            _refused(code, message)
        _refused(_extrema(lib, suffix, view), message)


@pytest.mark.parametrize("scalar", sorted(SCALAR_TYPES))
def test_bad_batches_are_refused(shared_library, scalar):
    lib = _capi.library()
    view_type, suffix = SCALAR_TYPES[scalar]
    view = _view(view_type)
    for code in _queries(lib, suffix, view, count=-1):
        _refused(code, "negative count")
    for code in _queries(lib, suffix, view, count=3, points=None):
        _refused(code, "null query buffer")
    for code in _queries(lib, suffix, view, count=0x7fffffff * 128 + 1):
        _refused(code, "too many query points")
    project = getattr(lib, "vgt_b200_sdf_project_out_of_collision" + suffix)
    for multiplier, steps in ((0.0, 10), (-1.0, 10), (float("nan"), 10), (0.1, 0)):
        _refused(project(ctypes.byref(view), FAKE_DEVICE_POINTER, 4, 0.0, multiplier, steps, 0,
                         FAKE_DEVICE_POINTER, FAKE_DEVICE_POINTER, None), "max_steps")
    # an empty batch returns before any device call, so it succeeds without a device
    assert _queries(lib, suffix, view, count=0, points=None) == [_capi.OK] * 4


@pytest.mark.parametrize("scalar", sorted(SCALAR_TYPES))
def test_extrema_map_refuses_2_31_cells(shared_library, scalar):
    lib = _capi.library()
    view_type, suffix = SCALAR_TYPES[scalar]
    for dims in ((8192, 8192, 32), (8192, 8192, 8192), (4096, 8192, 65)):
        _refused(_extrema(lib, suffix, _view(view_type, dims=dims)), "2^31 cells")
    _refused(_extrema(lib, suffix, _view(view_type), out=None), "null extrema buffer")


def test_view_types_are_not_interchangeable(shared_library):
    lib = _capi.library()
    with pytest.raises(ctypes.ArgumentError):
        lib.vgt_b200_sdf_local_extrema_map_f64_dev(ctypes.byref(_view(_capi.SdfView)), 0,
                                                   FAKE_DEVICE_POINTER, None)
    with pytest.raises(ctypes.ArgumentError):
        lib.vgt_b200_sdf_local_extrema_map_dev(ctypes.byref(_view(_capi.SdfViewF64)), 0,
                                               FAKE_DEVICE_POINTER, None)
