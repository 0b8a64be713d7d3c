"""GPU: the batched queries and the local extrema map on a device-resident
SignedDistanceField<double> (the float64 instantiation of csrc/sdf_queries.cu through the *_f64_dev
C-ABI entries) against the double restatement, oracle/sdf_queries_oracle_f64.py with
dtype=np.float64: equal values (NaN equals NaN, as in the float suite) and equal status bytes.

The fields with special values are chosen so that rounding them to float changes some result;
each such test first shows that on the oracle, so that it can tell the two scalar types apart."""
import numpy as np
import pytest

from tests.test_gpu_sdf_queries import _posed, _world_points
from voxelized_geometry_tools_b200 import synthetic

pytestmark = pytest.mark.gpu


def _double_oracle(field, res, pose):
    from oracle.sdf_queries_oracle_f64 import SdfOracle
    return SdfOracle(field, res, pose, dtype=np.float64)


def _rounded_oracle(field, res, pose):
    """The float oracle of the field rounded to float32 (what a float query would see)."""
    from oracle.sdf_queries_oracle_f64 import SdfOracle
    with np.errstate(over="ignore"):
        return SdfOracle(field.astype(np.float32), res, pose)


def _device_field(field, res, pose):
    import torch
    from voxelized_geometry_tools_b200 import device as vdev
    return vdev.DeviceSignedDistanceField(
        torch.from_numpy(np.ascontiguousarray(field, dtype=np.float64)).to("cuda:0"), res, pose)


def _to_device(points):
    import torch
    return torch.from_numpy(np.ascontiguousarray(points, dtype=np.float64)).to("cuda:0")


def _arrays(want):
    return (np.array([w[0] for w in want], dtype=np.uint8),
            np.array([w[1] for w in want], dtype=np.float64))


def _compare(got_values, got_valid, want):
    want_valid, want_values = _arrays(want)
    np.testing.assert_array_equal(got_valid.cpu().numpy(), want_valid)
    np.testing.assert_array_equal(got_values.cpu().numpy().reshape(want_values.shape),
                                  want_values)


def _differ(a, b):
    (status_a, values_a), (status_b, values_b) = _arrays(a), _arrays(b)
    return bool((status_a != status_b).any()) or not np.array_equal(values_a, values_b,
                                                                    equal_nan=True)


# ---- the scene of tests/test_gpu_sdf_queries.py, with the SDF generated as double

@pytest.fixture(scope="module")
def scene(shared_library):
    import torch
    from voxelized_geometry_tools_b200 import device as vdev
    rng = np.random.default_rng(11)
    dims, res = (28, 22, 25), 0.05
    occupancy = synthetic.clustered_spheres_occupancy(dims)
    sdf, _ = vdev.signed_distance_field_f64(torch.from_numpy(occupancy).to("cuda:0"), res)
    assert sdf.dtype == torch.float64
    pose = _posed(rng)
    field = sdf.cpu().numpy()
    points = _world_points(rng, pose, dims, res, 3000)
    return {"gpu": vdev.DeviceSignedDistanceField(sdf, res, pose),
            "oracle": _double_oracle(field, res, pose), "field": field, "points": points,
            "device_points": _to_device(points), "res": res, "pose": pose}


def test_scene_holds_double_values(scene):
    field = scene["field"]
    assert (field.astype(np.float32).astype(np.float64) != field).mean() > 0.5


def test_estimate_location_distance(scene):
    values, valid = scene["gpu"].EstimateLocationDistance(scene["device_points"])
    want = [scene["oracle"].estimate_distance(p) for p in scene["points"]]
    _compare(values, valid, want)
    assert 0.5 < np.mean([w[0] for w in want]) < 1.0
    rounded = _rounded_oracle(scene["field"], scene["res"], scene["pose"])
    assert _differ(want[:200], [rounded.estimate_distance(p) for p in scene["points"][:200]])


@pytest.mark.parametrize("edge", [False, True])
def test_coarse_gradient(scene, edge):
    values, valid = scene["gpu"].GetLocationCoarseGradient(scene["device_points"], edge)
    want = [scene["oracle"].coarse_gradient(p, edge) for p in scene["points"]]
    _compare(values, valid, want)


@pytest.mark.parametrize("window", [0.05, 0.013, 0.4])
def test_fine_gradient(scene, window):
    values, valid = scene["gpu"].GetLocationFineGradient(scene["device_points"][:1500], window)
    want = [scene["oracle"].fine_gradient(p, window) for p in scene["points"][:1500]]
    _compare(values, valid, want)
    statuses = {w[0] for w in want}
    if window == 0.4:
        assert 2 in statuses          # the window is too large along some axis: THROWS


@pytest.mark.parametrize("minimum_distance,multiplier", [(0.0, 0.1), (0.04, 0.25), (0.02, 0.5)])
def test_project_out_of_collision(scene, minimum_distance, multiplier):
    subset = scene["points"][:600]
    values, valid = scene["gpu"].ProjectLocationOutOfCollisionToMinimumDistance(
        scene["device_points"][:600], minimum_distance, multiplier, max_steps=20000)
    want = [scene["oracle"].project_out_of_collision(p, minimum_distance, multiplier, 20000)
            for p in subset]
    _compare(values, valid, want)
    moved = np.any(values.cpu().numpy() != subset, axis=1) & (valid.cpu().numpy() == 1)
    assert moved.sum() > 20
    again, ok = scene["gpu"].EstimateLocationDistance(values[valid == 1])
    assert bool((again[ok == 1] > minimum_distance).all())


def test_project_out_of_collision_runs_out_of_steps(scene):
    subset = scene["points"][:600]
    values, valid = scene["gpu"].ProjectLocationOutOfCollisionToMinimumDistance(
        scene["device_points"][:600], 0.04, 0.1, max_steps=3)
    want = [scene["oracle"].project_out_of_collision(p, 0.04, 0.1, 3) for p in subset]
    _compare(values, valid, want)
    assert sum(w[0] == 2 for w in want) > 20


def test_local_extrema_map_of_an_sdf(scene):
    got = scene["gpu"].ComputeLocalExtremaMap().cpu().numpy()
    want = scene["oracle"].local_extrema_map()
    np.testing.assert_array_equal(got, want)
    assert np.isinf(got).any() and np.isfinite(got).any()


# ---- fields whose float rounding changes results

def _exact_base(rng, dims):
    """Multiples of 1/256 below 4 in magnitude: exact in float32, and so are their differences."""
    return np.round(rng.normal(size=dims) * 0.3 * 256) / 256


def _tiny_field(rng, dims):
    # -1e-300 rounds to -0.0 in float: the half-cell correction and the walk's sign flip
    field = _exact_base(rng, dims)
    pick = rng.random(dims)
    field[pick < 0.15] = -1e-300
    field[(pick >= 0.15) & (pick < 0.2)] = 1e-300
    field[(pick >= 0.2) & (pick < 0.25)] = 0.0
    field[(pick >= 0.25) & (pick < 0.3)] = -0.0
    return field


def _close_field(rng, dims):
    # steps of 1e-9 on top of values near 1: far below float's spacing there (1.2e-7)
    return 1.0 + _exact_base(rng, dims) * 0.25 + rng.integers(-3, 4, dims) * 1e-9


def _infinite_field(rng, dims):
    # inf next to 1e300 and 3.5e38: both round to inf in float, where inf - inf is NaN
    field = _exact_base(rng, dims)
    field[2:5, 2:5, 2:5] = np.inf
    field[5, 2:5, 2:5] = 1e300
    field[1, 2:5, 2:5] = 3.5e38
    field[7:9, 5:8, 6:9] = -np.inf
    field[9, 5:8, 6:9] = -1e300
    field[6, 5:8, 6:9] = -3.5e38
    return field


SPECIAL_FIELDS = {"tiny": _tiny_field, "close": _close_field, "infinite": _infinite_field}


def _query_results(checker, points):
    return {
        "distance": [checker.estimate_distance(p) for p in points],
        "coarse": [checker.coarse_gradient(p, False) for p in points],
        "coarse_edge": [checker.coarse_gradient(p, True) for p in points],
        "fine": [checker.fine_gradient(p, 0.07) for p in points],
        "project": [checker.project_out_of_collision(p, 0.03, 0.25, 300) for p in points[:300]],
    }


@pytest.mark.parametrize("name", sorted(SPECIAL_FIELDS))
def test_fields_that_float_would_get_wrong(shared_library, name):
    rng = np.random.default_rng(sorted(SPECIAL_FIELDS).index(name) + 20)
    dims, res = (12, 10, 11), 0.1
    field = SPECIAL_FIELDS[name](rng, dims)
    pose = _posed(rng)
    points = _world_points(rng, pose, dims, res, 800)
    checker = _double_oracle(field, res, pose)
    want = _query_results(checker, points)
    want_extrema = checker.local_extrema_map()
    # the two scalar types are told apart on this field
    rounded = _rounded_oracle(field, res, pose)
    rounded_results = _query_results(rounded, points)
    assert (any(_differ(want[k], rounded_results[k]) for k in want)
            or not np.array_equal(want_extrema, rounded.local_extrema_map(), equal_nan=True))

    gpu = _device_field(field, res, pose)
    device_points = _to_device(points)
    _compare(*gpu.EstimateLocationDistance(device_points), want["distance"])
    _compare(*gpu.GetLocationCoarseGradient(device_points, False), want["coarse"])
    _compare(*gpu.GetLocationCoarseGradient(device_points, True), want["coarse_edge"])
    _compare(*gpu.GetLocationFineGradient(device_points, 0.07), want["fine"])
    _compare(*gpu.ProjectLocationOutOfCollisionToMinimumDistance(device_points[:300], 0.03, 0.25,
                                                                 300), want["project"])
    np.testing.assert_array_equal(gpu.ComputeLocalExtremaMap().cpu().numpy(), want_extrema)


def test_tiny_negative_cells_change_the_extrema_map(shared_library):
    # the sign test of the walk on its own: -1e-300 walks downhill in double, uphill in float
    field = np.repeat(np.arange(6, dtype=np.float64)[:, None, None] * 0.5, 5, axis=1)
    field = np.repeat(field, 5, axis=2)
    field[2:4, 1:4, 1:4] = -1e-300
    checker = _double_oracle(field, 0.1, np.eye(4))
    want = checker.local_extrema_map()
    assert not np.array_equal(want, _rounded_oracle(field, 0.1, np.eye(4)).local_extrema_map())
    got = _device_field(field, 0.1, np.eye(4)).ComputeLocalExtremaMap().cpu().numpy()
    np.testing.assert_array_equal(got, want)


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_local_extrema_map_with_loops(shared_library, seed):
    """The rough field of the float suite, drawn as double: walks that close loops."""
    rng = np.random.default_rng(seed)
    dims, res = (14, 11, 13), 0.1
    field = rng.normal(size=dims) * 0.3
    field[rng.random(dims) < 0.1] = 0.0
    if seed == 2:
        field[2:5, 2:5, 2:5] = np.inf      # inf - inf = NaN gradients: cells that stay put
    pose = _posed(rng) if seed else np.eye(4)
    checker = _double_oracle(field, res, pose)
    loops = 0
    for start in np.ndindex(*dims):
        seen, current = {start}, start
        while True:
            g = checker.coarse_gradient_at_index(*current, True)[1]
            if checker._effectively_flat(g):
                break
            current = checker._next_from_gradient(current, g)
            if not checker._in_bounds(current):
                break
            if current in seen:
                loops += 1
                break
            seen.add(current)
    assert loops > 20
    got = _device_field(field, res, pose).ComputeLocalExtremaMap().cpu().numpy()
    np.testing.assert_array_equal(got, checker.local_extrema_map())


# ---- float and double on the same exact values

def test_float_and_double_fields_agree_on_exact_values(shared_library):
    import torch
    from voxelized_geometry_tools_b200 import device as vdev
    rng = np.random.default_rng(5)
    dims, res = (20, 17, 19), 0.05
    index = np.indices(dims).transpose(1, 2, 3, 0)
    distance = np.linalg.norm((index + 0.5) * res - np.array(dims) * res / 2, axis=-1) - 0.3
    field = np.round(distance * 1024) / 1024 + _exact_base(rng, dims) / 64
    assert np.array_equal(field.astype(np.float32).astype(np.float64), field)
    pose = _posed(rng)
    points = _to_device(_world_points(rng, pose, dims, res, 4000))
    single = vdev.DeviceSignedDistanceField(
        torch.from_numpy(field.astype(np.float32)).to("cuda:0"), res, pose)
    double = _device_field(field, res, pose)
    calls = [("EstimateLocationDistance", ()), ("GetLocationCoarseGradient", (False,)),
             ("GetLocationCoarseGradient", (True,)), ("GetLocationFineGradient", (0.03,)),
             ("GetLocationFineGradient", (0.6,)),
             ("ProjectLocationOutOfCollisionToMinimumDistance", (0.02, 0.25, 5000))]
    for name, arguments in calls:
        a_values, a_valid = getattr(single, name)(points, *arguments)
        b_values, b_valid = getattr(double, name)(points, *arguments)
        assert torch.equal(a_valid, b_valid), name
        np.testing.assert_array_equal(a_values.cpu().numpy(), b_values.cpu().numpy(), name)
    assert torch.equal(single.ComputeLocalExtremaMap(), double.ComputeLocalExtremaMap())


# ---- the Python interface

def test_python_argument_errors(shared_library):
    import torch
    from voxelized_geometry_tools_b200 import device as vdev
    from voxelized_geometry_tools_b200._capi import BackendUnavailable
    for dtype in (torch.float16, torch.int32, torch.bfloat16):
        with pytest.raises(ValueError):
            vdev.DeviceSignedDistanceField(torch.zeros((4, 4, 4), dtype=dtype, device="cuda:0"),
                                           0.1)
    with pytest.raises(ValueError):
        vdev.DeviceSignedDistanceField(torch.zeros((4, 16), dtype=torch.float64, device="cuda:0"),
                                       0.1)
    with pytest.raises(BackendUnavailable):
        vdev.DeviceSignedDistanceField(torch.zeros((4, 4, 4), dtype=torch.float64), 0.1)
    field = vdev.DeviceSignedDistanceField(
        torch.zeros((4, 4, 4), dtype=torch.float64, device="cuda:0"), 0.1)
    with pytest.raises(BackendUnavailable):           # points on the host
        field.EstimateLocationDistance(torch.zeros((3, 3), dtype=torch.float64))
    with pytest.raises(ValueError):
        field.EstimateLocationDistance(torch.zeros((3, 3), dtype=torch.float32, device="cuda:0"))
    with pytest.raises(ValueError):
        field.GetLocationCoarseGradient(torch.zeros((3, 2), dtype=torch.float64, device="cuda:0"))
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError):
            field.GetLocationFineGradient(
                torch.zeros((3, 3), dtype=torch.float64, device="cuda:1"), 0.1)


def test_empty_batch_launches_nothing(shared_library):
    import torch
    from voxelized_geometry_tools_b200 import _capi
    lib = _capi.library()
    field = _device_field(np.zeros((4, 5, 6)), 0.1, np.eye(4))
    points = torch.zeros((0, 3), dtype=torch.float64, device="cuda:0")
    before = lib.vgt_b200_kernel_launch_count()
    results = [field.EstimateLocationDistance(points),
               field.GetLocationCoarseGradient(points, True),
               field.GetLocationFineGradient(points, 0.1),
               field.ProjectLocationOutOfCollision(points)]
    assert lib.vgt_b200_kernel_launch_count() == before
    assert [tuple(v.shape) for v, _ in results] == [(0,), (0, 3), (0, 3), (0, 3)]
    assert all(tuple(valid.shape) == (0,) for _, valid in results)
