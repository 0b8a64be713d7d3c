"""CPU: host-side mirror of the reference interface (no GPU needed)."""
import numpy as np
import pytest

import voxelized_geometry_tools_b200 as vgt
from voxelized_geometry_tools_b200 import synthetic
from voxelized_geometry_tools_b200.sharded import split_range


def test_grid_sizes_follow_the_reference_fixture():
    # test/sdf_generation_test.cpp:267-272: (1.0, 2.0, 3.0) @ 0.25 -> 4 x 8 x 12
    sizes = vgt.VoxelGridSizes.FromGridSizes(0.25, (1.0, 2.0, 3.0))
    assert sizes.shape == (4, 8, 12)
    assert vgt.VoxelGridSizes.FromVoxelCounts(0.125, (40, 40, 40)).sizes() == (5.0, 5.0, 5.0)
    with pytest.raises(ValueError):
        vgt.VoxelGridSizes.FromGridSizes(0.0, (1, 1, 1))


def test_filter_options_validation_and_rule(oracle):
    # pointcloud_voxelization_interface.hpp:30-41 and :55-86
    for bad in ((0.0, 1, 1), (1.01, 1, 1), (0.5, 0, 1), (0.5, 1, 0)):
        with pytest.raises(ValueError):
            vgt.PointCloudVoxelizationFilterOptions(*bad)
    options = vgt.PointCloudVoxelizationFilterOptions(0.9, 2, 1)
    assert options.CountsSeenAs(3, 0) == vgt.SeenAs.FREE
    assert options.CountsSeenAs(0, 1) == vgt.SeenAs.UNKNOWN      # below the outlier threshold
    assert options.CountsSeenAs(0, 2) == vgt.SeenAs.FILLED
    assert options.CountsSeenAs(18, 2) == vgt.SeenAs.FREE        # 0.9 >= 0.9
    assert options.CountsSeenAs(17, 2) == vgt.SeenAs.FILLED
    assert options.CountsSeenAs(0, 0) == vgt.SeenAs.UNKNOWN
    # the host rule agrees with the oracle's filter on every small count pair
    for free in range(0, 6):
        for filled in range(0, 6):
            counts = np.array([[[[[free, filled]]]]], dtype=np.int32)
            got = oracle.filter_grids(counts, np.zeros((1, 1, 1), np.float32), 0.9, 2, 1)[0, 0, 0]
            want = {vgt.SeenAs.FREE: 0.0, vgt.SeenAs.FILLED: 1.0,
                    vgt.SeenAs.UNKNOWN: 0.5}[options.CountsSeenAs(free, filled)]
            assert got == want


def test_voxelizer_runtime_and_argument_checks():
    with pytest.raises(ValueError):
        vgt.VoxelizerRuntime(-1.0, 0.0)
    runtime = vgt.VoxelizerRuntime(0.25, 0.5)
    assert (runtime.RaycastingTime(), runtime.FilteringTime()) == (0.25, 0.5)

    class Recorder(vgt.PointCloudVoxelizationInterface):
        def DoVoxelizePointClouds(self, static, options, clouds, output):
            output.GetMutableRawData()[...] = 0.25
            return vgt.VoxelizerRuntime(0.0, 0.0)

    sizes = vgt.VoxelGridSizes.FromVoxelCounts(0.5, (2, 2, 2))
    static = vgt.OccupancyMap(np.eye(4), "world", sizes)
    out = Recorder().VoxelizePointClouds(static, vgt.PointCloudVoxelizationFilterOptions(), [])
    assert np.all(out.GetImmutableRawData() == 0.25) and np.all(static.GetImmutableRawData() == 0)
    with pytest.raises(ValueError):   # pcv_if.hpp:281-289
        Recorder().VoxelizePointClouds(static, vgt.PointCloudVoxelizationFilterOptions(), [None])
    other = vgt.OccupancyMap(np.eye(4), "world", vgt.VoxelGridSizes.FromVoxelCounts(0.5, (2, 2, 3)))
    with pytest.raises(ValueError):   # pcv_if.hpp:275-280
        Recorder().VoxelizePointClouds(static, vgt.PointCloudVoxelizationFilterOptions(), [],
                                       output_environment=other)


def test_point_cloud_wrapper():
    cloud = vgt.VectorPointCloudWrapper()
    cloud.PushBack((1.0, 2.0, 3.0))
    cloud.PushBack((4.0, 5.0, 6.0))
    assert cloud.Size() == 2 and cloud.MaxRange() == float("inf")
    np.testing.assert_array_equal(cloud.GetPointLocationVector4d(1), [4.0, 5.0, 6.0, 1.0])
    with pytest.raises(IndexError):
        cloud.GetPointLocationVector4d(2)
    generic = vgt.PointCloudWrapper.PointsAsDoubleArray(cloud)   # per-point path
    np.testing.assert_array_equal(generic, cloud.PointsAsDoubleArray())


def test_inverse_origin_transform():
    transform = synthetic.look_at_pose((1.0, -2.0, 0.5))
    sizes = vgt.VoxelGridSizes.FromVoxelCounts(0.5, (2, 2, 2))
    occupancy_map = vgt.OccupancyMap(transform, "world", sizes)
    np.testing.assert_allclose(occupancy_map.InverseOriginTransform() @ transform, np.eye(4),
                               atol=1e-12)


def test_sdf_container_lock_semantics():
    sizes = vgt.VoxelGridSizes.FromVoxelCounts(1.0, (1, 1, 3))
    sdf = vgt.SignedDistanceField(np.eye(4), "f", sizes,
                                  np.array([[[-1.0, 1.0, 2.0]]], dtype=np.float32), float("inf"))
    with pytest.raises(RuntimeError):
        sdf.GetMinimumMaximum()
    sdf.Lock()
    assert sdf.GetMinimumMaximum() == (-1.0, 2.0)
    assert sdf.GetIndexImmutable(0, 0, 5) == np.float32(np.inf)   # OOB value


def test_split_range_covers_everything():
    for total in (1, 7, 8, 9, 513):
        for parts in (1, 2, 3, 8):
            if parts > total:
                continue
            edges = [split_range(total, parts, i) for i in range(parts)]
            assert edges[0][0] == 0 and edges[-1][1] == total
            assert all(a[1] == b[0] for a, b in zip(edges, edges[1:]))
            sizes = [e[1] - e[0] for e in edges]
            assert max(sizes) - min(sizes) <= 1


def test_synthetic_generators_are_deterministic_and_consistent():
    import torch
    a = synthetic.clustered_spheres_occupancy((48, 40, 56))
    b = synthetic.clustered_spheres_occupancy_torch((48, 40, 56), "cpu").numpy()
    np.testing.assert_array_equal(a, b)
    slab = synthetic.clustered_spheres_occupancy_torch((48, 40, 56), "cpu", x_range=(12, 30))
    np.testing.assert_array_equal(a[12:30], slab.numpy())
    assert 0.05 < (a == 1.0).mean() < 0.16 and 0.005 < (a == 0.5).mean() < 0.015
    rng = synthetic.Mt19937_64(5489)
    assert rng.next_u64() == 14514284786278117030     # the published first output of mt19937_64


def test_bench_finds_the_ncu_traffic_of_every_pass():
    # bench.py reports roofline.traffic from profiles/ncu_traffic.json; a renamed kernel label
    # would silently turn it into null
    import importlib.util
    from pathlib import Path
    repo = Path(__file__).resolve().parents[1]
    spec = importlib.util.spec_from_file_location("bench_module", repo / "bench.py")
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    dims = bench.workload_dims(1)
    for name in bench.PASS_NAMES:
        traffic = bench.ncu_dram_bytes_per_launch(dims, name, check_build=False)
        assert traffic is not None, name
        voxels = dims[0] * dims[1] * dims[2]
        # between the algorithmic 8 B/voxel (minus what L2 keeps) and twice that
        assert 0.9 * bench.PASS_BYTES_PER_VOXEL * voxels < traffic < 2 * bench.PASS_BYTES_PER_VOXEL * voxels
        # the numbers belong to ONE build of the kernels: with the build check on they are
        # attached iff the table's source hash is the current one
        import json
        from voxelized_geometry_tools_b200 import build as cuda_build
        entry = json.loads(bench.NCU_TRAFFIC_FILE.read_text())["x".join(map(str, dims))][name]
        checked = bench.ncu_dram_bytes_per_launch(dims, name)
        assert (checked is not None) == (entry.get("sources_sha1") == cuda_build._sources_signature())


def test_bench_dumps_a_fixed_sample_of_the_sdf(tmp_path):
    # bench.py --dump-outputs: the same output gives the same files, so two builds compare
    # value for value; every file is float32 or float64
    import importlib.util
    from pathlib import Path

    import torch
    repo = Path(__file__).resolve().parents[1]
    spec = importlib.util.spec_from_file_location("bench_module", repo / "bench.py")
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    sdf = torch.from_numpy(np.random.default_rng(3).standard_normal((40, 48, 56), np.float32))
    min_max = torch.tensor([sdf.min(), sdf.max()])
    for name in ("a", "b"):
        bench.dump_outputs(tmp_path / name, sdf, min_max)
    for name in ("sdf_min_max.npy", "sdf_sample.npy", "sdf_sample_index.npy"):
        first, second = np.load(tmp_path / "a" / name), np.load(tmp_path / "b" / name)
        assert first.dtype in (np.float32, np.float64)
        np.testing.assert_array_equal(first, second)
    index = np.load(tmp_path / "a" / "sdf_sample_index.npy").astype(np.int64)
    assert len(index) > sdf.numel() // 2 and np.all(np.diff(index) > 0)
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "sdf_sample.npy"),
                                  sdf.numpy().reshape(-1)[index])
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "sdf_min_max.npy"), min_max.numpy())
    # sharded: every rank samples its own slab, rank 0 adds the global min/max
    for rank in (0, 1):
        bench.dump_outputs(tmp_path / "sharded", sdf, min_max, rank=rank, world=2)
    assert sorted(path.name for path in (tmp_path / "sharded").iterdir()) == [
        "sdf_min_max.npy", "sdf_sample_index_rank0.npy", "sdf_sample_index_rank1.npy",
        "sdf_sample_rank0.npy", "sdf_sample_rank1.npy"]
    for rank in (0, 1):
        index = np.load(tmp_path / "sharded" / f"sdf_sample_index_rank{rank}.npy").astype(np.int64)
        assert 0 < len(index) <= sdf.numel()
        np.testing.assert_array_equal(np.load(tmp_path / "sharded" / f"sdf_sample_rank{rank}.npy"),
                                      sdf.numpy().reshape(-1)[index])
