"""GPU: the per-slab connected-component phases (vgt_b200_components_*) and the torch.distributed
driver (ShardedConnectedComponents) against the one-device entry, byte for byte: the component
words and every word left untouched (occupancy, object id, spatial segment)."""
import os
import socket
import sys
from pathlib import Path

import numpy as np
import pytest

REPO = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(REPO))

pytestmark = pytest.mark.gpu


def label_emulating_ranks(cells, world):
    """Labels a copy of `cells` (CUDA int32 [nx, ny, nz, words]) as `world` ranks on one GPU
    would, moving what the collectives move by hand. Returns (labelled cells, count)."""
    import torch
    from voxelized_geometry_tools_b200 import device as vdev
    from voxelized_geometry_tools_b200.sharded import split_range
    nx, ny, nz, _ = cells.shape
    plane = ny * nz
    ranges = [split_range(nx, world, r) for r in range(world)]
    slabs = [cells[x0:x1].clone() for x0, x1 in ranges]
    states = [vdev.ComponentSlab(slab, x0 * plane) for slab, (x0, _) in zip(slabs, ranges)]
    roots = [state.local(r + 1 < world) for r, state in enumerate(states)]
    edges = [states[r].face_edges(slabs[r - 1][-1].clone(), roots[r - 1].clone(),
                                  ranges[r - 1][0] * plane) for r in range(1, world)]
    # every rank resolves the gathered edges; the ranks' lists in rank order, as all_gather has it
    gathered = torch.cat(edges) if edges else torch.zeros((0, 2), dtype=torch.int64,
                                                          device=cells.device)
    num_nodes = {state.resolve(gathered.clone(), nx * plane) for state in states}
    assert len(num_nodes) == 1
    counts = [state.count() for state in states]
    published = [state.publish(sum(counts[:r])) for r, state in enumerate(states)]
    summed = torch.stack(published).sum(dim=0).to(torch.int32)   # the all_reduce SUM
    for state in states:
        state.write(summed.clone())
    return torch.cat(slabs), sum(counts)


def reference(cells):
    from voxelized_geometry_tools_b200 import device as vdev
    want = cells.clone()
    count = vdev.connected_components(want)
    return want, int(count.item())


def spheres_on_device(shape, seed, device, count=60):
    """8-byte cells of a map of filled balls, built on the device; component words all ones."""
    import torch
    rng = np.random.default_rng(seed)
    nx, ny, nz = shape
    x = torch.arange(nx, device=device, dtype=torch.float32).view(-1, 1, 1)
    y = torch.arange(ny, device=device, dtype=torch.float32).view(1, -1, 1)
    z = torch.arange(nz, device=device, dtype=torch.float32).view(1, 1, -1)
    occupancy = torch.zeros(shape, dtype=torch.float32, device=device)
    for _ in range(count):
        cx, cy, cz = rng.uniform(0, shape)
        radius = rng.uniform(4, min(shape) / 8)
        inside = (x - cx) ** 2 + (y - cy) ** 2 + (z - cz) ** 2 <= radius ** 2
        occupancy[inside] = 1.0
    cells = torch.full(shape + (2,), -1, dtype=torch.int32, device=device)
    cells[..., 0] = occupancy.view(torch.int32)
    return cells


@pytest.mark.parametrize("world", range(1, 9))
def test_phases_emulating_ranks_on_one_gpu(shared_library, world):
    import torch
    from tests.test_components_sharded_gloo import scenes, words_of
    dev = torch.device("cuda", 0)
    for name, cells in scenes(world):
        full = torch.from_numpy(words_of(cells)).to(dev)
        want, want_count = reference(full)
        got, count = label_emulating_ranks(full, world)
        assert count == want_count, name
        assert torch.equal(got, want), name


def test_phases_on_a_512_cubed_spheres_map(shared_library):
    import torch
    dev = torch.device("cuda", 0)
    cells = spheres_on_device((512, 512, 512), 512, dev)
    want, want_count = reference(cells)
    assert want_count > 2
    for world in range(1, 9):
        got, count = label_emulating_ranks(cells, world)
        assert count == want_count, world
        assert torch.equal(got, want), world
        del got
    torch.cuda.synchronize()


# ---- across processes (NCCL) -------------------------------------------------------------------
def _nccl_worker(rank, world, port, result_dir):
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world,
                            device_id=torch.device("cuda", rank))
    try:
        from tests.test_components_sharded_gloo import scenes, words_of
        from voxelized_geometry_tools_b200.sharded import ShardedConnectedComponents
        dev = torch.device("cuda", rank)
        failures, counts = [], []
        named = list(scenes(world)) + [("spheres", None)]
        for name, cells in named:
            if cells is None:
                full = spheres_on_device((96, 80, 72), 5, dev, count=12)
            else:
                full = torch.from_numpy(words_of(cells)).to(dev)
            plan = ShardedConnectedComponents(tuple(full.shape[:3]))
            x0, x1 = plan.x_range
            slab = full[x0:x1].clone()
            count = plan.label(slab)
            counts.append(count)
            slabs = [None] * world
            dist.all_gather_object(slabs, slab.cpu().numpy())
            if rank == 0:
                got = np.concatenate(slabs)
                want, want_count = reference(full)
                if count != want_count or not np.array_equal(got, want.cpu().numpy()):
                    failures.append(f"{name}: differs from the one-device entry")
                multi = full.cpu().numpy().copy()
                _run_multi_entry(multi, world)
                if not np.array_equal(got, multi):
                    failures.append(f"{name}: differs from the host multi entry")
        Path(result_dir, f"rank{rank}.txt").write_text(
            "\n".join(failures) + f"\ncounts {counts}")
    finally:
        dist.destroy_process_group()


def _run_multi_entry(cells, world):
    import ctypes
    from voxelized_geometry_tools_b200 import _capi
    count = ctypes.c_uint32()
    devices = (ctypes.c_int * world)(*range(world))
    nx, ny, nz, words = cells.shape
    _capi.check(_capi.library().vgt_b200_connected_components_multi(
        cells.ctypes.data, 4 * words, nx, ny, nz, devices, world, ctypes.byref(count)))
    return count.value


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _visible_gpus():
    import torch
    return torch.cuda.device_count()


@pytest.mark.parametrize("world", ["2", "all"])
def test_nccl_ranks_match_the_one_device_entry(shared_library, tmp_path, world):
    import torch.multiprocessing as mp
    gpus = _visible_gpus()
    if gpus < 2:
        pytest.skip("needs 2 GPUs or more")
    if world == "all" and gpus == 2:
        pytest.skip("all visible GPUs are two: the world-2 case")
    world = 2 if world == "2" else gpus
    mp.spawn(_nccl_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    reports = [(tmp_path / f"rank{r}.txt").read_text() for r in range(world)]
    failures = reports[0].rsplit("\ncounts", 1)[0].strip()
    assert failures == "", failures
    # the same counts on every rank
    assert len({report.rsplit("counts", 1)[1] for report in reports}) == 1, reports
