"""CPU: the x-slab connected-component driver (ShardedConnectedComponents) over gloo, world sizes
1 to 4. The device phases are replaced by numpy stand-ins built from the slab model of
tests/test_components_slabs_model.py, so this exercises the host-side logic of the per-rank path:
slab ranges, the face hand-over from rank r to rank r + 1, the gathered edges, the offsets and
the summed node ids. Every rank's slab must equal the whole-grid labelling (scipy, renumbered by
first occurrence), and every rank must return the same count."""
import os
import socket
import sys
import zlib
from pathlib import Path

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

REPO = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(REPO))


def words_of(cells):
    """Structured cells -> int32 words [nx, ny, nz, 2 | 4] (the layout the driver labels)."""
    words = len(cells.dtype.names)
    return np.ascontiguousarray(cells).view(np.int32).reshape(cells.shape + (words,))


def expected_words(cells):
    """The cells' words with the component word set to the whole-grid labelling, and the count."""
    from tests import components
    ids, count = components.scipy_components(cells)
    words = words_of(cells).copy()
    words[..., 1 if words.shape[3] == 2 else 2] = ids.view(np.int32)
    return words, count


def scenes(world):
    """(name, structured cells) of every scene, for a map cut into `world` slabs."""
    from tests import components, slab_scenes
    rng = np.random.default_rng(zlib.crc32(b"sharded components %d" % world))
    nx = 3 * world + 2
    result = [
        ("checkerboard", components.make_cells(components.checkerboard((nx, 5, 4)), rng=rng)),
        ("serpentine", components.make_cells(slab_scenes.x_serpentine((nx, 9, 3)), rng=rng)),
        ("ring", components.make_cells(slab_scenes.ring_closed_in_slab((nx, 6, 4), nx - 1),
                                       rng=rng)),
        ("last_slab", components.make_cells(
            slab_scenes.last_slab_components((nx, 7, 5), nx - 1), rng=rng)),
        ("special", components.make_cells(components.special_values(rng, (nx, 4, 6)), rng=rng)),
        ("tagged", components.make_cells(
            (rng.random((nx, 5, 6)) < 0.5).astype(np.float32),
            rng.integers(0, 3, (nx, 5, 6), dtype=np.uint32), rng)),
        ("one_plane", components.make_cells(components.special_values(rng, (world, 6, 5)),
                                            rng.integers(0, 2, (world, 6, 5), dtype=np.uint32),
                                            rng)),
        ("one_plane_8B", components.make_cells(components.checkerboard((world, 3, 7)), rng=rng)),
    ]
    return result


# ---- numpy stand-ins of the device phases ------------------------------------------------------
def _keys(words):
    """The connection key of cells given as int32 words [..., 2 | 4]."""
    occupancy = np.ascontiguousarray(words[..., 0]).view(np.float32)
    key = (occupancy > np.float32(0.5)).astype(np.int64)
    if words.shape[-1] == 4:
        key += 2 * np.ascontiguousarray(words[..., 1]).view(np.uint32).astype(np.int64)
    return key


def numpy_stages(seed, count_override=None):
    from tests.test_components_slabs_model import local_roots
    from voxelized_geometry_tools_b200.sharded import ComponentStages
    rng = np.random.default_rng(seed)

    def local(cells_slab, base, face_roots):
        words = cells_slab.view(torch.int32).numpy()
        key = _keys(words)
        roots = local_roots(key)
        plane = key.shape[1] * key.shape[2]
        state = dict(words=words, key=key, roots=roots, unique=np.unique(roots), base=base,
                     plane=plane, nz=key.shape[2])
        face = torch.from_numpy(roots[-plane:].astype(np.int32)) if face_roots else None
        return state, face

    def face_edges(state, below_cells, below_roots, below_base):
        plane = state["plane"]
        below_key = _keys(below_cells.numpy()).reshape(-1)
        above_key = state["key"][0].reshape(-1)
        z = np.arange(plane) % state["nz"]
        implied = np.zeros(plane, dtype=bool)
        implied[1:] = (z[1:] > 0) & (above_key[:-1] == above_key[1:]) \
            & (below_key[:-1] == above_key[1:])
        emit = np.flatnonzero((below_key == above_key) & ~implied)
        edges = np.stack([below_base + below_roots.numpy()[emit].astype(np.int64),
                          state["base"] + state["roots"][emit]], axis=1)
        return torch.from_numpy(edges[rng.permutation(len(edges))].reshape(-1, 2))

    def resolve(state, edges, num_cells):
        edges = edges.numpy()
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
        state["nodes"] = nodes
        state["node_roots"] = np.array([find(k) for k in range(nodes.size)], dtype=np.int64)
        first, last = np.searchsorted(nodes, [state["base"], state["base"] + state["roots"].size])
        state["first"], state["last"] = int(first), int(last)
        state["node_ranks"] = np.searchsorted(state["unique"], nodes[first:last] - state["base"])
        return nodes.size

    def count(state):
        bits = np.ones(state["unique"].size, dtype=bool)
        own = np.arange(state["first"], state["last"])
        bits[state["node_ranks"][state["node_roots"][own] != own]] = False
        state["bits"] = bits
        return int(bits.sum()) if count_override is None else count_override

    def publish(state, offset):
        final = np.zeros(state["bits"].size, dtype=np.int64)
        final[state["bits"]] = offset + 1 + np.arange(int(state["bits"].sum()))
        state["final"] = final
        node_ids = np.zeros(state["nodes"].size, dtype=np.uint32)
        node_ids[state["first"]:state["last"]] = final[state["node_ranks"]]
        return torch.from_numpy(node_ids.view(np.int32))

    def write(state, node_ids):
        ids = node_ids.numpy().view(np.uint32).astype(np.int64)
        own = np.arange(state["first"], state["last"])
        final = state["final"]
        final[state["node_ranks"]] = ids[state["node_roots"][own]]
        ranks = np.searchsorted(state["unique"], state["roots"])
        words = state["words"]
        component = final[ranks].astype(np.uint32).view(np.int32).reshape(words.shape[:3])
        words[..., 1 if words.shape[3] == 2 else 2] = component

    return ComponentStages(local, face_edges, resolve, count, publish, write)


# ---- the driver on each rank -------------------------------------------------------------------
def label_every_scene(rank, world, stage_seed):
    """Labels every scene; returns the failures (empty when every slab is right)."""
    from voxelized_geometry_tools_b200.sharded import ShardedConnectedComponents
    failures = []
    for name, cells in scenes(world):
        want, want_count = expected_words(cells)
        plan = ShardedConnectedComponents(cells.shape, rank=rank, world_size=world,
                                          stages=numpy_stages(stage_seed + rank))
        x0, x1 = plan.x_range
        slab = torch.from_numpy(words_of(cells)[x0:x1].copy())
        count = plan.label(slab)
        if count != want_count:
            failures.append(f"{name}: count {count} != {want_count}")
        if not np.array_equal(slab.numpy(), want[x0:x1]):
            failures.append(f"{name}: slab [{x0}, {x1}) differs")
    return failures


def _worker(rank, world, port, result_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from voxelized_geometry_tools_b200.sharded import ShardedConnectedComponents
        failures = label_every_scene(rank, world, stage_seed=7 * world)
        # counts that add up past the 32-bit component word: the same error on every rank, and no
        # cell written
        cells = scenes(world)[0][1]
        plan = ShardedConnectedComponents(cells.shape,
                                          stages=numpy_stages(rank, count_override=0x80000000))
        x0, x1 = plan.x_range
        before = words_of(cells)[x0:x1].copy()
        slab = torch.from_numpy(before.copy())
        try:
            plan.label(slab)
            failures.append("no error past 0xFFFFFFFF components")
        except NotImplementedError as error:
            message = str(error)
            if str(0x80000000 * world) not in message:
                failures.append(f"unexpected message {message}")
        if not np.array_equal(slab.numpy(), before):
            failures.append("cells written after the overflow")
        # every rank's counts and message are compared by the test
        Path(result_dir, f"rank{rank}.txt").write_text("\n".join(failures) or "ok")
    finally:
        dist.destroy_process_group()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.parametrize("world", [2, 3, 4])
def test_sharded_components_match_the_whole_grid(tmp_path, world):
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    for rank in range(world):
        assert (tmp_path / f"rank{rank}.txt").read_text() == "ok", rank


def test_world_size_one_needs_no_process_group():
    assert label_every_scene(0, 1, stage_seed=1) == []


def test_overflow_at_world_size_one_leaves_the_cells():
    from voxelized_geometry_tools_b200.sharded import ShardedConnectedComponents
    cells = scenes(1)[0][1]
    words = words_of(cells).copy()
    plan = ShardedConnectedComponents(cells.shape, rank=0, world_size=1,
                                      stages=numpy_stages(0, count_override=0x100000000))
    slab = torch.from_numpy(words.copy())
    with pytest.raises(NotImplementedError, match="4294967296 components"):
        plan.label(slab)
    assert np.array_equal(slab.numpy(), words)


def test_more_ranks_than_x_planes_are_refused():
    from voxelized_geometry_tools_b200.sharded import ShardedConnectedComponents
    with pytest.raises(ValueError, match="more ranks"):
        ShardedConnectedComponents((3, 4, 4), rank=0, world_size=4, stages=numpy_stages(0))
