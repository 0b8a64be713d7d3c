"""CPU: the per-slab connected-component entries (vgt_b200_components_*) refuse bad arguments
with the right code before any device call, and without a device a call with good arguments
fails: nothing runs on the CPU. The pointers below are never dereferenced on the host; the calls
with good arguments are made only where no GPU is present."""
import ctypes

import pytest

FAKE = 0x1000  # a non-null device pointer the checks accept (never used: no device here)


def entries():
    """name -> (arguments that pass every check, {argument index: what it is})."""
    size = ctypes.c_size_t()
    dims = (4, 3, 5)
    local = (FAKE, 8, *dims, 0, FAKE, FAKE, FAKE, FAKE, 64, FAKE, None)
    face_edges = (FAKE, FAKE, 0, FAKE, 16, *dims, 60, 0, FAKE, FAKE, FAKE, None)
    resolve = (FAKE, 10, 120, 60, 120, 0, FAKE, FAKE, FAKE, None)
    count = (*dims, 60, 7, 0, FAKE, FAKE, FAKE, FAKE, 9, 2, 3, FAKE, FAKE, FAKE, 64, None)
    publish = (*dims, 60, 7, 11, 0, FAKE, FAKE, FAKE, 9, 2, 3, FAKE, FAKE, FAKE, FAKE, None)
    write = (FAKE, 8, *dims, 60, 7, 0, FAKE, FAKE, FAKE, FAKE, FAKE, 9, 2, 3, FAKE, FAKE, None)
    return {
        "vgt_b200_components_slab_scan_bytes": ((*dims, 0, ctypes.byref(size)), {4: "scan size"}),
        "vgt_b200_components_slab_local": (local, {0: "cell array", 6: "parent array",
                                                   7: "root mask", 8: "word prefix",
                                                   9: "scan storage"}),
        "vgt_b200_components_slab_face_edges": (face_edges, {0: "face cell array",
                                                             1: "face roots", 3: "cell array",
                                                             10: "parent array",
                                                             11: "edge array",
                                                             12: "edge count"}),
        "vgt_b200_components_resolve": (resolve, {6: "node array", 7: "node roots",
                                                  8: "node range"}),
        "vgt_b200_components_slab_count": (count, {6: "root mask", 7: "word prefix",
                                                   8: "node array", 9: "node roots",
                                                   13: "root bits", 14: "root bit prefix",
                                                   15: "scan storage"}),
        "vgt_b200_components_slab_publish": (publish, {7: "root mask", 8: "word prefix",
                                                       9: "node array", 13: "root bits",
                                                       14: "root bit prefix",
                                                       15: "final id array",
                                                       16: "node id array"}),
        "vgt_b200_components_slab_write": (write, {0: "cell array", 8: "parent array",
                                                   9: "root mask", 10: "word prefix",
                                                   11: "node array", 12: "node roots",
                                                   16: "node id array", 17: "final id array"}),
    }


# where each entry takes (cell_bytes or None, nx, ny, nz)
SLAB_ARGUMENTS = {
    "vgt_b200_components_slab_scan_bytes": (None, 0),
    "vgt_b200_components_slab_local": (1, 2),
    "vgt_b200_components_slab_face_edges": (4, 5),
    "vgt_b200_components_slab_count": (None, 0),
    "vgt_b200_components_slab_publish": (None, 0),
    "vgt_b200_components_slab_write": (1, 2),
}


def call(name, arguments):
    from voxelized_geometry_tools_b200 import _capi
    return getattr(_capi.library(), name)(*arguments)


@pytest.mark.parametrize("name", sorted(entries()))
def test_entry_refuses_bad_arguments(shared_library, name):
    from voxelized_geometry_tools_b200 import _capi
    good, pointers = entries()[name]

    def refused(code, text, **changes):
        arguments = list(good)
        for index, value in changes.items():
            arguments[int(index[1:])] = value
        assert call(name, arguments) == code, (name, changes)
        assert text in _capi.last_error(), (name, changes, _capi.last_error())

    invalid = _capi.ERR_INVALID_ARGUMENT
    for index, what in pointers.items():
        refused(invalid, f"null {what}", **{f"a{index}": None})
    if name in SLAB_ARGUMENTS:
        cell_bytes_at, nx_at = SLAB_ARGUMENTS[name]
        if cell_bytes_at is not None:
            for cell_bytes in (0, 4, 12, 32):
                refused(invalid, "cell size", **{f"a{cell_bytes_at}": cell_bytes})
        for bad in ((0, 3, 5), (4, 0, 5), (4, 3, -1), (8193, 3, 5)):
            refused(invalid, "out of range", **{f"a{nx_at + k}": v for k, v in enumerate(bad)})
        # slabs of 2^32 cells or more
        refused(_capi.ERR_UNSUPPORTED, "2^32",
                **{f"a{nx_at + k}": v for k, v in enumerate((4096, 1024, 1024))})
    if name == "vgt_b200_components_resolve":
        refused(invalid, "edges", a1=-1)
        refused(invalid, "edges", a0=None)            # edges promised, none given
        refused(invalid, "outside", a4=121)           # slab end past the map
        refused(invalid, "outside", a3=120)           # empty slab
    if name == "vgt_b200_components_slab_face_edges":
        refused(invalid, "out of order", a8=10)       # the slab below ends past this base
    if name in ("vgt_b200_components_slab_count", "vgt_b200_components_slab_publish",
                "vgt_b200_components_slab_write"):
        components_at = good.index(7)
        refused(invalid, "local components", **{f"a{components_at}": 0})
        refused(invalid, "local components", **{f"a{components_at}": 61})
        nodes_at = good.index(9)
        refused(invalid, "node range", **{f"a{nodes_at}": 4})          # first + own > nodes
        refused(invalid, "node range", **{f"a{nodes_at + 2}": -1})
    if name == "vgt_b200_components_slab_publish":
        refused(invalid, "offset", a5=-1)
        refused(invalid, "offset", a5=1 << 32)


@pytest.mark.parametrize("name", sorted(entries()))
def test_no_cpu_fallback_without_device(shared_library, name):
    from voxelized_geometry_tools_b200 import _capi
    if _capi.device_count() > 0:
        pytest.skip("a GPU is present")
    good, _ = entries()[name]
    assert call(name, good) == _capi.ERR_DEVICE
    assert "Cuda error" in _capi.last_error()


def test_no_cpu_fallback_in_the_python_driver(shared_library):
    import torch
    import voxelized_geometry_tools_b200 as vgt
    from voxelized_geometry_tools_b200 import device
    from voxelized_geometry_tools_b200.sharded import ShardedConnectedComponents
    cells = torch.zeros((4, 3, 5, 2), dtype=torch.int32)
    with pytest.raises(vgt.BackendUnavailable):
        device.ComponentSlab(cells, 0)
    plan = ShardedConnectedComponents((4, 3, 5), rank=0, world_size=1)
    with pytest.raises(vgt.BackendUnavailable):
        plan.label(cells)
    assert not cells.any()
