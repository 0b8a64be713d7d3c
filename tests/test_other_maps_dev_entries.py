"""CPU: the device cell entries (vgt_b200_sdf_from_cells_*_dev, vgt_b200_sdf_per_object_*_dev,
vgt_b200_sdf_free_and_named_*_dev) refuse bad arguments before they touch a device, and with
good arguments and no device they fail instead of computing anything on the CPU. The device
pointers here are never dereferenced."""
import numpy as np
import pytest

from voxelized_geometry_tools_b200 import _capi

CELLS = 0x10000   # aligned stand-ins for device pointers
OUT = 0x20000
MIN_MAX = 0x30000
IDS = np.array([3, 1, 3], dtype=np.uint32)


def entries(suffix):
    lib = _capi.library()

    def from_cells(cells, cell_bytes, dims, resolution, ids, num_ids, out, min_max):
        return getattr(lib, f"vgt_b200_sdf_from_cells_{suffix}_dev")(
            cells, cell_bytes, *dims, resolution, 1, 0, ids, num_ids, 0, out, min_max, None)

    def per_object(cells, cell_bytes, dims, resolution, ids, num_ids, out, min_max):
        return getattr(lib, f"vgt_b200_sdf_per_object_{suffix}_dev")(
            cells, cell_bytes, *dims, resolution, 1, 0, ids, num_ids, 0, out, min_max, None)

    def free_and_named(cells, cell_bytes, dims, resolution, ids, num_ids, out, min_max):
        return getattr(lib, f"vgt_b200_sdf_free_and_named_{suffix}_dev")(
            cells, cell_bytes, *dims, resolution, 1, 0, 0, out, min_max, None)

    return {"from_cells": from_cells, "per_object": per_object, "free_and_named": free_and_named}


GOOD = dict(cells=CELLS, cell_bytes=8, dims=(4, 5, 6), resolution=0.1, ids=IDS.ctypes.data,
            num_ids=IDS.size, out=OUT, min_max=MIN_MAX)

# (what, changed arguments, message fragment, whether free_and_named takes the argument)
REFUSALS = [
    ("null cells", dict(cells=None), "null", True),
    ("null output", dict(out=None), "null", True),
    ("cell size", dict(cell_bytes=12), "cell size", True),
    ("empty axis", dict(dims=(4, 0, 6)), "out of range", True),
    ("long axis", dict(dims=(4, 5, 8193)), "out of range", True),
    ("zero resolution", dict(resolution=0.0), "resolution", True),
    ("nan resolution", dict(resolution=float("nan")), "resolution", True),
    ("negative id count", dict(num_ids=-1), "object id list", False),
    ("ids missing", dict(ids=None), "object id list", False),
    ("too many ids", dict(num_ids=2 ** 31), "object id list", False),
    ("unaligned cells", dict(cells=CELLS + 2), "4-byte aligned", True),
    ("unaligned output", dict(out=OUT + 2), "aligned to their scalar", True),
    ("unaligned min/max", dict(min_max=MIN_MAX + 2), "aligned to their scalar", True),
]


@pytest.mark.parametrize("suffix", ["f32", "f64"])
@pytest.mark.parametrize("what,changed,fragment,free_and_named", REFUSALS,
                         ids=[r[0] for r in REFUSALS])
def test_bad_arguments_are_refused_without_a_device(shared_library, suffix, what, changed,
                                                    fragment, free_and_named):
    arguments = dict(GOOD, **changed)
    for name, entry in entries(suffix).items():
        if name == "free_and_named" and not free_and_named:
            continue
        assert entry(**arguments) == _capi.ERR_INVALID_ARGUMENT, (name, _capi.last_error())
        assert fragment in _capi.last_error(), (name, _capi.last_error())


@pytest.mark.parametrize("suffix,scalar_bytes", [("f32", 4), ("f64", 8)])
def test_batch_refuses_a_byte_count_beyond_int64(shared_library, suffix, scalar_bytes):
    # 8192^3 voxels: the largest batch whose bytes fit int64 has (2^63 - 1) // (2^39 * T) SDFs
    per_object = entries(suffix)["per_object"]
    largest = (2 ** 63 - 1) // (2 ** 39 * scalar_bytes)
    arguments = dict(GOOD, dims=(8192, 8192, 8192))
    assert per_object(**dict(arguments, num_ids=largest + 1)) == _capi.ERR_INVALID_ARGUMENT
    assert "overflow" in _capi.last_error()
    if _capi.device_count() > 0:
        pytest.skip("a GPU is present: the batch that fits would run")
    # one SDF fewer passes every check and stops at the missing device
    assert per_object(**dict(arguments, num_ids=largest)) == _capi.ERR_DEVICE


@pytest.mark.parametrize("suffix", ["f32", "f64"])
def test_no_cpu_fallback_without_device(shared_library, suffix):
    if _capi.device_count() > 0:
        pytest.skip("a GPU is present")
    for name, entry in entries(suffix).items():
        assert entry(**GOOD) == _capi.ERR_DEVICE, name
        assert "Cuda error" in _capi.last_error(), name
    # an empty batch launches nothing, but it still needs the device it was asked to use
    assert entries(suffix)["per_object"](**dict(GOOD, ids=None, num_ids=0)) == _capi.ERR_DEVICE


def test_python_functions_refuse_cpu_tensors():
    import torch
    from voxelized_geometry_tools_b200 import device as vdev
    cells = torch.zeros((4, 5, 6, 2), dtype=torch.int32)
    for call in (lambda: vdev.signed_distance_field_from_cells(cells, 0.1, [1]),
                 lambda: vdev.separate_object_sdfs(cells, 0.1, [1, 2]),
                 lambda: vdev.free_and_named_objects_sdf(cells, 0.1, dtype=torch.float64)):
        with pytest.raises(_capi.BackendUnavailable):
            call()
