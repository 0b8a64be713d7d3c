"""Times the cell-map SDF host entries and vgt_b200_sdf_f64_multi on one device against their
multi-device entries (the map cut into one x-slab per device):

* ``from_cells``: vgt_b200_sdf_from_cells_f32[_multi], objects_to_use = [2, 5];
* ``free_and_named``: vgt_b200_sdf_free_and_named_f32[_multi];
* ``per_object``: vgt_b200_sdf_per_object_f32[_multi], ids [2, 5];
* ``occupancy_f64``: vgt_b200_sdf_f64[_multi] on the float occupancy of the same scene.

    python profiles/time_cell_maps_multi.py [--out cell_maps_multi_b200.json] [--warmup 3]
                                            [--runs 10] [--sizes 512,1024] [--big 2048]

Sizes 512^3 and 1024^3 with 8- and 16-byte cells run on 1, 2, 4 and 8 devices (those that exist);
--big runs a 16-byte-cell map of that size on 8 devices only (at 2048^3 the one-device entries
need more memory than a B200 has). The scene: clustered spheres, object ids 0..6 in blocks of
256^3 voxels. Every call takes host buffers in and out and synchronises before it returns, so it
is timed with the host clock: median / min / max over --runs calls after --warmup untimed ones.
The host entries are bound by the bus: at sizes one device can hold, several devices may be
slower than one; what they add is the maps one device cannot hold.

Before it prints a case, the run checks that every device count gives the bytes of the first.
Prints one JSON line per case and writes the document, with the card's name and power limit read
in the same run, to --out when given.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import sys
import time
from pathlib import Path

import numpy as np
import torch

REPO = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(REPO))

from time_connected_components import card  # noqa: E402  (this script's directory)
from voxelized_geometry_tools_b200 import _capi, synthetic  # noqa: E402

RESOLUTION = 0.01
OBJECTS = [2, 5]
STEP = 256


def scene(n, cell_bytes):
    """(occupancy float[n,n,n], cells uint32[n,n,n,words]) built slab by slab on cuda:0."""
    words = cell_bytes // 4
    occupancy = np.empty((n, n, n), dtype=np.float32)
    cells = np.zeros((n, n, n, words), dtype=np.uint32)
    y = np.arange(n, dtype=np.uint32)[:, None] // 256
    z = np.arange(n, dtype=np.uint32)[None, :] // 256
    for x0 in range(0, n, STEP):
        x1 = min(n, x0 + STEP)
        slab = synthetic.clustered_spheres_occupancy_torch((n, n, n), "cuda:0", x_range=(x0, x1))
        occupancy[x0:x1] = slab.cpu().numpy()
        cells[x0:x1, :, :, 0] = occupancy[x0:x1].view(np.uint32)
        for x in range(x0, x1):
            cells[x, :, :, 1] = (x // 256 * 3 + y * 5 + z) % 7
    return occupancy, cells


def call(entry, occupancy, cells, devices, out, lows, highs):
    lib = _capi.library()
    n = occupancy.shape[0]
    ids = np.array(OBJECTS, dtype=np.uint32)
    cell_bytes = cells.shape[-1] * 4
    common = [cells.ctypes.data, cell_bytes, n, n, n, RESOLUTION, 1, 0]
    if len(devices) == 1:
        device_arguments, suffix = [devices[0]], ""
    else:
        device_arguments = [(ctypes.c_int * len(devices))(*devices), len(devices)]
        suffix = "_multi"
    if entry == "from_cells":
        code = getattr(lib, "vgt_b200_sdf_from_cells_f32" + suffix)(
            *common, ids.ctypes.data, ids.size, *device_arguments, out.ctypes.data,
            ctypes.byref(lows), ctypes.byref(highs))
    elif entry == "free_and_named":
        code = getattr(lib, "vgt_b200_sdf_free_and_named_f32" + suffix)(
            *common, *device_arguments, out.ctypes.data, ctypes.byref(lows), ctypes.byref(highs))
    elif entry == "per_object":
        extrema = np.empty((2, ids.size), dtype=np.float32)
        code = getattr(lib, "vgt_b200_sdf_per_object_f32" + suffix)(
            *common, ids.ctypes.data, ids.size, *device_arguments, out.ctypes.data,
            extrema[0].ctypes.data, extrema[1].ctypes.data)
    else:
        code = getattr(lib, "vgt_b200_sdf_f64" + suffix)(
            occupancy.ctypes.data, n, n, n, RESOLUTION, 1, 0, *device_arguments, out.ctypes.data,
            ctypes.byref(lows), ctypes.byref(highs))
    _capi.check(code)


def timed(function, warmup, runs):
    for _ in range(warmup):
        function()
    times = []
    for _ in range(runs):
        start = time.perf_counter()
        function()
        times.append((time.perf_counter() - start) * 1e3)
    return {"median_ms": statistics.median(times), "min_ms": min(times), "max_ms": max(times)}


def measure(n, cell_bytes, device_counts, entries, args):
    occupancy, cells = scene(n, cell_bytes)
    for entry in entries:
        results = 2 if entry == "per_object" else 1
        dtype = np.float64 if entry == "occupancy_f64" else np.float32
        scalar = ctypes.c_double if entry == "occupancy_f64" else ctypes.c_float
        out = np.empty((results, n, n, n), dtype=dtype)
        first = None
        case = {"n": n, "cell_bytes": cell_bytes, "entry": entry, "by_devices": {}}
        for count in device_counts:
            devices = list(range(count))
            lows, highs = scalar(), scalar()
            case["by_devices"][count] = timed(
                lambda: call(entry, occupancy, cells, devices, out, lows, highs), args.warmup,
                args.runs)
            if len(device_counts) > 1:
                digest = (hash(out.tobytes()), lows.value, highs.value)
                if first is None:
                    first = digest
                elif digest != first:
                    raise SystemExit(f"{entry} at {n}^3 differs on {count} devices")
        case["same_bytes_on_every_device_count"] = len(device_counts) > 1
        print(json.dumps(case), flush=True)
        yield case


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument("--out", default=None, help="file for the JSON document")
    parser.add_argument("--warmup", type=int, default=3)
    parser.add_argument("--runs", type=int, default=10)
    parser.add_argument("--sizes", default="512,1024")
    parser.add_argument("--big", type=int, default=2048, help="0 to skip")
    args = parser.parse_args()
    visible = torch.cuda.device_count()
    if visible < 2:
        raise SystemExit("needs at least 2 devices")
    counts = [c for c in (1, 2, 4, 8) if c <= visible]
    entries = ("from_cells", "free_and_named", "per_object", "occupancy_f64")
    result = {"card": card(), "devices_visible": visible, "warmup": args.warmup,
              "runs": args.runs, "objects": OBJECTS,
              "timing": "host clock around one synchronising call (host buffers in and out)",
              "cases": []}
    for n in (int(s) for s in args.sizes.split(",") if s):
        for cell_bytes in (8, 16):
            result["cases"] += list(measure(n, cell_bytes, counts, entries, args))
    if args.big:
        host = os.sysconf("SC_PAGE_SIZE") * os.sysconf("SC_PHYS_PAGES")
        # occupancy (4 B), cells (16 B), one field of 2 SDFs (8 B) per voxel
        needed = args.big ** 3 * (4 + 16 + 8)
        if visible < 8 or host < needed * 1.1:
            result["big"] = {"n": args.big, "skipped": f"{visible} devices, "
                                                       f"{host / 1e9:.0f} GB host memory; needs "
                                                       f"8 and {needed * 1.1 / 1e9:.0f} GB"}
            print(json.dumps(result["big"]), flush=True)
        else:
            result["cases"] += list(measure(args.big, 16, [8], entries[:3], args))
    if args.out:
        Path(args.out).write_text(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
