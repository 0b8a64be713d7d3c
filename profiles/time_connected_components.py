"""Times the connected-component labelling (vgt_b200_connected_components_dev) on device-resident
cells with CUDA events, and the host entry once, against the compulsory traffic of the call: the
cells read once and written once, 2 x cell_bytes per voxel, at the data-sheet 7.7 TB/s.

    python profiles/time_connected_components.py [--out connected_components.json]
                                                 [--warmup 3] [--runs 10] [--quick]

Prints one JSON line per case and writes the whole document to --out when given: the card's name
and power limit, read in the same run, then per case the median / min / max milliseconds, the
floor and the component count.
"""
from __future__ import annotations

import argparse
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

REPO = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(REPO))

from voxelized_geometry_tools_b200 import _capi, synthetic  # noqa: E402
from voxelized_geometry_tools_b200.grids import (OccupancyComponentMap,  # noqa: E402
                                                 VoxelGridSizes)

DATASHEET_BYTES_PER_S = 7.7e12


def card():
    try:
        text = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit",
                               "--format=csv,noheader"], capture_output=True, text=True,
                              timeout=60).stdout.strip().splitlines()
        name, power = (part.strip() for part in text[0].split(","))
        return {"name": name, "power_limit": power}
    except Exception as error:  # recorded, not fatal
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"unknown ({error})"}


def serpentine(n, device):
    occupancy = torch.zeros((n, n, n), dtype=torch.float32, device=device)
    occupancy[0::2, 0::2, :] = 1.0
    for y in range(1, n - 1, 2):
        occupancy[0::2, y, n - 1 if (y // 2) % 2 == 0 else 0] = 1.0
    occupancy[1:n - 1:2, 0, 0] = 1.0
    return occupancy


def occupancy_for(scene, n, device):
    if scene == "spheres":
        return synthetic.clustered_spheres_occupancy_torch((n, n, n), device)
    if scene == "noise50":
        generator = torch.Generator(device=device).manual_seed(50)
        return (torch.rand((n, n, n), generator=generator, device=device) < 0.5).float()
    if scene == "serpentine":
        return serpentine(n, device)
    raise ValueError(scene)


def cells_for(scene, n, cell_bytes, device):
    occupancy = occupancy_for(scene, n, device)
    words = cell_bytes // 4
    cells = torch.zeros((n, n, n, words), dtype=torch.int32, device=device)
    cells[..., 0] = occupancy.view(torch.int32)
    if words == 4:
        # object ids: eight slabs along x, so the id rule splits components too
        x = torch.arange(n, device=device, dtype=torch.int32).view(n, 1, 1)
        cells[..., 1] = (x * 8 // n).expand(n, n, n)
    del occupancy
    return cells


def time_device(cells, warmup, runs):
    lib = _capi.library()
    device = cells.device
    n = cells.shape[0]
    count = torch.zeros(1, dtype=torch.uint32, device=device)
    stream = torch.cuda.current_stream(device)
    counts = []

    def call():
        _capi.check(lib.vgt_b200_connected_components_dev(
            cells.data_ptr(), 4 * cells.shape[3], n, n, n, device.index or 0, count.data_ptr(),
            int(stream.cuda_stream)))

    for _ in range(warmup):
        call()
    torch.cuda.synchronize()
    times = []
    for _ in range(runs):
        start = torch.cuda.Event(enable_timing=True)
        stop = torch.cuda.Event(enable_timing=True)
        start.record(stream)
        call()
        stop.record(stream)
        stop.synchronize()
        times.append(start.elapsed_time(stop))
        counts.append(int(count.item()))
    assert len(set(counts)) == 1, counts
    return times, counts[0]


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument("--out", default=None, help="file for the JSON document")
    parser.add_argument("--warmup", type=int, default=3)
    parser.add_argument("--runs", type=int, default=10)
    parser.add_argument("--quick", action="store_true", help="small sizes (a rehearsal)")
    args = parser.parse_args()
    if not torch.cuda.is_available() or _capi.device_count() == 0:
        raise SystemExit("no usable CUDA device: nothing to measure")
    device = torch.device("cuda", 0)
    big, mid, huge = (64, 32, 96) if args.quick else (512, 256, 1024)
    cases = [("spheres", big, 8), ("noise50", big, 8), ("serpentine", big, 8),
             ("spheres", mid, 16), ("spheres", big, 16), ("spheres", huge, 8)]
    result = {"card": card(), "warmup": args.warmup, "runs": args.runs,
              "floor_rule": "2 x cell_bytes per voxel at 7.7 TB/s (data sheet)", "cases": []}
    for scene, n, cell_bytes in cases:
        cells = cells_for(scene, n, cell_bytes, device)
        times, count = time_device(cells, args.warmup, args.runs)
        floor_ms = 2.0 * cell_bytes * n ** 3 / DATASHEET_BYTES_PER_S * 1e3
        median = statistics.median(times)
        result["cases"].append({
            "entry": "dev", "scene": scene, "n": n, "cell_bytes": cell_bytes,
            "median_ms": round(median, 4), "min_ms": round(min(times), 4),
            "max_ms": round(max(times), 4), "floor_ms": round(floor_ms, 4),
            "times_floor": round(median / floor_ms, 2),
            "gvoxels_per_s": round(n ** 3 / median / 1e6, 2), "components": count})
        print(json.dumps(result["cases"][-1]), flush=True)
        del cells
        torch.cuda.empty_cache()

    # the host entry once (pageable numpy cells in and out, staged copies included), after one
    # untimed call that creates the staging slots and loads the kernels
    n = big
    occupancy = synthetic.clustered_spheres_occupancy((n, n, n))
    grid = OccupancyComponentMap(np.eye(4), "world", VoxelGridSizes.FromVoxelCounts(0.01, (n,) * 3))
    grid.GetMutableRawData()["occupancy"] = occupancy
    grid.UpdateConnectedComponents()
    begin = time.perf_counter()
    count = grid.UpdateConnectedComponents()
    host_ms = (time.perf_counter() - begin) * 1e3
    result["cases"].append({"entry": "host", "scene": "spheres", "n": n, "cell_bytes": 8,
                            "ms": round(host_ms, 3), "components": count})
    print(json.dumps(result["cases"][-1]), flush=True)

    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(result, indent=1) + "\n")
    print(json.dumps({"card": result["card"]}))


if __name__ == "__main__":
    main()
