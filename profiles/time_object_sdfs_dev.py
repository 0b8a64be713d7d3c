"""Times MakeSeparateObjectSDFs of a tagged map three ways, for 8 objects in 256^3 and 512^3 maps
with 8- and 16-byte cells:

* ``batch``: vgt_b200_sdf_per_object_f32_dev on device cells (one slot map for the 8 ids, then
  the three passes per object on "slot == key");
* ``single_calls``: 8 calls of vgt_b200_sdf_from_cells_f32_dev on the same device cells, one id
  each (each call classifies the cells into a mask again);
* ``host_entry``: vgt_b200_sdf_per_object_f32 on host cells (upload, the mask route per object,
  copy-out of every SDF to pageable host memory).

    python profiles/time_object_sdfs_dev.py [--out object_sdfs_dev.json] [--warmup 3] [--runs 10]
                                            [--quick]

The scene is bench.py's tagged map: clustered spheres, object ids in blocks of 64 x 128 x 128
voxels, ids 1..8. The device routes are timed with CUDA events around each call, the host entry
(which synchronises) with the host clock; median / min / max over --runs calls after --warmup
untimed ones. The cells (134 MB at 256^3 with 8-byte cells and more everywhere else) do not
stay in the 126 MB of L2 between objects; the 1-byte mask or slot map (16 / 134 MB) may.

Per object, the classification moves 8 or 16 B of cells plus the 1 B mask it writes in the
single-call route; the batch moves them once for all 8 objects and then reads 1 B of slot map
per object, as the single calls read their mask. The three passes that follow are the same.

Before it prints, the run checks that all three routes give the same bytes on every object.
Prints one JSON line per case and writes the document, with the card's name and power limit
read in the same run, to --out when given.
"""
from __future__ import annotations

import argparse
import ctypes
import json
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
from voxelized_geometry_tools_b200 import device as vdev  # noqa: E402

RESOLUTION = 0.01
OBJECTS = 8


def tagged_cells(n, words, device):
    """[n, n, n, words] int32 cells: occupancy bits, object id, zero padding."""
    occupancy = synthetic.clustered_spheres_occupancy_torch((n, n, n), device)
    axis = torch.arange(n, device=device)
    block = ((axis // 64)[:, None, None] + (axis // 64 * 2)[None, :, None]
             + (axis // 128)[None, None, :])
    cells = torch.zeros((n, n, n, words), dtype=torch.int32, device=device)
    cells[..., 0] = occupancy.view(torch.int32)
    cells[..., 1] = (block % OBJECTS + 1).to(torch.int32)
    return cells


def time_events(call, warmup, runs):
    for _ in range(warmup):
        call()
    torch.cuda.synchronize()
    stream = torch.cuda.current_stream()
    times = []
    for _ in range(runs):
        start = torch.cuda.Event(enable_timing=True)
        stop = torch.cuda.Event(enable_timing=True)
        start.record(stream)
        result = call()
        stop.record(stream)
        stop.synchronize()
        times.append(start.elapsed_time(stop))
    return times, result


def time_host(call, warmup, runs):
    for _ in range(warmup):
        call()
    times = []
    for _ in range(runs):
        begin = time.perf_counter()
        result = call()
        times.append((time.perf_counter() - begin) * 1e3)
    return times, result


def summary(times):
    return {"median_ms": round(statistics.median(times), 4), "min_ms": round(min(times), 4),
            "max_ms": round(max(times), 4)}


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
    sizes = (64, 128) if args.quick else (256, 512)
    ids = list(range(1, OBJECTS + 1))
    id_array = (ctypes.c_uint32 * OBJECTS)(*ids)
    lib = _capi.library()
    result = {"card": card(), "warmup": args.warmup, "runs": args.runs, "objects": OBJECTS,
              "scene": "clustered spheres, object ids 1..8 in blocks of 64 x 128 x 128 voxels",
              "sdf": "float32, unknown_is_filled, no virtual border",
              "timing": "device routes: CUDA events around one call; host entry: host clock",
              "cases": []}
    for n in sizes:
        for cell_bytes in (8, 16):
            cells = tagged_cells(n, cell_bytes // 4, device)
            host_cells = cells.cpu().numpy()
            host_out = np.empty((OBJECTS, n, n, n), dtype=np.float32)
            lows = (ctypes.c_float * OBJECTS)()
            highs = (ctypes.c_float * OBJECTS)()

            def batch():
                return vdev.separate_object_sdfs(cells, RESOLUTION, ids)

            def single_calls():
                return [vdev.signed_distance_field_from_cells(cells, RESOLUTION, [i])
                        for i in ids]

            def host_entry():
                _capi.check(lib.vgt_b200_sdf_per_object_f32(
                    host_cells.ctypes.data, cell_bytes, n, n, n, RESOLUTION, 1, 0, id_array,
                    OBJECTS, 0, host_out.ctypes.data, lows, highs))
                return host_out

            batch_times, (batch_sdfs, batch_min_max) = time_events(batch, args.warmup, args.runs)
            single_times, singles = time_events(single_calls, args.warmup, args.runs)
            host_times, _ = time_host(host_entry, args.warmup, args.runs)

            single_sdfs = torch.stack([sdf for sdf, _ in singles])
            single_min_max = torch.stack([min_max for _, min_max in singles])
            same = (torch.equal(batch_sdfs.view(torch.int32), single_sdfs.view(torch.int32))
                    and torch.equal(batch_min_max.view(torch.int32),
                                    single_min_max.view(torch.int32))
                    and batch_sdfs.cpu().numpy().tobytes() == host_out.tobytes()
                    and batch_min_max[:, 0].cpu().numpy().tobytes()
                    == np.frombuffer(lows, dtype=np.float32).tobytes()
                    and batch_min_max[:, 1].cpu().numpy().tobytes()
                    == np.frombuffer(highs, dtype=np.float32).tobytes())
            if not same:
                raise SystemExit(f"routes disagree at {n}^3, {cell_bytes}-byte cells")
            voxels = n ** 3
            case = {"n": n, "cell_bytes": cell_bytes, "same_bytes_on_all_routes": same,
                    "batch": summary(batch_times),
                    "single_calls": summary(single_times),
                    "host_entry": summary(host_times),
                    "batch_ms_per_object": round(statistics.median(batch_times) / OBJECTS, 4),
                    "single_calls_over_batch": round(statistics.median(single_times)
                                                     / statistics.median(batch_times), 3),
                    "host_entry_over_batch": round(statistics.median(host_times)
                                                   / statistics.median(batch_times), 2),
                    "batch_gvoxels_per_s": round(OBJECTS * voxels
                                                 / statistics.median(batch_times) / 1e6, 1)}
            result["cases"].append(case)
            print(json.dumps(case), flush=True)
            del cells, host_cells, host_out, batch_sdfs, batch_min_max, singles, single_sdfs
            torch.cuda.empty_cache()

    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(result, indent=1) + "\n")
    print(json.dumps({"card": result["card"]}))


if __name__ == "__main__":
    main()
