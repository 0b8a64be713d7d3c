"""Times the x-slab connected-component labelling (vgt_b200_connected_components_multi) against
the one-device host entry (vgt_b200_connected_components) on the same pageable cells, and splits
one call of each device list into its stages with torch.profiler in a separate pass.

    python profiles/time_connected_components_multi.py [--out connected_components_multi.json]
                                                       [--warmup 2] [--runs 5] [--quick]
                                                       [--no-big]

Both entries are synchronous host calls that end in a device synchronise, so a host clock around
each call is its end-to-end time (PCIe copies of the whole map in and out included). Every timed
result is checked against the one-device entry, byte for byte. The map of more than 2^32 cells
(4096 x 1024 x 1025, 8-byte cells, the scene of tests/test_gpu_connected_components_slabs.py)
runs on [0, 0] and [0, 1] when host RAM and device memory allow. Writes the card's name and power
limit, read in the same run, beside the numbers.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import time
from collections import defaultdict
from pathlib import Path

import numpy as np
import torch

REPO = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(REPO))

from voxelized_geometry_tools_b200 import _capi, synthetic  # noqa: E402
from voxelized_geometry_tools_b200.grids import OCCUPANCY_COMPONENT_CELL  # noqa: E402


def card():
    try:
        text = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit",
                               "--format=csv,noheader"], capture_output=True, text=True,
                              timeout=60).stdout.strip().splitlines()
        name, power = (part.strip() for part in text[0].split(","))
        return {"name": name, "power_limit": power, "devices": len(text)}
    except Exception as error:  # recorded, not fatal
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"unknown ({error})"}


def cells_for(scene, n):
    cells = np.zeros((n, n, n), dtype=OCCUPANCY_COMPONENT_CELL)
    if scene == "spheres":
        cells["occupancy"] = synthetic.clustered_spheres_occupancy((n, n, n))
    elif scene == "noise50":
        rng = np.random.default_rng(50)
        for x in range(n):
            cells["occupancy"][x] = (rng.random((n, n)) < 0.5).astype(np.float32)
    else:
        raise ValueError(scene)
    return cells


def call(cells, devices):
    lib = _capi.library()
    count = ctypes.c_uint32()
    if devices is None:
        code = lib.vgt_b200_connected_components(cells.ctypes.data, cells.dtype.itemsize,
                                                 *cells.shape, 0, ctypes.byref(count))
    else:
        listed = (ctypes.c_int * len(devices))(*devices)
        code = lib.vgt_b200_connected_components_multi(cells.ctypes.data, cells.dtype.itemsize,
                                                       *cells.shape, listed, len(devices),
                                                       ctypes.byref(count))
    _capi.check(code)
    return int(count.value)


def timed(cells, devices, warmup, runs):
    work = cells.copy()
    for _ in range(warmup):
        call(work, devices)
    times = []
    for _ in range(runs):
        begin = time.perf_counter()
        count = call(work, devices)
        times.append((time.perf_counter() - begin) * 1e3)
    return times, count, work


STAGES = [  # (stage, substrings of kernel names), first match wins
    ("face", ("FaceRootsKernel", "FaceEdgesKernel")),
    ("resolve", ("NodeInitKernel", "NodeUnionKernel", "NodeFlattenKernel", "RadixSort",
                 "Select", "Unique")),
    ("numbering", ("GlobalRootBitsInitKernel", "ClearMergedBitsKernel", "BitCountsKernel",
                   "FinalIdsKernel", "PublishNodeIdsKernel", "NodeIdsFromRootsKernel",
                   "ApplyNodeIdsKernel")),
    ("write", ("WriteSlabComponentsKernel", "WriteComponentsKernel")),
    ("local", ("InitRunsKernel", "MergeKernel", "MarkRootsKernel", "Scan")),
    ("copy_h2d", ("HtoD",)),
    ("copy_d2h", ("DtoH",)),
    ("copy_d2d", ("DtoD",)),
]


def stage_of(name):
    for stage, keys in STAGES:
        if any(key in name for key in keys):
            return stage
    return "other"


def profile_split(cells, devices):
    """Device time per stage (summed over devices and streams) of one call, after a warm-up."""
    from torch.profiler import ProfilerActivity, profile
    work = cells.copy()
    call(work, devices)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        call(work, devices)
    stages = defaultdict(float)
    kernels = defaultdict(float)
    for event in prof.events():
        if event.device_type != torch.autograd.DeviceType.CUDA:
            continue
        us = event.device_time_total if hasattr(event, "device_time_total") \
            else event.cuda_time_total
        stages[stage_of(event.name)] += us / 1e3
        kernels[event.name[:120]] += us / 1e3
    return ({k: round(v, 3) for k, v in sorted(stages.items())},
            {k: round(v, 3) for k, v in sorted(kernels.items(), key=lambda kv: -kv[1])[:25]})


def big_map():
    from tests.test_gpu_connected_components_slabs import BIG, big_scene_plane
    cells = np.empty(BIG, dtype=OCCUPANCY_COMPONENT_CELL)
    for x in range(BIG[0]):
        cells["occupancy"][x] = big_scene_plane(x)[0]
        cells["component"][x] = 0
    return cells


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument("--out", default=None, help="file for the JSON document")
    parser.add_argument("--warmup", type=int, default=2)
    parser.add_argument("--runs", type=int, default=5)
    parser.add_argument("--quick", action="store_true", help="small sizes (a rehearsal)")
    parser.add_argument("--no-big", action="store_true", help="skip the > 2^32-cell map")
    args = parser.parse_args()
    if not torch.cuda.is_available() or _capi.device_count() == 0:
        raise SystemExit("no usable CUDA device: nothing to measure")
    count = _capi.device_count()
    lists = [[0, 0], [0, 1], list(range(min(count, 4))), list(range(min(count, 8)))]
    lists = [d for k, d in enumerate(lists) if max(d) < count and d not in lists[:k]]
    sizes = (64, 96) if args.quick else (512, 1024)
    result = {"card": card(), "warmup": args.warmup, "runs": args.runs,
              "timing": "host clock around the synchronous host entry; median of runs",
              "cases": [], "split": []}

    def record(case):
        result["cases"].append(case)
        print(json.dumps(case), flush=True)

    for n in sizes:
        for scene in ("spheres", "noise50"):
            cells = cells_for(scene, n)
            base, base_count, want = timed(cells, None, args.warmup, args.runs)
            record({"entry": "one device", "devices": [0], "scene": scene, "n": n,
                    "median_ms": round(statistics.median(base), 3),
                    "min_ms": round(min(base), 3), "max_ms": round(max(base), 3),
                    "components": base_count})
            for devices in lists:
                times, got_count, got = timed(cells, devices, args.warmup, args.runs)
                assert got_count == base_count and got.tobytes() == want.tobytes(), devices
                record({"entry": "multi", "devices": devices, "scene": scene, "n": n,
                        "median_ms": round(statistics.median(times), 3),
                        "min_ms": round(min(times), 3), "max_ms": round(max(times), 3),
                        "vs_one_device": round(statistics.median(times)
                                               / statistics.median(base), 3),
                        "components": got_count})
                del got
            del want
            if scene == "spheres":
                for devices in [None] + lists:
                    stages, kernels = profile_split(cells, devices)
                    result["split"].append({"devices": devices or [0], "entry": "multi"
                                            if devices else "one device", "scene": scene,
                                            "n": n, "stage_ms": stages, "top_kernels": kernels})
                    print(json.dumps(result["split"][-1]["stage_ms"]), flush=True)
            del cells

    host = os.sysconf("SC_PAGE_SIZE") * os.sysconf("SC_PHYS_PAGES")
    device_memory = torch.cuda.get_device_properties(0).total_memory
    if args.no_big or args.quick or host < 100e9 or device_memory < 100e9:
        result["big"] = {"skipped": f"host {host / 1e9:.0f} GB, device {device_memory / 1e9:.0f} "
                                    f"GB, flags no_big={args.no_big} quick={args.quick}"}
    else:
        cells = big_map()
        for devices in [[0, 0]] + ([[0, 1]] if count >= 2 else []):
            times, got_count, _ = timed(cells, devices, 1, 2)
            record({"entry": "multi", "devices": devices, "scene": "big_walls_bar_u",
                    "shape": list(cells.shape), "median_ms": round(statistics.median(times), 3),
                    "min_ms": round(min(times), 3), "max_ms": round(max(times), 3),
                    "components": got_count})
        stages, kernels = profile_split(cells, [0, 0])
        result["split"].append({"devices": [0, 0], "entry": "multi", "scene": "big_walls_bar_u",
                                "shape": list(cells.shape), "stage_ms": stages,
                                "top_kernels": kernels})
        del cells

    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(result, indent=1) + "\n")
    print(json.dumps({"card": result["card"]}))


if __name__ == "__main__":
    main()
