"""Times the batched SignedDistanceField queries on a device-resident SDF, float and double side by
side, with CUDA events: EstimateLocationDistance, GetLocationCoarseGradient, GetLocationFineGradient
and ProjectLocationOutOfCollisionToMinimumDistance on 1 Mi and 16 Mi points, and the local extrema
map.

    python profiles/time_sdf_queries.py [--out sdf_queries.json] [--warmup 3] [--runs 10] [--quick]

The queries run on the SDF of a 512^3 clustered-spheres grid (0.01 m cells; 512 MB as float, 1 GB
as double, both well beyond the 126 MB of L2) at seeded uniform points in the grid and 15 % of
its extent around it, in random order, under a fixed pose. Every query gathers a few cells per
point at addresses set by the point, so the kernels are bound by gather latency and sector
traffic, not by a compute or a streaming-bandwidth roof: the figure of merit is queries per
second, not a fraction of a roofline. The extrema map runs on the SDF of a 256^3 grid.

Prints one JSON line per case and writes the whole document to --out when given: the card's name
and power limit, read in the same run, then per case the median / min / max milliseconds over
--runs timed calls after --warmup untimed ones, the rate and the share of points with a value.
"""
from __future__ import annotations

import argparse
import json
import statistics
import sys
from pathlib import Path

import numpy as np
import torch

REPO = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(REPO))

from time_connected_components import card  # noqa: E402  (this script's directory)
from voxelized_geometry_tools_b200 import _capi, synthetic  # noqa: E402
from voxelized_geometry_tools_b200 import device as vdev  # noqa: E402

RESOLUTION = 0.01
PROJECTION_MAX_STEPS = 10_000
POSE = np.array([[0.8, -0.6, 0.0, 0.3],
                 [0.6, 0.8, 0.0, -1.2],
                 [0.0, 0.0, 1.0, 0.5],
                 [0.0, 0.0, 0.0, 1.0]])


def fields(n, device):
    occupancy = synthetic.clustered_spheres_occupancy_torch((n, n, n), device)
    single, _ = vdev.signed_distance_field(occupancy, RESOLUTION)
    double, _ = vdev.signed_distance_field_f64(occupancy, RESOLUTION)
    del occupancy
    return {"float": vdev.DeviceSignedDistanceField(single, RESOLUTION, POSE),
            "double": vdev.DeviceSignedDistanceField(double, RESOLUTION, POSE)}


def world_points(n, count, device):
    generator = torch.Generator(device=device).manual_seed(20261021)
    extent = n * RESOLUTION
    grid = (torch.rand((count, 3), generator=generator, device=device, dtype=torch.float64)
            * 1.3 - 0.15) * extent
    rotation = torch.tensor(POSE[:3, :3], device=device)
    return (grid @ rotation.T + torch.tensor(POSE[:3, 3], device=device)).contiguous()


def time_call(call, warmup, runs):
    for _ in range(warmup):
        result = call()
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
    n, n_extrema = (64, 32) if args.quick else (512, 256)
    counts = (1 << 14, 1 << 16) if args.quick else (1 << 20, 1 << 24)
    result = {"card": card(), "warmup": args.warmup, "runs": args.runs,
              "scene": f"clustered spheres {n}^3, resolution {RESOLUTION}, fixed pose",
              "points": "uniform in the grid and 15 % of its extent around it, random order",
              "fine_gradient_window": RESOLUTION,
              "projection": {"minimum_distance": 0.0, "stepsize_multiplier": 0.1,
                             "max_steps": PROJECTION_MAX_STEPS},
              "cases": []}
    sdfs = fields(n, device)
    queries = {
        "EstimateLocationDistance": lambda f, p: f.EstimateLocationDistance(p),
        "GetLocationCoarseGradient": lambda f, p: f.GetLocationCoarseGradient(p, False),
        "GetLocationFineGradient": lambda f, p: f.GetLocationFineGradient(p, RESOLUTION),
        "ProjectLocationOutOfCollisionToMinimumDistance":
            lambda f, p: f.ProjectLocationOutOfCollisionToMinimumDistance(
                p, 0.0, 0.1, PROJECTION_MAX_STEPS),
    }
    for count in counts:
        points = world_points(n, count, device)
        for query, call in queries.items():
            for scalar, field in sdfs.items():
                times, (_, valid) = time_call(lambda: call(field, points), args.warmup, args.runs)
                case = {"query": query, "scalar": scalar, "n": n, "points": count,
                        **summary(times),
                        "mqueries_per_s": round(count / statistics.median(times) / 1e3, 1),
                        "valid_share": round(float((valid == 1).double().mean()), 4)}
                result["cases"].append(case)
                print(json.dumps(case), flush=True)
        del points
    del sdfs
    torch.cuda.empty_cache()

    for scalar, field in fields(n_extrema, device).items():
        times, extrema = time_call(field.ComputeLocalExtremaMap, args.warmup, args.runs)
        cells = n_extrema ** 3
        case = {"query": "ComputeLocalExtremaMap", "scalar": scalar, "n": n_extrema,
                "cells": cells, **summary(times),
                "mcells_per_s": round(cells / statistics.median(times) / 1e3, 1),
                "off_grid_share": round(float(torch.isinf(extrema[..., 0]).double().mean()), 4)}
        result["cases"].append(case)
        print(json.dumps(case), flush=True)

    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(result, indent=1) + "\n")
    print(json.dumps({"card": result["card"]}))


if __name__ == "__main__":
    main()
