"""Times ShardedConnectedComponents.label (one process per GPU, NCCL) on a 1024^3 map of 8-byte
cells (filled balls) at world sizes 1, 2, 4 and 8, against vgt_b200_connected_components_dev on
one GPU. CUDA events around each call after warm-ups, the median of the repeats; every rank's slab
is checked byte for byte against the one-device labelling of the same cells. World sizes above
the number of visible GPUs are reported as skipped. The card's name and power limit are read in
the same run.

    python profiles/time_connected_components_sharded.py [--n 1024] [--warmup 2] [--repeats 7]
                                                         [--out results.json]
"""
import argparse
import json
import os
import socket
import subprocess
import sys
import tempfile
from pathlib import Path

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

REPO = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(REPO))


def spheres_slab(n, x0, x1, device, seed=1024, count=200):
    """Rows [x0, x1) of an n^3 map of 8-byte cells: filled balls, component words all ones."""
    rng = np.random.default_rng(seed)
    x = torch.arange(x0, x1, device=device, dtype=torch.float32).view(-1, 1, 1)
    y = torch.arange(n, device=device, dtype=torch.float32).view(1, -1, 1)
    z = torch.arange(n, device=device, dtype=torch.float32).view(1, 1, -1)
    occupancy = torch.zeros((x1 - x0, n, n), dtype=torch.float32, device=device)
    for _ in range(count):
        cx, cy, cz = rng.uniform(0, n, 3)
        radius = rng.uniform(n / 64, n / 12)
        if cx + radius < x0 or cx - radius >= x1:
            continue
        occupancy[(x - cx) ** 2 + (y - cy) ** 2 + (z - cz) ** 2 <= radius ** 2] = 1.0
    cells = torch.full((x1 - x0, n, n, 2), -1, dtype=torch.int32, device=device)
    cells[..., 0] = occupancy.view(torch.int32)
    return cells


def median_ms(run, warmup, repeats, barrier=None):
    times = []
    for i in range(warmup + repeats):
        if barrier is not None:
            barrier()
        torch.cuda.synchronize()
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        result = run()
        end.record()
        torch.cuda.synchronize()
        if i >= warmup:
            times.append(start.elapsed_time(end))
    return float(np.median(times)), times, result


def _worker(rank, world, port, n, warmup, repeats, result_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        from voxelized_geometry_tools_b200 import device as vdev
        from voxelized_geometry_tools_b200.sharded import ShardedConnectedComponents
        plan = ShardedConnectedComponents((n, n, n))
        x0, x1 = plan.x_range
        original = spheres_slab(n, x0, x1, dev)
        # the one-device labelling of the whole map, this rank's rows kept for the check
        full = spheres_slab(n, 0, n, dev)
        count_dev = vdev.connected_components(full)
        want = full[x0:x1].clone()
        want_count = int(count_dev.item())
        dev_ms = None
        if rank == 0 and world == 1:
            dev_ms, dev_times, _ = median_ms(lambda: vdev.connected_components(full), warmup,
                                             repeats)
        del full
        slab = original.clone()
        ms, times, count = median_ms(lambda: plan.label(slab), warmup, repeats,
                                     barrier=lambda: dist.barrier(device_ids=[rank]))
        same = bool(torch.equal(slab, want)) and count == want_count
        slowest = torch.tensor([ms], device=dev)
        dist.all_reduce(slowest, op=dist.ReduceOp.MAX)
        Path(result_dir, f"w{world}_r{rank}.json").write_text(json.dumps(dict(
            world=world, rank=rank, label_ms_median=ms, label_ms=times, count=count,
            want_count=want_count, bytes_equal=same, slowest_rank_median_ms=float(slowest.item()),
            dev_ms_median=dev_ms, dev_ms=dev_times if dev_ms is not None else None)))
    finally:
        dist.destroy_process_group()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument("--n", type=int, default=1024)
    parser.add_argument("--warmup", type=int, default=2)
    parser.add_argument("--repeats", type=int, default=7)
    parser.add_argument("--worlds", default="1,2,4,8")
    parser.add_argument("--out", default=None)
    args = parser.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures on the GPU only")
    gpus = torch.cuda.device_count()
    cards = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True).stdout.strip().splitlines()
    report = dict(n=args.n, cell_bytes=8, warmup=args.warmup, repeats=args.repeats,
                  gpus_visible=gpus, cards=cards, worlds={}, skipped=[])
    for world in [int(w) for w in args.worlds.split(",")]:
        if world > gpus:
            report["skipped"].append(world)
            continue
        with tempfile.TemporaryDirectory() as result_dir:
            mp.spawn(_worker, args=(world, _free_port(), args.n, args.warmup, args.repeats,
                                    result_dir), nprocs=world, join=True)
            ranks = [json.loads(Path(result_dir, f"w{world}_r{r}.json").read_text())
                     for r in range(world)]
        report["worlds"][world] = dict(
            label_ms_median=ranks[0]["slowest_rank_median_ms"],
            bytes_equal=all(r["bytes_equal"] for r in ranks),
            counts=sorted({r["count"] for r in ranks}), ranks=ranks)
        if world == 1:
            report["dev_ms_median"] = ranks[0]["dev_ms_median"]
    text = json.dumps(report, indent=1)
    print(text)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(text)
    if not all(w["bytes_equal"] for w in report["worlds"].values()):
        raise SystemExit("the sharded labelling differs from the one-device entry")


if __name__ == "__main__":
    main()
