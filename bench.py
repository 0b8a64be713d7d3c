#!/usr/bin/env python3
"""Benchmark of the occupancy -> SDF hot path on B200 (BASELINE.json metric: SDF Gvoxels/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

One "step" = one ExtractSignedDistanceField<float> over one synthetic occupancy grid.
Workload (weak scaling, 512^3 voxels per GPU, x-slab sharded):
    N=1  512 x 512 x 512      (BASELINE config 2: clustered spheres ~10 % filled, 1 % unknown)
    N=2  1024 x 512 x 512
    N=4  1024 x 1024 x 512
    N=8  1024 x 1024 x 1024   (BASELINE config 4)
Every grid is far larger than the 126 MB L2 (>= 512 MiB in, >= 512 MiB out), so no L2 flush is
needed between iterations.

value  = voxels / s with the occupancy already resident in HBM (CUDA events, max over ranks).
e2e    = the same through the drop-in host entry point vgt_b200_sdf_f32 (host buffers in, host
         buffers out; H2D + D2H inside the timed region), per rank on its slab at N>1.
roofline: the dominant kernel (the slowest of the three passes, normally x + finalize), algorithmic 8 B/voxel, timed with CUDA events
         between the kernels on the launching stream (vgt_b200_sdf_f32_dev_profile).
cpu_baseline / --impl reference: the reference's own EDT source (oracle/_ref) when it was built,
         else our restatement of it, on the host cores over the SAME grid (all host threads).
"""
from __future__ import annotations

import argparse
import os

# (idle OpenMP workers of the CPU reference legs sleep instead of spinning next to the thread
# that launches kernels; must be set before libgomp is loaded)
os.environ.setdefault("OMP_WAIT_POLICY", "PASSIVE")
import ctypes  # noqa: E402
import json  # noqa: E402
import statistics  # noqa: E402
import subprocess
import sys
import threading
import time
from pathlib import Path

REPO = Path(__file__).resolve().parent
if str(REPO) not in sys.path:
    sys.path.insert(0, str(REPO))

RESOLUTION = 0.02
SDF_BYTES_PER_VOXEL = 24           # 3 passes x (4 B in + 4 B out), SURVEY.md section 8d
PASS_BYTES_PER_VOXEL = 8
PASS_NAMES = ["ScanContiguousAxisRegistersKernel (z)", "EnvelopeAxisWindowKernel (y)",
              "EnvelopeAxisWindowKernel (x + finalize)"]
NCU_TRAFFIC_FILE = REPO / "profiles" / "ncu_traffic.json"


def ncu_dram_bytes_per_launch(dims, kernel, check_build=True):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed
    `ncu --set full` capture of this very workload (profiles/ncu_traffic.json, written by
    profiles/ncu_traffic.py from the .ncu-rep); None for anything not captured, and None when
    the capture was taken from another build (the table records the hash of the kernel sources)."""
    try:
        table = json.loads(NCU_TRAFFIC_FILE.read_text())
        entry = table["x".join(map(str, dims))][kernel]
        from voxelized_geometry_tools_b200 import build as cuda_build
        if check_build and entry.get("sources_sha1") != cuda_build._sources_signature():
            return None     # captured from another build of the kernels: not this library's traffic
        return float(entry["dram_bytes_read"]) + float(entry["dram_bytes_write"])
    except Exception:
        return None


def workload_dims(n_gpus: int):
    return {1: (512, 512, 512), 2: (1024, 512, 512), 4: (1024, 1024, 512),
            8: (1024, 1024, 1024)}.get(n_gpus, (512 * n_gpus, 512, 512))


def measured_peaks():
    path = REPO / "MEASURED_PEAKS.json"
    if path.exists():
        try:
            return float(json.loads(path.read_text())["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


class ClockSampler:
    """Samples nvidia-smi clocks and throttle reasons during the timed region."""

    QUERY = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index: int):
        self.device_index = device_index
        self.samples = []
        self._stop = threading.Event()
        self._thread = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(
                    ["nvidia-smi", f"--id={self.device_index}", f"--query-gpu={self.QUERY}",
                     "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                fields = [f.strip() for f in out.stdout.strip().split(",")]
                if len(fields) >= 6:
                    self.samples.append(fields)
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        self._thread.join(timeout=10)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = [float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [name for i, name in enumerate(names)
                   if any(s[2 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": float(self.samples[0][1]) if self.samples[0][1].isdigit() else None,
                "reasons": reasons, "samples": len(self.samples)}


def host_threads() -> int:
    """The host threads this process may use. Passed explicitly to the CPU path: under
    torch.distributed.run OMP_NUM_THREADS is forced to 1, which must not apply to it."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def available_host_bytes() -> int:
    try:
        import psutil
        return int(psutil.virtual_memory().available)
    except Exception:
        return 0


def cpu_reference_arm(steps: int, warmup: int, dims):
    """Times the CPU path on the host cores over the grid `dims`: kind 'reference' when
    oracle/_ref exists (the reference's own signed_distance_field_generation.cpp), else 'port'
    (our restatement). The grid is the workload itself when host memory allows (the reference
    keeps two double fields: 24 B per voxel with occupancy and SDF), else the largest leading
    part of it along x that fits; the result is per voxel either way."""
    import numpy as np
    from oracle import oracle
    from voxelized_geometry_tools_b200 import synthetic
    dims = tuple(int(d) for d in dims)
    wanted = dims
    budget = available_host_bytes() * 0.6
    while budget and 28.0 * float(np.prod(dims)) > budget and dims[0] > 64:
        dims = (dims[0] // 2, dims[1], dims[2])
    # (the x-range of the workload grid itself, not a smaller grid of another shape; generated
    # with torch on the GPU when there is one - identical bits, seconds instead of a minute)
    occupancy = None
    try:
        import torch
        if torch.cuda.is_available():
            occupancy = synthetic.clustered_spheres_occupancy_torch(
                wanted, torch.device("cuda", 0), x_range=(0, dims[0])).cpu().numpy()
            torch.cuda.empty_cache()
    except Exception:
        occupancy = None
    if occupancy is None:
        occupancy = synthetic.clustered_spheres_occupancy(wanted, x_range=(0, dims[0]))
    threads = host_threads()
    kind = "port"
    runner = lambda: oracle.sdf(occupancy, RESOLUTION, threads=threads)  # noqa: E731
    try:
        from oracle import reference_oracle
        if reference_oracle.available():
            kind = "reference"
            runner = lambda: reference_oracle.sdf(occupancy, RESOLUTION, threads=threads)  # noqa: E731
    except Exception:
        pass
    for _ in range(warmup):
        runner()
    times = []
    for _ in range(steps):
        begin = time.perf_counter()
        runner()
        times.append(time.perf_counter() - begin)
    seconds = sum(times) / len(times)
    voxels = float(np.prod(dims))
    same = dims == wanted
    return {"value": voxels / seconds / 1e9, "unit": "Gvoxels/s", "cores": threads, "kind": kind,
            "sample": f"{'x'.join(map(str, dims))} clustered-spheres grid ("
                      + ("the whole workload" if same else
                         f"the first {dims[0]} x-planes of the {'x'.join(map(str, wanted))} "
                         "workload: host memory; per-voxel figure")
                      + f"), ExtractSignedDistanceField<float>, {steps} run(s), "
                      f"{seconds:.3f} s each, {threads} threads",
            "seconds_per_sample": seconds, "same_config": same, "sample_dims": list(dims)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = max(1, min(args.steps, 3))
    warmup = min(args.warmup, 1)
    dims = workload_dims(args.gpus)
    baseline = cpu_reference_arm(steps, warmup, dims)
    line = {
        "impl": "reference", "metric": "sdf_gvoxels_per_s", "value": baseline["value"],
        "unit": "Gvoxels/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
        "ms_per_step": baseline["seconds_per_sample"] * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{'x'.join(map(str, dims))} occupancy -> SDF<float> "
                               "(clustered spheres ~10% filled, 1% unknown)",
                   "sample": baseline["sample"], "same_config": baseline["same_config"]},
        "cpu_baseline": {k: baseline[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": baseline["value"], "unit": "Gvoxels/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def time_cpp_adapter(n: int):
    """The real drop-in call (C++ host adapter compiled against the reference's headers): the
    prebuilt adapter_test binaries time b200::ExtractSignedDistanceFieldFromOccupancyMap on an
    n^3 map with std::vector storage, piece by piece. None when they were not built."""
    build = REPO / "voxelized_geometry_tools_b200" / "cpp" / "_build"
    timed = {}
    for key, name in (("reference_lock", "adapter_test"),
                      ("with_known_extrema_accessor", "adapter_test_fast_lock")):
        binary = build / name
        if not binary.exists():
            continue
        try:
            out = subprocess.run([str(binary), "--time", str(n)], capture_output=True, text=True,
                                 timeout=600)
            timed[key] = json.loads(out.stdout.strip().splitlines()[-1])
        except Exception as error:     # a timing aid must not break the bench line
            timed[key] = {"error": repr(error)}
    return timed or None


def sharded_parity(sharded, vdev, synthetic, plan, result, dims, dev, rank, world):
    """Outside the timed region: (1) the sharded SDF of the bench grid == the one-GPU SDF of the
    same grid, bit for bit, slab by slab on rank 0 (plus min/max); (2) a 256^3 grid through the
    same sharded path == the CPU oracle (the reference's own EDT source when oracle/_ref is
    there). The oracle is only the checker here."""
    import numpy as np
    import torch
    import torch.distributed as dist
    sdf, min_max = result
    equal = True
    if rank == 0:
        whole = synthetic.clustered_spheres_occupancy_torch(dims, dev)
        single, single_min_max = vdev.signed_distance_field(whole, RESOLUTION)
        del whole
        equal = single_min_max.tolist() == min_max.tolist()
        for peer in range(world):
            y0, y1 = sharded.split_range(dims[1], world, peer)
            if peer == 0:
                piece = sdf
            else:
                piece = torch.empty((dims[0], y1 - y0, dims[2]), dtype=torch.float32, device=dev)
                dist.recv(piece, src=peer)
            equal = equal and bool(torch.equal(piece, single[:, y0:y1, :]))
        del single
    else:
        dist.send(sdf.contiguous(), dst=0)
    torch.cuda.empty_cache()
    small = (256, 256, 256)
    small_plan = sharded.ShardedSignedDistanceField(small, rank=rank, world_size=world)
    slab = synthetic.clustered_spheres_occupancy_torch(small, dev, x_range=small_plan.x_range)
    small_sdf, _ = small_plan.extract(slab, RESOLUTION)
    full = small_plan.gather_to_host(small_sdf)
    oracle_ok, oracle_kind = None, None
    if rank == 0:
        from oracle import oracle
        occupancy = synthetic.clustered_spheres_occupancy(small)
        oracle_kind = "port"
        want = None
        try:
            from oracle import reference_oracle
            if reference_oracle.available():
                want, _ = reference_oracle.sdf(occupancy, RESOLUTION, threads=host_threads())
                oracle_kind = "reference"
        except Exception:
            want = None
        if want is None:
            want, _ = oracle.sdf(occupancy, RESOLUTION, threads=host_threads())
        oracle_ok = bool(np.array_equal(full.numpy(), want))
    return {"equals_single_gpu": bool(equal), "oracle_256": oracle_ok, "oracle_kind": oracle_kind,
            "grid": "x".join(map(str, dims)), "exchange": plan.exchange_used}


def strong_scaling_1024(sharded, vdev, synthetic, dev, rank, world, steps):
    """BASELINE config 4: the SAME 1024^3 grid at every N (strong scaling), device-resident."""
    import torch
    import torch.distributed as dist
    dims = (1024, 1024, 1024)
    distributed = world > 1
    if distributed:
        plan = sharded.ShardedSignedDistanceField(dims, rank=rank, world_size=world)
        occupancy = synthetic.clustered_spheres_occupancy_torch(dims, dev, x_range=plan.x_range)
        step = lambda: plan.extract(occupancy, 0.01)  # noqa: E731
    else:
        occupancy = synthetic.clustered_spheres_occupancy_torch(dims, dev)
        out = torch.empty_like(occupancy)
        min_max = torch.empty(2, dtype=torch.float32, device=dev)
        step = lambda: vdev.signed_distance_field(occupancy, 0.01, out=out, min_max=min_max)  # noqa: E731
    for _ in range(3):
        step()
    torch.cuda.synchronize(dev)
    if distributed:
        dist.barrier()
    # every step between its own pair of events (no host synchronisation in between): the mean
    # is the number reported, the per-step list shows whether a step paid for an allocation
    marks = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    marks[0].record()
    for index in range(steps):
        step()
        marks[index + 1].record()
    torch.cuda.synchronize(dev)
    step_ms = [marks[i].elapsed_time(marks[i + 1]) for i in range(steps)]
    mean_ms = marks[0].elapsed_time(marks[steps]) / steps
    # (the median step: a step that has to grow the stream-ordered memory pool by the 4 GiB
    # scratch pays ~30 ms for it once; the list and the mean are reported next to it)
    ms = statistics.median(step_ms)
    if distributed:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
    voxels = 1024.0 ** 3
    peak, _ = measured_peaks()
    return {"config": "1024^3 occupancy -> SDF<float> @0.01 m, the same grid at every N",
            "scaling": "strong", "n_gpus": world, "ms_per_step": ms,
            "step_ms": [round(v, 3) for v in step_ms], "mean_ms_per_step": mean_ms,
            "value": voxels / (ms * 1e-3) / 1e9, "unit": "Gvoxels/s",
            "hbm_roofline_frac_24B": SDF_BYTES_PER_VOXEL * voxels / (ms * 1e-3) / 1e9
            / (peak * world)}


def config5_2048(sharded, vdev, synthetic, dev, rank, world, steps):
    """BASELINE config 5 at 8 GPUs: the 2048^3 clustered-spheres grid (8.6 Gvoxel), slab-sharded,
    generated on the devices; device-timed like the main line, and checked against a one-GPU run
    of the whole grid on rank 0 (exact checksums of the float bit patterns, slab by slab)."""
    import torch
    import torch.distributed as dist
    dims = (2048, 2048, 2048)
    resolution = 0.01

    def checksum(sdf):
        bits = sdf.contiguous().view(torch.int32).to(torch.int64)
        weights = torch.arange(bits.numel(), device=bits.device, dtype=torch.int64).view_as(bits) % 1021
        return int(bits.sum().item()), int((bits * (weights + 1)).sum().item())

    plan = sharded.ShardedSignedDistanceField(dims, rank=rank, world_size=world)
    occupancy = synthetic.clustered_spheres_occupancy_torch(dims, dev, x_range=plan.x_range)
    sdf, min_max = plan.extract(occupancy, resolution)
    torch.cuda.synchronize(dev)
    mine = checksum(sdf)
    del sdf
    gathered = [None] * world
    dist.all_gather_object(gathered, mine)
    for _ in range(2):
        plan.extract(occupancy, resolution)
    torch.cuda.synchronize(dev)
    dist.barrier()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(steps):
        plan.extract(occupancy, resolution)
    stop.record()
    torch.cuda.synchronize(dev)
    ms = start.elapsed_time(stop) / steps
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    del occupancy
    torch.cuda.empty_cache()
    same = None
    if rank == 0:
        whole = synthetic.clustered_spheres_occupancy_torch(dims, dev)
        torch.cuda.empty_cache()
        single, single_min_max = vdev.signed_distance_field(whole, resolution)
        del whole
        same = single_min_max.tolist() == min_max.tolist()
        for peer in range(world):
            y0, y1 = sharded.split_range(dims[1], world, peer)
            same = same and checksum(single[:, y0:y1, :]) == tuple(gathered[peer])
        del single
        torch.cuda.empty_cache()
    dist.barrier()
    voxels = float(dims[0]) * dims[1] * dims[2]
    peak, _ = measured_peaks()
    nvlink_bytes = 4.0 * voxels / world * (world - 1) / world
    return {"config": "2048^3 occupancy -> SDF<float> @0.01 m across 8 GPUs (BASELINE config 5)",
            "n_gpus": world, "ms_per_step": ms, "value": voxels / (ms * 1e-3) / 1e9,
            "unit": "Gvoxels/s", "equals_single_gpu": same,
            "hbm_roofline_frac_24B": SDF_BYTES_PER_VOXEL * voxels / (ms * 1e-3) / 1e9
            / (peak * world),
            "nvlink_floor_ms": nvlink_bytes / 770e9 * 1e3,
            "hbm_floor_ms": SDF_BYTES_PER_VOXEL * voxels / world / (peak * 1e9) * 1e3}


DUMP_SAMPLE_VOXELS = 4 << 20


def dump_outputs(directory, sdf, min_max, rank=0, world=1):
    """Writes what the last timed step returned, so that two builds can be compared output for
    output: the SDF's (min, max) and the SDF at a fixed, seeded sample of up to 4 Mi distinct
    voxel positions in all (the whole field is 512 MiB per GPU), with the flat [x, y, z] indices
    of the sample. Files: sdf_min_max.npy, sdf_sample.npy, sdf_sample_index.npy (float64 holds
    every index exactly); at most 48 MiB in all. At N > 1 every rank samples its own y-slab
    (4 Mi / N positions, indices within the slab) into sdf_sample_rank<r>.npy and
    sdf_sample_index_rank<r>.npy, and rank 0 writes the global (min, max)."""
    import numpy as np
    import torch
    directory = Path(directory)
    directory.mkdir(parents=True, exist_ok=True)
    flat = sdf.reshape(-1)
    index = np.unique(np.random.default_rng(rank).integers(
        0, flat.numel(), min(flat.numel(), DUMP_SAMPLE_VOXELS // world)))
    values = flat[torch.from_numpy(index).to(flat.device)].cpu().numpy()
    suffix = "" if world == 1 else f"_rank{rank}"
    if rank == 0:
        np.save(directory / "sdf_min_max.npy", min_max.cpu().numpy().astype(np.float32))
    np.save(directory / f"sdf_sample{suffix}.npy", values.astype(np.float32))
    np.save(directory / f"sdf_sample_index{suffix}.npy", index.astype(np.float64))


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from voxelized_geometry_tools_b200 import _capi, device as vdev, sharded, synthetic

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise _capi.BackendUnavailable("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    distributed = world > 1
    if distributed:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    n_gpus = world if distributed else 1
    dims = workload_dims(n_gpus)
    voxels = float(np.prod(dims))

    plan = sharded.ShardedSignedDistanceField(dims, rank=rank, world_size=n_gpus,
                                              chunks=args.chunks, exchange=args.exchange) \
        if distributed else None
    x_range = plan.x_range if distributed else (0, dims[0])
    occupancy = synthetic.clustered_spheres_occupancy_torch(dims, dev, x_range=x_range)
    torch.cuda.synchronize(dev)

    def barrier():
        if distributed:
            dist.barrier()
        torch.cuda.synchronize(dev)

    out = None if distributed else torch.empty_like(occupancy)
    min_max = torch.empty(2, dtype=torch.float32, device=dev)

    def step():
        if distributed:
            return plan.extract(occupancy, RESOLUTION)
        return vdev.signed_distance_field(occupancy, RESOLUTION, out=out, min_max=min_max)

    for _ in range(max(3, args.warmup)):
        result = step()
    barrier()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    count_launches = _capi.library().vgt_b200_kernel_launch_count
    with ClockSampler(local_rank) as sampler:
        barrier()
        launches_before = count_launches()
        start.record()
        for _ in range(args.steps):
            result = step()
        stop.record()
        launches = count_launches() - launches_before     # this rank's kernels, counted
        barrier()
    elapsed_ms = start.elapsed_time(stop)
    if distributed:
        t = torch.tensor([elapsed_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms = float(t.item())
    ms_per_step = elapsed_ms / args.steps
    value = voxels / (ms_per_step * 1e-3) / 1e9
    sdf_min_max = [float(v) for v in result[1].tolist()]
    # (before the legs below: the per-kernel timing writes into the same output buffer)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *result, rank=rank, world=n_gpus)

    stage_ms = None
    if distributed:
        plan.profile = True
        collected = []
        for _ in range(3):
            plan.extract(occupancy, RESOLUTION)
            torch.cuda.synchronize(dev)
            collected.append(plan.stage_ms())
        plan.profile = False
        stage_ms = {k: statistics.mean(c[k] for c in collected) for k in collected[0]}

    parity = None
    if distributed and not args.skip_parity:
        parity = sharded_parity(sharded, vdev, synthetic, plan, result, dims, dev, rank, n_gpus)

    # ---- per-kernel timing for the roofline (rank-local grid, events between the kernels) ----
    pass_ms = None
    if not distributed:
        samples = [vdev.signed_distance_field_profile(occupancy, RESOLUTION, out, min_max,
                                                      kernels=True)
                   for _ in range(max(3, args.steps))]
        pass_ms = [statistics.mean(s[i] for s in samples) for i in range(3)]
        # the launch duration of each pass's main kernel (the z scan is one launch; a strided
        # pass is pilot probe + decision + window kernel + stack kernel over the hand-over list)
        kernel_ms = [pass_ms[0]] + [statistics.mean(s[i] for s in samples) or pass_ms[i - 2]
                                    for i in (3, 4)]
    peak, peak_kind = measured_peaks()
    roofline = None
    if pass_ms is not None:
        dominant = max(range(3), key=lambda i: kernel_ms[i])
        names = PASS_NAMES
        achieved = PASS_BYTES_PER_VOXEL * voxels / (kernel_ms[dominant] * 1e-3) / 1e9
        roofline = {"bound": "hbm", "kernel": names[dominant], "achieved": achieved, "peak": peak,
                    "unit": "GB/s", "frac": achieved / peak,
                    "traffic": ncu_dram_bytes_per_launch(dims, names[dominant]),
                    "traffic_source": "profiles/ncu_traffic.json (ncu --set full, same workload)",
                    "peak_kind": peak_kind,
                    "algorithmic_bytes_per_launch": PASS_BYTES_PER_VOXEL * voxels,
                    "kernel_ms": {"z_scan": kernel_ms[0], "y_envelope_window": kernel_ms[1],
                                  "x_envelope_window_finalize": kernel_ms[2]},
                    "kernel_frac_of_peak": {
                        name: PASS_BYTES_PER_VOXEL * voxels / (ms * 1e-3) / 1e9 / peak
                        for name, ms in zip(("z_scan", "y_envelope_window",
                                             "x_envelope_window_finalize"), kernel_ms)},
                    "pass_ms": {"z_scan": pass_ms[0], "y_envelope": pass_ms[1],
                                "x_envelope_finalize": pass_ms[2]},
                    "pass_note": ("a strided pass = pilot probe + decision + window kernel + "
                                  "stack kernel over the hand-over list; frac is the dominant "
                                  "KERNEL's launch duration"),
                    "pass_frac_of_peak": {
                        name: PASS_BYTES_PER_VOXEL * voxels / (ms * 1e-3) / 1e9 / peak
                        for name, ms in zip(("z_scan", "y_envelope", "x_envelope_finalize"),
                                            pass_ms)},
                    "whole_sdf": {"achieved": SDF_BYTES_PER_VOXEL * voxels / (ms_per_step * 1e-3) / 1e9,
                                  "frac": SDF_BYTES_PER_VOXEL * voxels / (ms_per_step * 1e-3) / 1e9
                                  / (peak * n_gpus),
                                  "bytes_per_voxel": SDF_BYTES_PER_VOXEL}}
    else:
        whole = SDF_BYTES_PER_VOXEL * voxels / (ms_per_step * 1e-3) / 1e9
        nvlink_bytes = 4.0 * (voxels / n_gpus) * (n_gpus - 1) / n_gpus   # per GPU, per direction
        roofline = {"bound": "hbm", "kernel": "whole SDF (3 passes + all-to-all)",
                    "achieved": whole, "peak": peak * n_gpus, "unit": "GB/s",
                    "frac": whole / (peak * n_gpus), "traffic": None, "peak_kind": peak_kind,
                    "rank0_stage_ms": stage_ms, "exchange_chunks": args.chunks,
                    "exchange": plan.exchange_used,
                    "nvlink_bytes_per_gpu_per_direction": nvlink_bytes,
                    "nvlink_floor_ms_at_770GBs": nvlink_bytes / 770e9 * 1e3,
                    "hbm_floor_ms": SDF_BYTES_PER_VOXEL * (voxels / n_gpus) / (peak * 1e9) * 1e3}

    # ---- BASELINE config 4 (the same 1024^3 grid at every N). Runs BEFORE the legs that time
    # the CPU reference: idle OpenMP workers spin for a while after a parallel region and starve
    # the launching thread (measured: 10.8 ms instead of 6.7 ms per 1024^3 SDF at N = 1).
    strong = None
    if not args.skip_strong:
        if n_gpus == 8:
            # (the N = 8 bench grid IS the 1024^3 grid)
            strong = {"config": "1024^3 occupancy -> SDF<float>, the same grid at every N",
                      "scaling": "strong", "n_gpus": 8, "ms_per_step": ms_per_step,
                      "value": value, "unit": "Gvoxels/s",
                      "hbm_roofline_frac_24B": SDF_BYTES_PER_VOXEL * voxels
                      / (ms_per_step * 1e-3) / 1e9 / (peak * n_gpus)}
        else:
            strong = strong_scaling_1024(sharded, vdev, synthetic, dev, rank, n_gpus,
                                         max(3, min(args.steps, 10)))

    # ---- end to end through the host C-ABI (pinned host buffers, H2D + D2H timed) ----
    lib = _capi.library()
    local_shape = tuple(occupancy.shape)
    host_in = torch.empty(local_shape, dtype=torch.float32).pin_memory()
    host_in.copy_(occupancy)
    host_out = torch.empty(local_shape, dtype=torch.float32).pin_memory()
    torch.cuda.synchronize(dev)
    e2e = None
    if not distributed:
        lo, hi = ctypes.c_float(), ctypes.c_float()

        def host_step():
            code = lib.vgt_b200_sdf_f32(host_in.data_ptr(), *local_shape, RESOLUTION, 1, 0,
                                        local_rank, host_out.data_ptr(), ctypes.byref(lo),
                                        ctypes.byref(hi))
            _capi.check(code)

        for _ in range(2):
            host_step()
        begin = time.perf_counter()
        e2e_steps = max(2, min(args.steps, 5))
        for _ in range(e2e_steps):
            host_step()
        e2e_seconds = (time.perf_counter() - begin) / e2e_steps
        e2e = {"value": voxels / e2e_seconds / 1e9, "unit": "Gvoxels/s",
               "h2d_bytes_per_step": int(4 * voxels), "d2h_bytes_per_step": int(4 * voxels + 8),
               "ms_per_step": e2e_seconds * 1e3,
               "api": "vgt_b200_sdf_f32 (host pointers, pinned)"}
        # the same call with PAGEABLE buffers (what std::vector / numpy callers hand over): the
        # library stages them through pinned slots with several host threads
        pageable_in = host_in.numpy().copy()
        pageable_out = np.empty_like(pageable_in)

        def pageable_step():
            code = lib.vgt_b200_sdf_f32(pageable_in.ctypes.data, *local_shape, RESOLUTION, 1, 0,
                                        local_rank, pageable_out.ctypes.data, ctypes.byref(lo),
                                        ctypes.byref(hi))
            _capi.check(code)

        for _ in range(2):
            pageable_step()
        begin = time.perf_counter()
        for _ in range(e2e_steps):
            pageable_step()
        pageable_seconds = (time.perf_counter() - begin) / e2e_steps
        e2e["pageable_buffers"] = {"value": voxels / pageable_seconds / 1e9,
                                   "unit": "Gvoxels/s", "ms_per_step": pageable_seconds * 1e3,
                                   "equals_pinned_result": bool(
                                       np.array_equal(pageable_out, host_out.numpy()))}
        e2e["cpp_adapter"] = time_cpp_adapter(dims[0])
    else:
        # Per-rank host slabs in, y-slabs out, through the sharded public API; pinned buffers on
        # both sides (as at N=1), reused across steps.
        device_in = torch.empty_like(occupancy)
        host_sdf = torch.empty(plan.y_slab_shape(), dtype=torch.float32).pin_memory()

        def host_step():
            device_in.copy_(host_in, non_blocking=True)
            sdf, mm = plan.extract(device_in, RESOLUTION)
            host_sdf.copy_(sdf, non_blocking=True)
            mm.tolist()
            torch.cuda.synchronize(dev)
            return host_sdf

        for _ in range(2):
            host_step()
        barrier()
        begin = time.perf_counter()
        e2e_steps = max(2, min(args.steps, 5))
        for _ in range(e2e_steps):
            host_step()
        barrier()
        e2e_seconds = (time.perf_counter() - begin) / e2e_steps
        t = torch.tensor([e2e_seconds], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_seconds = float(t.item())
        e2e = {"value": voxels / e2e_seconds / 1e9, "unit": "Gvoxels/s",
               "h2d_bytes_per_step": int(4 * voxels), "d2h_bytes_per_step": int(4 * voxels + 8),
               "ms_per_step": e2e_seconds * 1e3,
               "api": "ShardedSignedDistanceField.extract (host slabs in/out per rank)"}

    # ---- voxelizer (config 3) on rank 0 at N=1: Mrays/s beside the main metric ----
    voxelizer = None
    if not distributed and not args.skip_voxelizer:
        voxelizer = bench_voxelizer(dev, peak, include_cpu=not args.skip_cpu)

    # ---- BASELINE configs 1 and 3 (parity-test cases): device-resident SDF time beside the line
    other_configs = None
    if not distributed:
        other_configs = {}
        box = torch.from_numpy(synthetic.box_scene(128)).to(dev)
        box_out = torch.empty_like(box)
        for _ in range(3):
            vdev.signed_distance_field(box, RESOLUTION, out=box_out)
        torch.cuda.synchronize(dev)
        box_ms = [sum(vdev.signed_distance_field_profile(box, RESOLUTION, box_out))
                  for _ in range(10)]
        other_configs["config1_128^3_box_scene_sdf_ms"] = statistics.median(box_ms)
        other_configs["config1_note"] = ("8 MiB per buffer: L2-resident, so a time, not a "
                                         "roofline fraction (SURVEY.md section 8d)")

    # ---- SURVEY 8f rank 1: per-object SDF batch of a tagged map through the host entry ----
    other_map_types = None
    if not distributed:
        other_map_types = bench_tagged_map(local_rank, include_cpu=not args.skip_cpu)

    # ---- SURVEY 8f rank 4: the mesh rasterizer (an occupancy producer in front of the path) ----
    mesh = None
    if not distributed and not args.skip_voxelizer:
        mesh = bench_mesh_rasterizer(dev, include_cpu=not args.skip_cpu)

    config5 = None
    if distributed and n_gpus == 8 and not args.skip_config5:
        occupancy = None  # (drops the bench grid)
        torch.cuda.empty_cache()
        try:
            config5 = config5_2048(sharded, vdev, synthetic, dev, rank, n_gpus, 5)
        except Exception as error:  # the main line must survive a failure here
            config5 = {"error": repr(error)[:300]}

    cpu_baseline = None
    if rank == 0 and not distributed and not args.skip_cpu:
        full = cpu_reference_arm(2, 1, dims)
        cpu_baseline = {k: full[k] for k in ("value", "unit", "cores", "kind", "sample")}

    if rank == 0:
        line = {
            "metric": "sdf_gvoxels_per_s", "value": value, "unit": "Gvoxels/s", "n_gpus": n_gpus,
            "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32",
            "data": "synthetic",
            "config": {"workload": f"{'x'.join(map(str, dims))} occupancy -> SDF<float> "
                                   "(clustered spheres ~10% filled, 1% unknown), "
                                   + ("x-slab sharded, exchange fused into the y pass as NVLink "
                                      "peer stores" if distributed and plan.exchange_used ==
                                      "peer_store" else "x-slab sharded, NCCL all-to-all"
                                      if distributed else "one GPU"),
                       "voxels": int(voxels), "resolution": RESOLUTION,
                       "l2_policy": "inputs larger than L2 (>= 512 MiB per pass), no flush",
                       "sdf_min_max": sdf_min_max},
            "clocks": sampler.summary(), "e2e": e2e,
            "gpu_launches": int(launches), "roofline": roofline,
            "cpu_baseline": cpu_baseline,
        }
        if parity is not None:
            line["parity"] = parity
        if strong is not None:
            line["strong_scaling_1024"] = strong
        if config5 is not None:
            line["config5_2048"] = config5
        if voxelizer is not None:
            line["voxelizer"] = voxelizer
        if other_configs is not None:
            line["other_configs"] = other_configs
        if other_map_types is not None:
            line["other_map_types"] = other_map_types
        if mesh is not None:
            line["mesh_rasterizer"] = mesh
        print(json.dumps(line), flush=True)
    if distributed:
        dist.destroy_process_group()


def _icosphere(subdivisions, radius, centre):
    """A subdivided icosahedron: (vertices float64 [n, 3], triangles int32 [20 * 4^s, 3])."""
    import numpy as np
    t = (1.0 + 5.0 ** 0.5) / 2.0
    vertices = [np.array(v, dtype=np.float64) / np.linalg.norm(v) for v in (
        (-1, t, 0), (1, t, 0), (-1, -t, 0), (1, -t, 0), (0, -1, t), (0, 1, t),
        (0, -1, -t), (0, 1, -t), (t, 0, -1), (t, 0, 1), (-t, 0, -1), (-t, 0, 1))]
    faces = [(0, 11, 5), (0, 5, 1), (0, 1, 7), (0, 7, 10), (0, 10, 11), (1, 5, 9), (5, 11, 4),
             (11, 10, 2), (10, 7, 6), (7, 1, 8), (3, 9, 4), (3, 4, 2), (3, 2, 6), (3, 6, 8),
             (3, 8, 9), (4, 9, 5), (2, 4, 11), (6, 2, 10), (8, 6, 7), (9, 8, 1)]
    for _ in range(subdivisions):
        cache, refined = {}, []

        def midpoint(a, b):
            key = (min(a, b), max(a, b))
            if key not in cache:
                m = vertices[a] + vertices[b]
                vertices.append(m / np.linalg.norm(m))
                cache[key] = len(vertices) - 1
            return cache[key]

        for a, b, c in faces:
            ab, bc, ca = midpoint(a, b), midpoint(b, c), midpoint(c, a)
            refined += [(a, ab, ca), (b, bc, ab), (c, ca, bc), (ab, bc, ca)]
        faces = refined
    return (np.array(vertices) * radius + np.array(centre, dtype=np.float64),
            np.array(faces, dtype=np.int32))


def bench_mesh_rasterizer(dev, include_cpu=True):
    """mesh_rasterizer::RasterizeMesh (mesh_rasterizer.cpp:205-230): a sphere of 81920 triangles
    into a device-resident 512^3 map (vgt_b200_rasterize_mesh_dev, CUDA events), the host entry
    on a 256^3 map, and the reference's CPU rasterizer on the same mesh beside them."""
    import ctypes as ct
    import numpy as np
    import torch
    from voxelized_geometry_tools_b200 import _capi
    lib = _capi.library()
    n, resolution = 512, 0.01
    vertices, triangles = _icosphere(6, 2.2, (2.56, 2.56, 2.56))
    d_vertices = torch.from_numpy(vertices).to(dev)
    d_triangles = torch.from_numpy(triangles).to(dev)
    occupancy = torch.zeros((n, n, n), dtype=torch.float32, device=dev)
    flags = torch.zeros(1, dtype=torch.int32, device=dev)
    identity = np.ascontiguousarray(np.eye(4).T).reshape(16)
    pointer = identity.ctypes.data_as(ct.POINTER(ct.c_double))
    stream = torch.cuda.current_stream(dev)
    times = []
    for _ in range(6):
        begin, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        begin.record(stream)
        _capi.check(lib.vgt_b200_rasterize_mesh_dev(
            d_vertices.data_ptr(), len(vertices), d_triangles.data_ptr(), len(triangles),
            occupancy.data_ptr(), 4, n, n, n, resolution, pointer, pointer, 1,
            dev.index or 0, flags.data_ptr(), stream.cuda_stream))
        end.record(stream)
        end.synchronize()
        times.append(begin.elapsed_time(end))
    _capi.check(lib.vgt_b200_rasterize_status(int(flags.item())))
    kernel_ms = statistics.median(times[1:])
    result = {"mesh": f"icosphere, {len(triangles)} triangles, {len(vertices)} vertices",
              "grid": f"{n}^3 @ {resolution} m (device-resident)",
              "kernel_ms": kernel_ms,
              "mtriangles_per_s": len(triangles) / (kernel_ms * 1e-3) / 1e6,
              "cells_filled": int((occupancy == 1.0).sum().item())}
    # host entry (pageable numpy map in and out) on a 256^3 map
    small = 256
    host_map = np.zeros((small, small, small), dtype=np.float32)
    half_vertices = vertices * 0.5
    calls = []
    for _ in range(3):
        begin = time.perf_counter()
        _capi.check(lib.vgt_b200_rasterize_mesh_f64(
            half_vertices.ctypes.data, len(vertices), triangles.ctypes.data, len(triangles),
            host_map.ctypes.data, 4, small, small, small, resolution, pointer, pointer, 1,
            dev.index or 0))
        calls.append(time.perf_counter() - begin)
    result["host_entry"] = {"api": "vgt_b200_rasterize_mesh_f64 (256^3 pageable map in and out)",
                            "ms_per_call": statistics.median(calls) * 1e3}
    if include_cpu:
        from oracle import oracle, reference_oracle
        cpu_map = np.zeros((small, small, small), dtype=np.float32)
        begin = time.perf_counter()
        if reference_oracle.available():
            reference_oracle.rasterize_mesh(half_vertices, triangles, cpu_map, resolution, None,
                                            False, threads=host_threads())
            kind, cores = "reference", host_threads()
        else:
            oracle.rasterize_mesh(half_vertices, triangles, cpu_map, resolution, None, True)
            kind, cores = "port", 1
        result["cpu"] = {"ms": (time.perf_counter() - begin) * 1e3, "kind": kind, "cores": cores,
                         "grid": f"{small}^3", "equals_device_result": bool(
                             np.array_equal(cpu_map, host_map))}
    return result


def bench_tagged_map(device_index, include_cpu=True):
    """TaggedObjectOccupancyMap::MakeSeparateObjectSDFs over a 256^3 map with 8 named objects
    (tagged_object_occupancy_map.hpp:249-262) and ExtractFreeAndNamedObjectsSignedDistanceField,
    host buffers in and out (vgt_b200_sdf_per_object_f32 / vgt_b200_sdf_free_and_named_f32)."""
    import numpy as np
    import voxelized_geometry_tools_b200 as vgt
    from voxelized_geometry_tools_b200 import grids, synthetic
    n, objects = 256, 8
    occupancy = synthetic.clustered_spheres_occupancy((n, n, n))
    cells = np.zeros((n, n, n), dtype=grids.TAGGED_OBJECT_OCCUPANCY_CELL)
    cells["occupancy"] = occupancy
    block = np.add.outer(np.add.outer(np.arange(n) // 64, np.arange(n) // 64 * 2),
                         np.arange(n) // 128)
    cells["object_id"] = (block % objects + 1).astype(np.uint32)
    sizes = vgt.VoxelGridSizes.FromVoxelCounts(RESOLUTION, (n, n, n))
    tagged = vgt.TaggedObjectOccupancyMap(np.eye(4), "world", sizes, cells)
    parameters = vgt.SignedDistanceFieldGenerationParameters()
    ids = list(range(1, objects + 1))
    tagged.MakeSeparateObjectSDFs(ids[:2], parameters, device=device_index)
    begin = time.perf_counter()
    tagged.MakeSeparateObjectSDFs(ids, parameters, device=device_index)
    batch_seconds = time.perf_counter() - begin
    begin = time.perf_counter()
    tagged.ExtractFreeAndNamedObjectsSignedDistanceField(parameters, device=device_index)
    merged_seconds = time.perf_counter() - begin
    voxels = float(n) ** 3
    # the C-ABI call alone, caller-owned output reused across calls (what a C++ caller that keeps
    # its SDF storage pays; the Python mirror above allocates 8 fresh grids per call)
    import ctypes as ct
    from voxelized_geometry_tools_b200 import _capi
    lib = _capi.library()
    out = np.zeros((objects, n, n, n), dtype=np.float32)
    lows, highs = (ct.c_float * objects)(), (ct.c_float * objects)()
    id_array = (ct.c_uint32 * objects)(*ids)
    call_times = []
    for iteration in range(4):
        begin = time.perf_counter()
        _capi.check(lib.vgt_b200_sdf_per_object_f32(
            cells.ctypes.data, cells.dtype.itemsize, n, n, n, RESOLUTION, 1, 0, id_array, objects,
            device_index, out.ctypes.data, lows, highs))
        if iteration >= 1:
            call_times.append(time.perf_counter() - begin)
    c_abi_seconds = statistics.mean(call_times)
    result = {"grid": f"{n}^3 TaggedObjectOccupancyMap, {objects} objects",
              "c_abi_call_only": {"api": "vgt_b200_sdf_per_object_f32 (pageable buffers, reused)",
                                  "ms_per_call": c_abi_seconds * 1e3,
                                  "ms_per_object": c_abi_seconds * 1e3 / objects},
              "per_object_batch_ms": batch_seconds * 1e3,
              "per_object_batch_gvoxels_per_s": objects * voxels / batch_seconds / 1e9,
              "free_and_named_ms": merged_seconds * 1e3,
              "api": "MakeSeparateObjectSDFs / ExtractFreeAndNamedObjectsSignedDistanceField "
                     "(host buffers, pageable numpy arrays)"}
    if include_cpu:
        from oracle import oracle
        begin = time.perf_counter()
        oracle.sdf_from_cells(cells, RESOLUTION, objects_to_use=[1], threads=0)
        result["cpu_one_object_ms"] = (time.perf_counter() - begin) * 1e3
        result["cpu_cores"] = oracle.max_threads()
    return result


def bench_voxelizer(dev, peak, include_cpu=True):
    """BASELINE config 3: 4 cameras x 640x480 rays into 256^3, filter (0.9, 2, 2)."""
    import numpy as np
    import torch
    from voxelized_geometry_tools_b200 import device as vdev, synthetic
    from voxelized_geometry_tools_b200.grids import compose_rigid
    from voxelized_geometry_tools_b200.pointcloud_voxelization import (
        PointCloudVoxelizationFilterOptions)
    scene = synthetic.depth_camera_scene()
    n = scene["static_occupancy"].shape[0]
    x_gw = np.eye(4)
    x_gw[:3, 3] = -scene["origin_transform"][:3, 3]
    clouds = [(torch.from_numpy(points).to(dev), compose_rigid(x_gw, x_wc), max_range)
              for points, x_wc, max_range in scene["clouds"]]
    finite_rays = int(sum(np.isfinite(points).all(axis=1).sum() for points, _, _ in scene["clouds"]))
    counts = torch.zeros((len(clouds), n, n, n, 2), dtype=torch.int32, device=dev)
    static = torch.from_numpy(scene["static_occupancy"]).to(dev)
    occupancy = static.clone()
    options = PointCloudVoxelizationFilterOptions(0.9, 2, 2)
    events = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    raycast_ms, filter_ms, zero_ms = [], [], []
    increments = 0
    for iteration in range(6):
        occupancy.copy_(static)
        events[0].record()
        counts.zero_()
        events[1].record()
        for index, (points, x_gc, max_range) in enumerate(clouds):
            vdev.raycast_cloud(points, x_gc, max_range, counts[index], scene["voxel_size"])
        events[2].record()
        vdev.filter_grids(counts, occupancy, options)
        events[3].record()
        torch.cuda.synchronize(dev)
        if iteration >= 2:
            zero_ms.append(events[0].elapsed_time(events[1]))
            raycast_ms.append(events[1].elapsed_time(events[2]))
            filter_ms.append(events[2].elapsed_time(events[3]))
        increments = int(counts.sum(dtype=torch.int64).item())
    raycast = statistics.mean(raycast_ms)
    filt = statistics.mean(filter_ms)
    # "... then SDF" (config 3): the SDF of the voxelized map, device-resident
    sdf_out = torch.empty_like(occupancy)
    for _ in range(2):
        vdev.signed_distance_field(occupancy, scene["voxel_size"], out=sdf_out)
    torch.cuda.synchronize(dev)
    sdf_after_ms = statistics.median(
        sum(vdev.signed_distance_field_profile(occupancy, scene["voxel_size"], sdf_out))
        for _ in range(7))
    voxels = n ** 3
    filter_bytes = (8 * len(clouds) + 8) * voxels

    # end to end through the host entry point (host points + maps in, host map out)
    import voxelized_geometry_tools_b200 as vgt
    sizes = vgt.VoxelGridSizes.FromVoxelCounts(scene["voxel_size"], (n, n, n))
    static_map = vgt.OccupancyMap(scene["origin_transform"], "world", sizes,
                                  data=scene["static_occupancy"])
    wrappers = [vgt.VectorPointCloudWrapper(p, x, r) for p, x, r in scene["clouds"]]
    voxelizer = vgt.B200PointCloudVoxelizer({"CUDA_DEVICE": dev.index or 0})
    host_times = []
    for iteration in range(4):
        begin = time.perf_counter()
        voxelizer.VoxelizePointClouds(static_map, options, wrappers)
        if iteration >= 1:
            host_times.append(time.perf_counter() - begin)
    host_seconds = statistics.mean(host_times)
    # the C-ABI call alone (caller-owned pageable buffers reused across calls), double and
    # float32 clouds: what a C++ caller that keeps its output map pays
    import ctypes as ct
    from voxelized_geometry_tools_b200 import _capi
    lib = _capi.library()
    out_map = np.empty_like(scene["static_occupancy"])
    option_struct = options.as_struct()
    c_abi = {}
    for label, cloud_type, scalar, c_scalar, entry in (
            ("f64", _capi.Cloud, np.float64, ct.c_double, lib.vgt_b200_voxelize_f64),
            ("f32", _capi.CloudF32, np.float32, ct.c_float, lib.vgt_b200_voxelize_f32)):
        array = (cloud_type * len(scene["clouds"]))()
        keep = []
        for index, (points, x_wc, max_range) in enumerate(scene["clouds"]):
            held = np.ascontiguousarray(points, dtype=scalar)
            keep.append(held)
            array[index].points_xyz = held.ctypes.data_as(ct.POINTER(c_scalar))
            array[index].num_points = held.shape[0]
            array[index].x_gc = (ct.c_double * 16)(*compose_rigid(x_gw, x_wc).T.reshape(-1))
            array[index].max_range = float(max_range)
        seconds = (ct.c_double * 2)()
        times = []
        for iteration in range(5):
            begin = time.perf_counter()
            _capi.check(entry(scene["static_occupancy"].ctypes.data, n, n, n, scene["voxel_size"],
                              array, len(scene["clouds"]), ct.byref(option_struct),
                              dev.index or 0, out_map.ctypes.data, None, seconds))
            if iteration >= 1:
                times.append(time.perf_counter() - begin)
        c_abi[label] = {"ms_per_call": statistics.mean(times) * 1e3,
                        "mrays_per_s": finite_rays / statistics.mean(times) / 1e6,
                        "raycast_ms_reported": seconds[0] * 1e3,
                        "filter_ms_reported": seconds[1] * 1e3}

    cpu = None
    if include_cpu:
        from oracle import oracle
        prepared = [(p, compose_rigid(x_gw, x), r) for p, x, r in scene["clouds"]]
        kind, run_cpu = "port", oracle.voxelize
        try:
            from oracle import reference_oracle
            if reference_oracle.voxelizer_available():
                # the reference's own cpu_pointcloud_voxelization.cpp (oracle/_ref)
                kind, run_cpu = "reference", reference_oracle.voxelize
        except Exception:
            pass
        threads = host_threads()
        run_cpu(scene["static_occupancy"], prepared, scene["voxel_size"], 0.9, 2, 2,
                threads=threads)
        begin = time.perf_counter()
        run_cpu(scene["static_occupancy"], prepared, scene["voxel_size"], 0.9, 2, 2,
                threads=threads)
        cpu_seconds = time.perf_counter() - begin
        cpu = {"value": finite_rays / cpu_seconds / 1e6, "unit": "Mrays/s",
               "cores": threads, "kind": kind,
               "sample": f"the whole config-3 workload once ({cpu_seconds:.2f} s), raycast + "
                         "filter + the counter read-back of the test entry"}
    return {"metric": "voxelization_mrays_per_s", "value": finite_rays / (raycast * 1e-3) / 1e6,
            "unit": "Mrays/s", "rays": finite_rays, "grid": f"{n}^3", "cameras": len(clouds),
            "raycast_ms": raycast, "filter_ms": filt, "zero_ms": statistics.mean(zero_ms),
            "sdf_of_voxelized_map_ms": sdf_after_ms,
            "atomic_increments": increments,
            "counter_increments_per_s_G": increments / (raycast * 1e-3) / 1e9,
            "e2e": {"value": finite_rays / host_seconds / 1e6, "unit": "Mrays/s",
                    "ms_per_call": host_seconds * 1e3,
                    "api": "B200PointCloudVoxelizer.VoxelizePointClouds (vgt_b200_voxelize_f64, "
                           "host buffers, raycast + filter + the copy of the static map the "
                           "interface makes, pcv_if.hpp:252)",
                    "c_abi_call_only": c_abi},
            "cpu_baseline": cpu,
            "filter_roofline": {"bound": "hbm", "achieved": filter_bytes / (filt * 1e-3) / 1e9,
                                "peak": peak, "unit": "GB/s",
                                "frac": filter_bytes / (filt * 1e-3) / 1e9 / peak}}


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument("--gpus", type=int, default=1)
    parser.add_argument("--steps", type=int, default=10)
    parser.add_argument("--warmup", type=int, default=3)
    parser.add_argument("--impl", default="ours", choices=["ours", "reference"])
    parser.add_argument("--skip-cpu", action="store_true", help="skip the cpu_baseline leg")
    parser.add_argument("--skip-voxelizer", action="store_true")
    parser.add_argument("--skip-parity", action="store_true",
                        help="N > 1: skip the sharded == single-GPU / oracle checks")
    parser.add_argument("--skip-config5", action="store_true",
                        help="N = 8 only: skip the 2048^3 grid of BASELINE config 5")
    parser.add_argument("--skip-strong", action="store_true",
                        help="skip the 1024^3 strong-scaling leg (BASELINE config 4)")
    parser.add_argument("--exchange", default="auto", choices=["auto", "peer_store", "peer_copy", "nccl"])
    parser.add_argument("--chunks", type=int, default=2,
                        help="x-chunks per slab for overlapping the all-to-all (N > 1)")
    parser.add_argument("--dump-outputs", metavar="DIR",
                        help="write the SDF of the last timed step (a fixed sample) and its "
                             "min/max to DIR/*.npy")
    args = parser.parse_args()
    if args.steps < 1:
        parser.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        parser.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
