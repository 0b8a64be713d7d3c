"""Slab-sharded signed distance field across the GPUs of one box (one process per GPU).

Scheme (SURVEY.md section 8e): the grid is cut into x-slabs -- x is the slowest storage axis, so a
slab is one contiguous range of the reference's host vector. The z and y passes are independent
per x and run slab-local. One all-to-all then re-cuts the sign-fused int32 intermediate into
y-slabs laid out [nx, ny_local, nz], on which the x pass + finalize run, again with z contiguous.
min/max is reduced with one 2-float all-reduce. The result stays y-sharded on the devices;
``gather_to_host`` writes the slabs back to their x-major host positions (tests, small grids).

The reference has no multi-device path at all (SURVEY.md section 2.2); this is the B200-native
analogue of its OpenMP split over lines (sdfgen.cpp:286-389).

The compute stages are injectable so the exchange logic can be tested on CPU with the gloo
backend (tests/test_sharded_gloo.py); the product stages are the CUDA ones in ``device.py``.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Callable

import torch
import torch.distributed as dist


def split_range(total: int, parts: int, index: int) -> tuple[int, int]:
    """[begin, end) of part ``index`` when ``total`` items are cut into ``parts`` near-equal parts
    (the first ``total % parts`` parts get one extra item)."""
    base, extra = divmod(total, parts)
    begin = index * base + min(index, extra)
    return begin, begin + base + (1 if index < extra else 0)


@dataclass
class Stages:
    """local_passes(occupancy_slab[nxl, ny, nz] f32, unknown_is_filled) -> int32 [nxl, ny, nz]
    final_pass(packed[nx, nyl, nz] int32, y_offset, ny_total, resolution, add_virtual_border)
        -> (sdf f32 [nx, nyl, nz], min_max f32 [2])
    local_passes_send (optional): (occupancy_slab, unknown_is_filled, parts) -> flat int32 in send
        layout (parts blocks [nxl, rows_h, nz] back to back); may raise NotImplementedError."""
    local_passes: Callable
    final_pass: Callable
    local_passes_send: Callable | None = None
    # (occupancy_slab, rank, x_offset, nx_total, peer_buffer_ptrs, capacity_words,
    # unknown_is_filled) -> None: passes with the exchange fused in (peer stores); CUDA only.
    local_passes_scatter: Callable | None = None


def cuda_stages() -> Stages:
    from . import device

    def local_passes(occupancy_slab, unknown_is_filled):
        return device.edt_local_passes(occupancy_slab, unknown_is_filled)

    def local_passes_send(occupancy_slab, unknown_is_filled, parts):
        return device.edt_local_passes(occupancy_slab, unknown_is_filled,
                                       send_parts=parts).view(-1)

    def final_pass(packed, y_offset, ny_total, resolution, add_virtual_border):
        return device.edt_final_pass(packed, y_offset, ny_total, resolution, add_virtual_border)

    def local_passes_scatter(occupancy_slab, rank, x_offset, nx_total, peer_buffer_ptrs,
                             capacity_words, unknown_is_filled):
        device.edt_local_passes_scatter(occupancy_slab, rank, x_offset, nx_total,
                                        peer_buffer_ptrs, capacity_words, unknown_is_filled)

    return Stages(local_passes, final_pass, local_passes_send, local_passes_scatter)


class ShardedSignedDistanceField:
    def __init__(self, dims, rank: int | None = None, world_size: int | None = None,
                 group=None, stages: Stages | None = None, chunks: int = 1,
                 profile: bool = False, exchange: str = "auto"):
        """chunks > 1 cuts the x-slab into that many x-chunks: the slab-local passes of chunk c+1
        overlap the all-to-all of chunk c (NCCL runs on its own stream). profile=True records CUDA
        events around the stages (``last_stage_ms`` after a synchronise)."""
        # exchange: "peer_store" = the y pass stores straight into the peers' receive buffers over
        # NVLink (symmetric memory, no collective call); "peer_copy" = the y pass of x-chunk c
        # writes the send layout locally and the copy engines move its parts into the peers'
        # receive buffers while the passes of chunk c + 1 run (`chunks` chunks); "nccl" =
        # all-to-all; "auto" = peer_store when the stages and the device support it, else nccl.
        self.dims = tuple(int(d) for d in dims)
        self.group = group
        self.exchange = exchange
        self.exchange_used = None
        self._peer = None
        self._step = 0
        self.chunks = max(1, int(chunks))
        self.profile = profile
        self.last_stage_ms = None
        self._events = None
        self.rank = dist.get_rank(group) if rank is None else rank
        self.world_size = dist.get_world_size(group) if world_size is None else world_size
        nx, ny, _ = self.dims
        if self.world_size > min(nx, ny):
            raise ValueError("more ranks than voxels along x or y")
        self.stages = stages if stages is not None else cuda_stages()
        self.x_range = split_range(nx, self.world_size, self.rank)
        self.y_range = split_range(ny, self.world_size, self.rank)

    # ------------------------------------------------------------------ layout helpers
    def x_slab_shape(self):
        return (self.x_range[1] - self.x_range[0], self.dims[1], self.dims[2])

    def y_slab_shape(self):
        return (self.dims[0], self.y_range[1] - self.y_range[0], self.dims[2])

    def pack_send_layout(self, packed: torch.Tensor) -> torch.Tensor:
        """[nxl, ny, nz] -> send layout by a copy (fallback when the kernel cannot write it)."""
        ny = self.dims[1]
        chunks = []
        for peer in range(self.world_size):
            y0, y1 = split_range(ny, self.world_size, peer)
            chunks.append(packed[:, y0:y1, :].reshape(-1))
        return torch.cat(chunks)

    def _exchange(self, send: torch.Tensor) -> torch.Tensor:
        """All-to-all transpose: send layout of an x-slab -> y-slab [nx, nyl, nz].

        The block received from rank g is rows x in [x0_g, x1_g) of the y-slab, which is one
        contiguous range of the destination, so the collective writes straight into place."""
        nx, ny, nz = self.dims
        world = self.world_size
        nyl = self.y_range[1] - self.y_range[0]
        nxl = self.x_range[1] - self.x_range[0]
        send_splits = []
        for peer in range(world):
            y0, y1 = split_range(ny, world, peer)
            send_splits.append(nxl * (y1 - y0) * nz)
        recv_splits = []
        for peer in range(world):
            x0, x1 = split_range(nx, world, peer)
            recv_splits.append((x1 - x0) * nyl * nz)
        received = torch.empty(nx * nyl * nz, dtype=send.dtype, device=send.device)
        dist.all_to_all_single(received, send, recv_splits, send_splits, group=self.group)
        return received.view(nx, nyl, nz)

    # ------------------------------------------------------------------ the path
    def extract(self, occupancy_slab: torch.Tensor, resolution: float,
                unknown_is_filled: bool = True, add_virtual_border: bool = False):
        """occupancy_slab: this rank's x-slab [nxl, ny, nz] float32.
        Returns (sdf y-slab [nx, nyl, nz] float32, global (min, max) tensor [2])."""
        if tuple(occupancy_slab.shape) != self.x_slab_shape():
            raise ValueError(f"expected an x-slab of shape {self.x_slab_shape()}")
        self._mark("start", occupancy_slab)
        if (self.world_size > 1 and self.exchange in ("auto", "peer_store", "peer_copy")
                and self.stages.local_passes_scatter is not None and occupancy_slab.is_cuda
                and self._peer is None):
            self._setup_peer_store(occupancy_slab.device)
        if self.world_size > 1 and self._peer and self.exchange == "peer_copy":
            y_slab = self._peer_copy_local_and_exchange(occupancy_slab, unknown_is_filled)
            self.exchange_used = "peer_copy"
        elif self.world_size > 1 and self._peer:
            y_slab = self._peer_store_local_and_exchange(occupancy_slab, unknown_is_filled)
            self.exchange_used = "peer_store"
        elif self.world_size == 1:
            y_slab = self.stages.local_passes(occupancy_slab, unknown_is_filled)
            self._mark("local", occupancy_slab)
        elif self.chunks > 1 and self.stages.local_passes_send is not None:
            y_slab = self._chunked_local_and_exchange(occupancy_slab, unknown_is_filled)
            self.exchange_used = "nccl"
        else:
            send = None
            if self.stages.local_passes_send is not None:
                try:
                    send = self.stages.local_passes_send(occupancy_slab, unknown_is_filled,
                                                         self.world_size)
                except NotImplementedError:
                    send = None
            if send is None:
                send = self.pack_send_layout(
                    self.stages.local_passes(occupancy_slab, unknown_is_filled))
            self._mark("local", occupancy_slab)
            y_slab = self._exchange(send)
            self.exchange_used = "nccl"
        self._mark("exchange", occupancy_slab)
        sdf, min_max = self.stages.final_pass(
            y_slab, self.y_range[0], self.dims[1], resolution, add_virtual_border)
        self._mark("final", occupancy_slab)
        if self.world_size > 1:
            # one tiny all-reduce: max over (-min, max)
            folded = torch.stack([-min_max[0], min_max[1]])
            dist.all_reduce(folded, op=dist.ReduceOp.MAX, group=self.group)
            min_max = torch.stack([-folded[0], folded[1]])
        return sdf, min_max

    # ------------------------------------------------------------------ fused peer-store exchange
    def _setup_peer_store(self, device) -> None:
        """Two symmetric receive buffers (double-buffered across steps), mapped into every rank."""
        try:
            import torch.distributed._symmetric_memory as symm_mem
            nx, ny, nz = self.dims
            max_nyl = -(-ny // self.world_size)
            group = self.group if self.group is not None else dist.group.WORLD
            buffers, handles = [], []
            for _ in range(2):
                buffer = symm_mem.empty(nx * max_nyl * nz, dtype=torch.int32, device=device)
                handles.append(symm_mem.rendezvous(buffer, group))
                buffers.append(buffer)
            self._peer = {"buffers": buffers, "handles": handles}
        except Exception as error:  # no symmetric memory on this system: use NCCL
            if self.exchange in ("peer_store", "peer_copy"):
                raise
            self._peer = False
            self._peer_error = repr(error)

    def _peer_store_local_and_exchange(self, occupancy_slab, unknown_is_filled):
        nx, _, nz = self.dims
        nyl = self.y_range[1] - self.y_range[0]
        index = self._step % 2
        self._step += 1
        buffer, handle = self._peer["buffers"][index], self._peer["handles"][index]
        # The y pass of every rank writes its part of our y-slab into `buffer`. Double buffering
        # plus the barrier below keeps a rank from overwriting a buffer its owner still reads.
        self.stages.local_passes_scatter(occupancy_slab, self.rank, self.x_range[0], nx,
                                         [int(p) for p in handle.buffer_ptrs], buffer.numel(),
                                         unknown_is_filled)
        self._mark("local", occupancy_slab)
        handle.barrier(channel=0)
        return buffer[:nx * nyl * nz].view(nx, nyl, nz)

    # ------------------------------------------------------------------ peer copies (DMA)
    def _peer_copy_local_and_exchange(self, occupancy_slab, unknown_is_filled):
        """x-chunks of the slab: the z / y passes of chunk c write the send layout into local
        memory; its world parts then travel to their owners' receive buffers (symmetric memory,
        mapped into this process) as plain device-to-device copies on side streams - the copy
        engines, not the SMs, drive NVLink - while the passes of chunk c + 1 run. The block a
        chunk contributes to a peer's y-slab is rows x in [x0 + c0, x0 + c1): contiguous there.
        One symmetric-memory barrier, ordered after this rank's copies, separates the exchange
        from the x pass; receive buffers are double-buffered across steps."""
        nx, ny, nz = self.dims
        world = self.world_size
        nyl = self.y_range[1] - self.y_range[0]
        nxl = self.x_range[1] - self.x_range[0]
        x0 = self.x_range[0]
        index = self._step % 2
        self._step += 1
        buffer, handle = self._peer["buffers"][index], self._peer["handles"][index]
        device = occupancy_slab.device
        if "copy_streams" not in self._peer:
            self._peer["copy_streams"] = [torch.cuda.Stream(device=device) for _ in range(2)]
        copy_streams = self._peer["copy_streams"]
        compute = torch.cuda.current_stream(device)
        chunks = max(1, min(self.chunks, nxl))
        keep = []
        for c in range(chunks):
            c0, c1 = split_range(nxl, chunks, c)
            if c1 <= c0:
                continue
            send = self.stages.local_passes_send(occupancy_slab[c0:c1], unknown_is_filled, world)
            keep.append(send)
            ready = torch.cuda.Event()
            ready.record(compute)
            offsets, offset = [], 0
            for peer in range(world):
                y0, y1 = split_range(ny, world, peer)
                offsets.append((offset, (c1 - c0) * (y1 - y0) * nz))
                offset += offsets[-1][1]
            # peers in an order rotated by the rank: at any moment every rank copies to a
            # different peer
            for k in range(world):
                peer = (self.rank + 1 + k) % world
                start, count = offsets[peer]
                if count == 0:
                    continue
                py0, py1 = split_range(ny, world, peer)
                target = handle.get_buffer(peer, (count,), torch.int32,
                                           (x0 + c0) * (py1 - py0) * nz)
                stream = copy_streams[k % len(copy_streams)]
                stream.wait_event(ready)
                with torch.cuda.stream(stream):
                    target.copy_(send[start:start + count], non_blocking=True)
        for stream in copy_streams:
            compute.wait_stream(stream)
        self._peer["keep"] = keep  # (alive until the next step: the copies read them)
        self._mark("local", occupancy_slab)
        handle.barrier(channel=0)
        return buffer[:nx * nyl * nz].view(nx, nyl, nz)

    # ------------------------------------------------------------------ chunked overlap
    def _chunked_local_and_exchange(self, occupancy_slab, unknown_is_filled):
        """x-chunks of the slab: passes on chunk c+1 overlap the all-to-all of chunk c. The block
        that rank g's chunk c contributes to our y-slab is rows x in [x0_g + c0, x0_g + c1): a
        contiguous range of the destination, received in place."""
        nx, ny, nz = self.dims
        world = self.world_size
        nyl = self.y_range[1] - self.y_range[0]
        nxl = self.x_range[1] - self.x_range[0]
        received = torch.empty((nx, nyl, nz), dtype=torch.int32, device=occupancy_slab.device)
        # every rank must issue the same number of collectives: chunk the LARGEST slab size
        max_nxl = -(-nx // world)
        chunks = min(self.chunks, max_nxl)
        works, keep = [], []
        for c in range(chunks):
            c0, c1 = split_range(nxl, chunks, c)
            if c1 > c0:
                try:
                    send = self.stages.local_passes_send(
                        occupancy_slab[c0:c1], unknown_is_filled, world)
                except NotImplementedError:
                    send = self.pack_send_layout_rows(
                        self.stages.local_passes(occupancy_slab[c0:c1], unknown_is_filled))
            else:
                send = torch.empty(0, dtype=torch.int32, device=occupancy_slab.device)
            inputs, outputs, offset = [], [], 0
            for peer in range(world):
                y0, y1 = split_range(ny, world, peer)
                count = (c1 - c0) * (y1 - y0) * nz
                inputs.append(send[offset:offset + count])
                offset += count
                px0, px1 = split_range(nx, world, peer)
                pc0, pc1 = split_range(px1 - px0, chunks, c)
                outputs.append(received[px0 + pc0:px0 + pc1].view(-1))
            keep.append(send)
            # grouped point-to-point (works on NCCL and gloo alike); own block = local copy
            outputs[self.rank].copy_(inputs[self.rank])
            ops = []
            for peer in range(world):
                if peer == self.rank:
                    continue
                if inputs[peer].numel() > 0:
                    ops.append(dist.P2POp(dist.isend, inputs[peer], peer, group=self.group))
                if outputs[peer].numel() > 0:
                    ops.append(dist.P2POp(dist.irecv, outputs[peer], peer, group=self.group))
            if ops:
                works.extend(dist.batch_isend_irecv(ops))
        self._mark("local", occupancy_slab)
        for work in works:
            work.wait()
        return received

    def pack_send_layout_rows(self, packed: torch.Tensor) -> torch.Tensor:
        ny = self.dims[1]
        return torch.cat([packed[:, split_range(ny, self.world_size, p)[0]:
                                 split_range(ny, self.world_size, p)[1], :].reshape(-1)
                          for p in range(self.world_size)])

    # ------------------------------------------------------------------ optional stage timing
    def _mark(self, name: str, like: torch.Tensor) -> None:
        if not self.profile or not like.is_cuda:
            return
        if name == "start":
            self._events = []
        event = torch.cuda.Event(enable_timing=True)
        event.record()
        self._events.append((name, event))

    def stage_ms(self):
        """After a synchronise: {stage: ms} of the last profiled extract()."""
        if not self._events:
            return None
        return {name: self._events[i - 1][1].elapsed_time(event)
                for i, (name, event) in enumerate(self._events) if i > 0}

    def gather_to_host(self, sdf_y_slab: torch.Tensor) -> torch.Tensor | None:
        """Collects the y-slabs into one [nx, ny, nz] host tensor on rank 0 (small grids only)."""
        nx, ny, nz = self.dims
        local = sdf_y_slab.detach().cpu().contiguous()
        if self.world_size == 1:
            return local
        pieces = [None] * self.world_size if self.rank == 0 else None
        dist.gather_object(local, pieces, dst=0, group=self.group)
        if self.rank != 0:
            return None
        full = torch.empty((nx, ny, nz), dtype=local.dtype)
        for peer, piece in enumerate(pieces):
            y0, y1 = split_range(ny, self.world_size, peer)
            full[:, y0:y1, :] = piece
        return full


# --------------------------------------------------------------------------------------------------
# Sharded voxelizer (SURVEY.md section 8e, row 4): counters are additive over rays
# --------------------------------------------------------------------------------------------------
@dataclass
class VoxelizerStages:
    """raycast(points [n, 3] f64, x_gc 4x4, max_range, counts int32 [nx, ny, nz, 2], voxel_size)
        accumulates one cloud (or part of one) into counts;
    filter(counts int32 [cameras, nxl, ny, nz, 2], occupancy f32 [nxl, ny, nz], options)
        applies the per-camera rule and the combine in place on a slab."""
    raycast: Callable
    filter: Callable


def cuda_voxelizer_stages() -> VoxelizerStages:
    from . import device

    def raycast(points, x_gc, max_range, counts, voxel_size):
        device.raycast_cloud(points, x_gc, max_range, counts, voxel_size)

    def filter_slab(counts, occupancy, options):
        device.filter_grids(counts, occupancy, options)

    return VoxelizerStages(raycast, filter_slab)


class ShardedPointCloudVoxelizer:
    """PointCloudVoxelizationInterface::VoxelizePointClouds across the GPUs of one box.

    The rays of every cloud are split evenly over the ranks (rank r takes points r, r + G, ...);
    each rank raycasts its share into full-size tracking grids; one reduce-scatter (sum, int32)
    per camera adds the shares and leaves rank g with the x-slab the sharded SDF starts from.
    The per-camera rule (pointcloud_voxelization_interface.hpp:55-86) needs a camera's COMPLETE
    counters, so the rays of one camera are summed before it, and cameras are combined after
    it, slab-local (cpu_pointcloud_voxelization.cpp:438-497). The filtered occupancy x-slab feeds
    ShardedSignedDistanceField.extract directly: voxelize -> SDF never leaves the devices.

    The reference voxelizes in one process (cpu_pointcloud_voxelization.cpp:133-165); counts are
    integers, so the sharded result is bit-identical to it whatever the split."""

    def __init__(self, dims, voxel_size: float, rank: int | None = None,
                 world_size: int | None = None, group=None,
                 stages: VoxelizerStages | None = None):
        self.dims = tuple(int(d) for d in dims)
        self.voxel_size = float(voxel_size)
        self.group = group
        self.rank = dist.get_rank(group) if rank is None else rank
        self.world_size = dist.get_world_size(group) if world_size is None else world_size
        if self.world_size > self.dims[0]:
            raise ValueError("more ranks than voxels along x")
        self.stages = stages if stages is not None else cuda_voxelizer_stages()
        self.x_range = split_range(self.dims[0], self.world_size, self.rank)
        self.last_counts = None

    def share_of(self, points: torch.Tensor) -> torch.Tensor:
        """This rank's rays of a cloud that every rank holds in full."""
        return points[self.rank::self.world_size].contiguous()

    def _reduce_scatter_x(self, counts: torch.Tensor) -> torch.Tensor:
        """counts [nx, ny, nz, 2] (this rank's share) -> summed x-slab [nxl, ny, nz, 2]."""
        nx, ny, nz = self.dims
        world = self.world_size
        if world == 1:
            return counts
        x0, x1 = self.x_range
        backend = dist.get_backend(self.group)
        if nx % world == 0 and backend == "nccl":
            out = torch.empty((nx // world, ny, nz, 2), dtype=counts.dtype, device=counts.device)
            dist.reduce_scatter_tensor(out, counts, op=dist.ReduceOp.SUM, group=self.group)
            return out
        if backend == "nccl":
            # uneven slabs: reduce-scatter over a list of per-rank views (NCCL sends each one)
            pieces = [counts[split_range(nx, world, r)[0]:split_range(nx, world, r)[1]]
                      for r in range(world)]
            out = torch.empty_like(pieces[self.rank])
            works = [dist.reduce(piece, dst=r, op=dist.ReduceOp.SUM, group=self.group,
                                 async_op=True) for r, piece in enumerate(pieces)]
            for work in works:
                work.wait()
            out.copy_(pieces[self.rank])
            return out
        # gloo (CPU tests of the host logic): all-reduce, keep the own slab
        total = counts.clone()
        dist.all_reduce(total, op=dist.ReduceOp.SUM, group=self.group)
        return total[x0:x1].contiguous()

    def voxelize(self, static_occupancy_slab: torch.Tensor, clouds, filter_options,
                 points_are_shares: bool = False, keep_counts: bool = False) -> torch.Tensor:
        """static_occupancy_slab: this rank's x-slab [nxl, ny, nz] float32 of the static map.
        clouds: [(points float64 [n, 3] in the cloud frame, X_GC 4x4, max_range), ...] - the same
        list on every rank (points_are_shares=False: each rank takes its share of the rays) or
        already this rank's share. Returns the filtered occupancy x-slab (a new tensor)."""
        nx, ny, nz = self.dims
        x0, x1 = self.x_range
        if tuple(static_occupancy_slab.shape) != (x1 - x0, ny, nz):
            raise ValueError(f"expected an x-slab of shape {(x1 - x0, ny, nz)}")
        device = static_occupancy_slab.device
        slabs = []
        for points, x_gc, max_range in clouds:
            share = points if points_are_shares else self.share_of(points)
            counts = torch.zeros((nx, ny, nz, 2), dtype=torch.int32, device=device)
            self.stages.raycast(share, x_gc, max_range, counts, self.voxel_size)
            slabs.append(self._reduce_scatter_x(counts))
            del counts
        # at least one tracking grid even without clouds (device_pointcloud_voxelization.cpp:79-80)
        if not slabs:
            slabs.append(torch.zeros((x1 - x0, ny, nz, 2), dtype=torch.int32, device=device))
        camera_counts = torch.stack(slabs)
        occupancy = static_occupancy_slab.clone()
        self.stages.filter(camera_counts, occupancy, filter_options)
        self.last_counts = camera_counts if keep_counts else None
        return occupancy


# --------------------------------------------------------------------------------------------------
# Sharded connected components: one x-slab of a component map per rank (DESIGN.md section 8)
# --------------------------------------------------------------------------------------------------
@dataclass
class ComponentStages:
    """The device phases of ShardedConnectedComponents.label on one rank's x-slab:
    local(cells_slab, base, face_roots) -> (state, roots int32 [ny * nz] of the last x-plane, or
        None when not face_roots)
    face_edges(state, below_cells [ny, nz, words], below_roots [ny * nz], below_base)
        -> int64 [E, 2] (global root below, global root above)
    resolve(state, edges int64 [E, 2] of every face, num_cells) -> number of nodes
    count(state) -> count_g
    publish(state, offset) -> node ids int32 [number of nodes]: the slab's own set, zero elsewhere
    write(state, node_ids summed over the ranks) -> None: the slab's component words written."""
    local: Callable
    face_edges: Callable
    resolve: Callable
    count: Callable
    publish: Callable
    write: Callable


def cuda_component_stages() -> ComponentStages:
    from . import device

    def local(cells_slab, base, face_roots):
        state = device.ComponentSlab(cells_slab, base)
        return state, state.local(face_roots)

    return ComponentStages(
        local=local,
        face_edges=lambda state, cells, roots, base: state.face_edges(cells, roots, base),
        resolve=lambda state, edges, num_cells: state.resolve(edges, num_cells),
        count=lambda state: state.count(),
        publish=lambda state, offset: state.publish(offset),
        write=lambda state, node_ids: state.write(node_ids))


class ShardedConnectedComponents:
    """ComputeConnectedComponents (topology_computation.hpp:138-196) on a component map cut into
    x-slabs, one per rank, each on its rank's device: rank r holds the x-planes
    split_range(nx, world_size, r) (the cut of ShardedSignedDistanceField). The result is the
    whole-map labelling, the same bytes as the one-device entry.

    Collectives, in order: the last x-plane of rank r (cells and local roots) sent to rank r + 1;
    all_gather of the edge counts, then of the edges padded to the longest list; all_gather of
    count_g (the offsets and the total); all_reduce SUM of the node ids."""

    def __init__(self, dims, rank: int | None = None, world_size: int | None = None,
                 group=None, stages: ComponentStages | None = None):
        self.dims = tuple(int(d) for d in dims)
        self.group = group
        self.rank = dist.get_rank(group) if rank is None else rank
        self.world_size = dist.get_world_size(group) if world_size is None else world_size
        if self.world_size > self.dims[0]:
            raise ValueError("more ranks than voxels along x")
        self.stages = stages if stages is not None else cuda_component_stages()
        self.x_range = split_range(self.dims[0], self.world_size, self.rank)

    def x_slab_shape(self):
        return (self.x_range[1] - self.x_range[0], self.dims[1], self.dims[2])

    def label(self, cells_slab: torch.Tensor) -> int:
        """cells_slab: this rank's x-slab [nx_r, ny, nz, 2 | 4], a contiguous int32 or uint32
        tensor (2 words per OccupancyComponentCell, 4 per TaggedObjectOccupancyComponentCell).
        Its component words are written in place; returns the number of components of the whole
        map (the same on every rank). A map of more than 0xFFFFFFFF components raises
        NotImplementedError on every rank before any cell is written."""
        if tuple(cells_slab.shape[:3]) != self.x_slab_shape() or cells_slab.dim() != 4:
            raise ValueError(f"expected an x-slab of shape {self.x_slab_shape()} + (words,)")
        nx, ny, nz = self.dims
        plane = ny * nz
        world, rank = self.world_size, self.rank
        base = self.x_range[0] * plane
        stages = self.stages
        state, roots = stages.local(cells_slab, base, rank + 1 < world)
        edges = torch.zeros((0, 2), dtype=torch.int64, device=cells_slab.device)
        if world > 1:
            below_cells, below_roots = self._exchange_face(cells_slab, roots)
            if rank > 0:
                below_base = split_range(nx, world, rank - 1)[0] * plane
                edges = stages.face_edges(state, below_cells, below_roots, below_base)
            edges = self._gather_edges(edges)
        stages.resolve(state, edges, nx * plane)
        count = stages.count(state)
        counts = [count]
        if world > 1:
            gathered = self._all_gather(torch.tensor([count], dtype=torch.int64,
                                                     device=cells_slab.device))
            counts = [int(c) for c in gathered.tolist()]
        total = sum(counts)
        if total > 0xFFFFFFFF:
            raise NotImplementedError(f"connected components: {total} components do not fit the "
                                      "32-bit component word")
        node_ids = stages.publish(state, sum(counts[:rank]))
        if world > 1 and node_ids.numel() > 0:
            dist.all_reduce(node_ids, op=dist.ReduceOp.SUM, group=self.group)
        stages.write(state, node_ids)
        return total

    def _exchange_face(self, cells_slab, roots):
        """Rank r's last x-plane (cells as stored, their local roots) to rank r + 1."""
        ny, nz = self.dims[1], self.dims[2]
        words = cells_slab.shape[3]
        device = cells_slab.device
        below_cells = below_roots = None
        ops = []
        if self.rank + 1 < self.world_size:
            last = cells_slab[-1].contiguous().view(torch.int32)
            ops += [dist.P2POp(dist.isend, last, self.rank + 1, group=self.group),
                    dist.P2POp(dist.isend, roots, self.rank + 1, group=self.group)]
        if self.rank > 0:
            below_cells = torch.empty((ny, nz, words), dtype=torch.int32, device=device)
            below_roots = torch.empty(ny * nz, dtype=torch.int32, device=device)
            ops += [dist.P2POp(dist.irecv, below_cells, self.rank - 1, group=self.group),
                    dist.P2POp(dist.irecv, below_roots, self.rank - 1, group=self.group)]
        for work in dist.batch_isend_irecv(ops):
            work.wait()
        return below_cells, below_roots

    def _all_gather(self, tensor):
        pieces = [torch.empty_like(tensor) for _ in range(self.world_size)]
        dist.all_gather(pieces, tensor, group=self.group)
        return torch.cat(pieces)

    def _gather_edges(self, edges):
        """Every rank's face edges, on every rank: their counts, then the edges padded to the
        longest list."""
        counts = self._all_gather(torch.tensor([edges.shape[0]], dtype=torch.int64,
                                               device=edges.device)).tolist()
        longest = max(counts)
        if longest == 0:
            return edges[:0]
        padded = torch.zeros((longest, 2), dtype=torch.int64, device=edges.device)
        padded[:edges.shape[0]] = edges
        gathered = self._all_gather(padded.unsqueeze(0))
        return torch.cat([gathered[r, :counts[r]] for r in range(self.world_size)]).contiguous()
