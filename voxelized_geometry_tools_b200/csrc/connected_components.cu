// sm_100a connected-component labelling of the component maps and its C-ABI entry points.
//
// Replaces ComputeConnectedComponents (topology_computation.hpp:138-196) as the two component
// maps call it: a serial scan in storage order that flood-fills, breadth first over the 6 face
// neighbours, every cell whose component is still 0, numbering the fills 1, 2, 3, ... So
// component k is the component whose smallest linear index is the k-th smallest of all the
// components' smallest indices: the numbering follows from the partition alone.
//
// Here: union-find over the whole grid with the invariant parent[i] <= i (a root is always hung
// under the smaller of the two roots), so the root of every set is its smallest index and the
// reference's number of a component is the rank of its root plus one.
//   1. InitRunsKernel      parent[i] = start of i's run of equal keys along z inside its tile of
//                          kRunTile consecutive cells (warp ballots, then across the tile's warps)
//   2. MergeKernel         unions with the -y and -x neighbours and, at tile heads, with -z;
//                          a union already implied by the z runs is skipped
//   3. MarkRootsKernel     1 bit per cell (parent[i] == i) and its popcount per 32-cell word
//   4. an exclusive scan of the word counts (CUB), the last entry = the number of components
//   5. WriteComponentsKernel  find(i), rank of the root from the mask, the cell rewritten with the
//                          new component word; every other word is copied as it was read
// Scratch, stream-ordered: 4 B per cell (parent) + 1 bit per cell (root mask) + 4 B per 32 cells
// (word counts / prefix) + the scan's temporary storage.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>

#include <atomic>
#include <functional>
#include <initializer_list>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include "common.cuh"
#include "host_transfer.cuh"

namespace vgt_b200
{
namespace components
{
namespace
{
// ---------------------------------------------------------------------------------------------
// The connection rules: two face neighbours a and b are connected iff their keys are equal.
// Both rules are restated from the reference's member bodies (not checked against the reference's
// own members in this tree; DESIGN.md section 4). The float compare `occupancy > 0.5f` gives the
// reference's `occupancy > 0.5` (float promoted to double against the literal) exactly; NaN is
// not > 0.5 and so joins the free and unknown cells.
// ---------------------------------------------------------------------------------------------
struct Key
{
  uint32_t filled;
  uint32_t object_id;
};

__device__ __forceinline__ bool operator==(const Key& a, const Key& b)
{
  return a.filled == b.filled && a.object_id == b.object_id;
}

// OccupancyComponentMap (8-byte cells {float occupancy, uint32 component}):
// connected iff (occupancy_a > 0.5) == (occupancy_b > 0.5).
__device__ __forceinline__ Key OccupancyComponentKey(const uint32_t* cell)
{
  return Key{__uint_as_float(cell[0]) > 0.5f ? 1u : 0u, 0u};
}

// TaggedObjectOccupancyComponentMap (16-byte cells {occupancy, object_id, component,
// spatial_segment}): connected iff (occupancy_a > 0.5) == (occupancy_b > 0.5) and
// object_id_a == object_id_b.
__device__ __forceinline__ Key TaggedObjectComponentKey(const uint32_t* cell)
{
  return Key{__uint_as_float(cell[0]) > 0.5f ? 1u : 0u, cell[1]};
}

template <int kCellWords>
__device__ __forceinline__ Key CellKey(const uint32_t* __restrict__ cells, uint32_t i)
{
  const uint32_t* cell = cells + static_cast<size_t>(i) * kCellWords;
  if constexpr (kCellWords == 2)
  {
    return OccupancyComponentKey(cell);
  }
  else
  {
    return TaggedObjectComponentKey(cell);
  }
}

// The word of each layout the component is written to.
template <int kCellWords>
constexpr int kComponentWord = kCellWords == 2 ? 1 : 2;

constexpr int kThreads = 256;
constexpr int kRunTile = kThreads;  // the z runs of step 1 are found inside tiles of this many cells
constexpr int kWarps = kThreads / 32;

struct Grid
{
  uint32_t nx, ny, nz;
  uint32_t count;  // nx * ny * nz < 2^32
};

// ---------------------------------------------------------------------------------------------
// Union-find on parent[] (parent[i] <= i). find() halves the path it walks with plain stores:
// only non-roots are ever written that way, and a non-root never becomes a root again, while a
// link is made only by a compare-and-swap on a root (so the two never write the same word).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t Find(uint32_t* parent, uint32_t i)
{
  uint32_t current = __ldcg(parent + i);
  if (current != i)
  {
    uint32_t previous = i;
    uint32_t next;
    while (current > (next = __ldcg(parent + current)))
    {
      parent[previous] = next;
      previous = current;
      current = next;
    }
  }
  return current;
}

__device__ __forceinline__ void Union(uint32_t* parent, uint32_t a, uint32_t b)
{
  a = Find(parent, a);
  b = Find(parent, b);
  while (a != b)
  {
    if (a < b)
    {
      const uint32_t old = atomicCAS(parent + b, b, a);  // hang the larger root under the smaller
      if (old == b)
      {
        return;
      }
      b = old;
    }
    else
    {
      const uint32_t old = atomicCAS(parent + a, a, b);
      if (old == a)
      {
        return;
      }
      a = old;
    }
  }
}

// Step 1: parent[i] = the first cell of i's run of equal keys along z, within i's tile of
// kRunTile consecutive cells (linear order, so a tile may span several z rows); a tile head whose
// run began in the previous tile is its own parent until step 2 joins it to cell i - 1.
template <int kCellWords>
__global__ void __launch_bounds__(kThreads)
InitRunsKernel(const uint32_t* __restrict__ cells, Grid grid, uint32_t* __restrict__ parent)
{
  __shared__ int last_start[kWarps];
  const uint32_t tile_first = blockIdx.x * kRunTile;
  const uint32_t i = tile_first + threadIdx.x;
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  bool start = true;
  if (i < grid.count && threadIdx.x > 0 && (i % grid.nz) != 0)
  {
    start = !(CellKey<kCellWords>(cells, i) == CellKey<kCellWords>(cells, i - 1));
  }
  const uint32_t starts = __ballot_sync(0xffffffffu, start);
  if (lane == 31)
  {
    last_start[warp] = (starts != 0u) ? (warp * 32 + 31 - __clz(starts)) : -1;
  }
  __syncthreads();
  if (i >= grid.count)
  {
    return;
  }
  const uint32_t at_or_below = starts & (0xffffffffu >> (31 - lane));
  int run_start;
  if (at_or_below != 0u)
  {
    run_start = warp * 32 + 31 - __clz(at_or_below);
  }
  else
  {
    run_start = 0;  // thread 0 of the tile is always a start
    for (int w = warp - 1; w >= 0; w--)
    {
      if (last_start[w] >= 0)
      {
        run_start = last_start[w];
        break;
      }
    }
  }
  parent[i] = tile_first + static_cast<uint32_t>(run_start);
}

// Step 2: unions with the -y and -x face neighbours (and -z at tile heads). The union of i with
// its neighbour j = i - stride is implied, and skipped, when i - 1 and j - 1 lie in the same z
// rows and have the same key as i: i ~ i-1 and j ~ j-1 by their runs, i-1 ~ j-1 by the thread
// of i - 1 (or, recursively, by the implication one cell further down).
template <int kCellWords>
__global__ void __launch_bounds__(kThreads)
MergeKernel(const uint32_t* __restrict__ cells, Grid grid, uint32_t* parent)
{
  const uint32_t i = blockIdx.x * kThreads + threadIdx.x;
  if (i >= grid.count)
  {
    return;
  }
  const uint32_t z = i % grid.nz;
  const uint32_t row = i / grid.nz;
  const uint32_t y = row % grid.ny;
  const uint32_t x = row / grid.ny;
  const Key key = CellKey<kCellWords>(cells, i);
  const bool same_below = z > 0 && CellKey<kCellWords>(cells, i - 1) == key;
  if (same_below && (i % kRunTile) == 0)
  {
    Union(parent, i, i - 1);
  }
  if (y > 0)
  {
    const uint32_t j = i - grid.nz;
    if (CellKey<kCellWords>(cells, j) == key
        && !(same_below && CellKey<kCellWords>(cells, j - 1) == key))
    {
      Union(parent, i, j);
    }
  }
  if (x > 0)
  {
    const uint32_t j = i - grid.ny * grid.nz;
    if (CellKey<kCellWords>(cells, j) == key
        && !(same_below && CellKey<kCellWords>(cells, j - 1) == key))
    {
      Union(parent, i, j);
    }
  }
}

// Step 3: root mask and its popcount per 32-cell word (cells past the grid are not roots).
__global__ void __launch_bounds__(kThreads)
MarkRootsKernel(const uint32_t* __restrict__ parent, uint32_t count, uint32_t* __restrict__ mask,
                uint32_t* __restrict__ word_counts)
{
  const uint32_t i = blockIdx.x * kThreads + threadIdx.x;
  const bool root = i < count && __ldg(parent + i) == i;
  const uint32_t bits = __ballot_sync(0xffffffffu, root);
  if ((threadIdx.x & 31) == 0 && i < count)
  {
    mask[i >> 5] = bits;
    word_counts[i >> 5] = static_cast<uint32_t>(__popc(bits));
  }
}

// Step 5: component = rank of the root + 1, written into the cell; the other words are copied as
// read (raw bits: NaN payloads, object ids and spatial segments come back unchanged).
template <int kCellWords>
__global__ void __launch_bounds__(kThreads)
WriteComponentsKernel(uint32_t* __restrict__ cells, uint32_t count, uint32_t* parent,
                      const uint32_t* __restrict__ mask, const uint32_t* __restrict__ word_prefix)
{
  const uint32_t i = blockIdx.x * kThreads + threadIdx.x;
  if (i >= count)
  {
    return;
  }
  const uint32_t root = Find(parent, i);
  const uint32_t below = __ldg(mask + (root >> 5)) & ((1u << (root & 31)) - 1u);
  const uint32_t component = __ldg(word_prefix + (root >> 5)) + static_cast<uint32_t>(__popc(below))
                           + 1u;
  uint32_t* cell = cells + static_cast<size_t>(i) * kCellWords;
  uint32_t words[kCellWords];
#pragma unroll
  for (int w = 0; w < kCellWords; w++)
  {
    words[w] = __ldcs(cell + w);
  }
  words[kComponentWord<kCellWords>] = component;
#pragma unroll
  for (int w = 0; w < kCellWords; w++)
  {
    __stcs(cell + w, words[w]);
  }
}

int CheckArguments(const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz,
                   const void* num_components, Grid* grid)
{
  if (cells == nullptr)
  {
    return FailInvalid("null cell array");
  }
  if (num_components == nullptr)
  {
    return FailInvalid("null component count");
  }
  if (cell_bytes != 8 && cell_bytes != 16)
  {
    return FailInvalid("cell size must be 8 (OccupancyComponentCell) or 16 "
                       "(TaggedObjectOccupancyComponentCell) bytes");
  }
  if (!ValidDims(nx, ny, nz))
  {
    return FailInvalid("grid dimensions %lld x %lld x %lld out of range",
                       static_cast<long long>(nx), static_cast<long long>(ny),
                       static_cast<long long>(nz));
  }
  const int64_t count = nx * ny * nz;
  if (count >= (int64_t{1} << 32))
  {
    SetLastError("connected components: grids of 2^32 cells or more are not supported "
                 "(%lld cells)", static_cast<long long>(count));
    return VGT_B200_ERR_UNSUPPORTED;
  }
  *grid = Grid{static_cast<uint32_t>(nx), static_cast<uint32_t>(ny), static_cast<uint32_t>(nz),
               static_cast<uint32_t>(count)};
  return VGT_B200_OK;
}

template <int kCellWords>
int LaunchAll(uint32_t* d_cells, const Grid& grid, uint32_t* d_num_components,
              cudaStream_t stream)
{
  const uint32_t blocks = (grid.count + kThreads - 1) / kThreads;
  const uint32_t words = (grid.count + 31) / 32;
  StreamScratch<uint32_t> parent;
  StreamScratch<uint32_t> mask;
  StreamScratch<uint32_t> word_prefix;  // words + 1 entries: the last one ends as the total
  StreamScratch<char> scan_storage;
  VGT_CUDA_TRY(parent.Allocate(grid.count, stream), "parent allocation");
  VGT_CUDA_TRY(mask.Allocate(words, stream), "root mask allocation");
  VGT_CUDA_TRY(word_prefix.Allocate(int64_t{words} + 1, stream), "word count allocation");
  size_t scan_bytes = 0;
  VGT_CUDA_TRY(cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, word_prefix.get(),
                                             word_prefix.get(), static_cast<int>(words) + 1,
                                             stream),
               "scan size query");
  VGT_CUDA_TRY(scan_storage.Allocate(static_cast<int64_t>(std::max<size_t>(scan_bytes, 1)),
                                     stream),
               "scan storage allocation");
  VGT_CUDA_TRY(cudaMemsetAsync(word_prefix.get() + words, 0, sizeof(uint32_t), stream),
               "count reset");

  InitRunsKernel<kCellWords><<<blocks, kThreads, 0, stream>>>(d_cells, grid, parent.get());
  NoteKernelLaunch();
  VGT_CUDA_TRY(cudaGetLastError(), "InitRunsKernel launch");
  MergeKernel<kCellWords><<<blocks, kThreads, 0, stream>>>(d_cells, grid, parent.get());
  NoteKernelLaunch();
  VGT_CUDA_TRY(cudaGetLastError(), "MergeKernel launch");
  MarkRootsKernel<<<blocks, kThreads, 0, stream>>>(parent.get(), grid.count, mask.get(),
                                                   word_prefix.get());
  NoteKernelLaunch();
  VGT_CUDA_TRY(cudaGetLastError(), "MarkRootsKernel launch");
  VGT_CUDA_TRY(cub::DeviceScan::ExclusiveSum(scan_storage.get(), scan_bytes, word_prefix.get(),
                                             word_prefix.get(), static_cast<int>(words) + 1,
                                             stream),
               "root rank scan");
  NoteKernelLaunch();  // the scan is two kernels (tile-state init, then the scan)
  NoteKernelLaunch();
  WriteComponentsKernel<kCellWords><<<blocks, kThreads, 0, stream>>>(
      d_cells, grid.count, parent.get(), mask.get(), word_prefix.get());
  NoteKernelLaunch();
  VGT_CUDA_TRY(cudaGetLastError(), "WriteComponentsKernel launch");
  VGT_CUDA_TRY(cudaMemcpyAsync(d_num_components, word_prefix.get() + words, sizeof(uint32_t),
                               cudaMemcpyDeviceToDevice, stream),
               "component count copy");
  return VGT_B200_OK;
}

int Launch(void* d_cells, int cell_bytes, const Grid& grid, uint32_t* d_num_components,
           cudaStream_t stream)
{
  if (cell_bytes == 8)
  {
    return LaunchAll<2>(static_cast<uint32_t*>(d_cells), grid, d_num_components, stream);
  }
  return LaunchAll<4>(static_cast<uint32_t*>(d_cells), grid, d_num_components, stream);
}

// =============================================================================================
// The map cut into x-slabs (vgt_b200_connected_components_multi). Slab g = planes [x0_g, x1_g)
// (SplitRange) on devices[g] is labelled by steps 1-4 above as a grid of its own, with 32-bit
// local indices; local index l of slab g is global index x0_g * ny * nz + l (64 bits). Because a
// slab is one contiguous range of storage order and every local root is the smallest index of
// its local set, the smallest index of a component is a local root in the lowest slab it
// touches, and only the cells of the x-faces between slabs can join local sets of different
// slabs. So:
//   a. per face, FaceEdgesKernel emits (global root of the cell below, global root of the cell
//      above) where the keys are equal and the edge is not implied by the (y, z - 1) pair;
//   b. on every slab's device the endpoints of all faces' edges are sorted and made unique (the
//      nodes), the edges are mapped to compact node ids by binary search and joined by
//      union-find with parent <= self; compact order is global order, so a node's compact root
//      is the smallest global index of its merged set, and every slab gets the same table;
//   c. per slab, one bit per local component, cleared for the slab's nodes whose compact root is
//      another node; the bits left are the components whose smallest index lies in the slab,
//      count_g of them, and component ids are offset_g + 1 + rank among them (offset_g = the
//      sum of the counts of the slabs below): the reference's numbering;
//   d. each slab publishes the ids of its nodes into a node-id array that is zero elsewhere; with
//      the arrays of all slabs added up, every node takes the id of its compact root, and each
//      slab writes final[local rank] into the component word of its cells.
// In vgt_b200_connected_components_multi everything that crosses slabs (face planes and roots,
// edges, node ids) goes through host memory: it is O(num_slabs * ny * nz). The
// vgt_b200_components_* entries run the same phases on one slab per process and leave the
// crossing to the caller's collectives.
// Scratch per slab, on its device: the slab's cells + 4 B per cell (parent) + about 0.25 B per
// cell (root mask, word prefix) + 4 B per local component (final ids) + about 0.25 B per local
// component (root bits, word prefix), + O(ny * nz) for the faces, and the face graph of
// E = at most (num_slabs - 1) * ny * nz edges: at most 64 B per edge (the edges, their sorted
// endpoints, the nodes, their parents and compact roots).
// =============================================================================================
struct Edge
{
  uint64_t a, b;  // global indices of two local roots, a in the slab below
};

// Rank of local root r among the slab's local roots (step 3's mask and step 4's prefix).
__device__ __forceinline__ uint32_t RootRank(const uint32_t* __restrict__ mask,
                                             const uint32_t* __restrict__ word_prefix, uint32_t r)
{
  const uint32_t below = __ldg(mask + (r >> 5)) & ((1u << (r & 31)) - 1u);
  return __ldg(word_prefix + (r >> 5)) + static_cast<uint32_t>(__popc(below));
}

// The local root of each cell of the slab's last x-plane (first = its first local index).
__global__ void __launch_bounds__(kThreads)
FaceRootsKernel(uint32_t* parent, uint32_t first, uint32_t plane, uint32_t* __restrict__ roots)
{
  const uint32_t k = blockIdx.x * kThreads + threadIdx.x;
  if (k < plane)
  {
    roots[k] = Find(parent, first + k);
  }
}

// Step a, on the slab above the face: below_cells / below_roots are the last plane of the slab
// below (its cells and their local roots), cells / parent the slab's own (its first plane is
// local 0 .. plane - 1). The edge of (y, z) is implied when (y, z - 1) has the same key on both
// sides: each cell is in its z-neighbour's local set, and (y, z - 1) is joined or implied itself.
template <int kCellWords>
__global__ void __launch_bounds__(kThreads)
FaceEdgesKernel(const uint32_t* __restrict__ below_cells, const uint32_t* __restrict__ below_roots,
                uint64_t below_base, const uint32_t* __restrict__ cells, uint32_t* parent,
                uint64_t base, uint32_t plane, uint32_t nz, Edge* __restrict__ edges,
                uint32_t* __restrict__ edge_count)
{
  const uint32_t k = blockIdx.x * kThreads + threadIdx.x;
  bool emit = false;
  if (k < plane)
  {
    const Key key = CellKey<kCellWords>(cells, k);
    emit = CellKey<kCellWords>(below_cells, k) == key
        && !((k % nz) != 0 && CellKey<kCellWords>(cells, k - 1) == key
             && CellKey<kCellWords>(below_cells, k - 1) == key);
  }
  const uint32_t ballot = __ballot_sync(0xffffffffu, emit);
  if (ballot == 0u)
  {
    return;
  }
  const int lane = threadIdx.x & 31;
  uint32_t slot = 0;
  if (lane == __ffs(ballot) - 1)
  {
    slot = atomicAdd(edge_count, static_cast<uint32_t>(__popc(ballot)));
  }
  slot = __shfl_sync(0xffffffffu, slot, __ffs(ballot) - 1);
  if (emit)
  {
    slot += static_cast<uint32_t>(__popc(ballot & ((1u << lane) - 1u)));
    edges[slot] = Edge{below_base + __ldg(below_roots + k), base + Find(parent, k)};
  }
}

// Step b: the first index of sorted[0, n) that is >= value.
__device__ __forceinline__ uint32_t LowerBound(const uint64_t* __restrict__ sorted, uint32_t n,
                                               uint64_t value)
{
  uint32_t lo = 0;
  uint32_t hi = n;
  while (lo < hi)
  {
    const uint32_t mid = lo + (hi - lo) / 2;
    if (__ldg(sorted + mid) < value)
    {
      lo = mid + 1;
    }
    else
    {
      hi = mid;
    }
  }
  return lo;
}

__global__ void __launch_bounds__(kThreads)
NodeInitKernel(uint32_t* __restrict__ node_parent, uint32_t num_nodes)
{
  const uint32_t k = blockIdx.x * kThreads + threadIdx.x;
  if (k < num_nodes)
  {
    node_parent[k] = k;
  }
}

__global__ void __launch_bounds__(kThreads)
NodeUnionKernel(const Edge* __restrict__ edges, uint32_t num_edges,
                const uint64_t* __restrict__ nodes, uint32_t num_nodes, uint32_t* node_parent)
{
  const uint32_t e = blockIdx.x * kThreads + threadIdx.x;
  if (e < num_edges)
  {
    const Edge edge = edges[e];
    Union(node_parent, LowerBound(nodes, num_nodes, edge.a), LowerBound(nodes, num_nodes, edge.b));
  }
}

// node_roots[k] = compact root of k (a separate array: a store into node_parent could be
// overwritten by another thread's path halving), and where each slab's nodes begin:
// slab_first[g] = the first node >= slab_base[g] (num_slabs + 1 entries; the last base is the
// grid's cell count).
__global__ void __launch_bounds__(kThreads)
NodeFlattenKernel(uint32_t* node_parent, const uint64_t* __restrict__ nodes, uint32_t num_nodes,
                  const uint64_t* __restrict__ slab_base, int num_bases,
                  uint32_t* __restrict__ node_roots, uint32_t* __restrict__ slab_first)
{
  const uint32_t k = blockIdx.x * kThreads + threadIdx.x;
  if (k < num_nodes)
  {
    node_roots[k] = Find(node_parent, k);
  }
  if (k < static_cast<uint32_t>(num_bases))
  {
    slab_first[k] = LowerBound(nodes, num_nodes, slab_base[k]);
  }
}

// Step c: one bit per local component, set for all but the last word's padding.
__global__ void __launch_bounds__(kThreads)
GlobalRootBitsInitKernel(uint32_t* __restrict__ bits, uint32_t num_components)
{
  const uint32_t w = blockIdx.x * kThreads + threadIdx.x;
  if (w < (num_components + 31) / 32)
  {
    const uint32_t left = num_components - w * 32;
    bits[w] = left >= 32 ? 0xffffffffu : ((1u << left) - 1u);
  }
}

// Nodes k of the slab (node_first + k in compact ids) whose compact root is another node are not
// global roots: their bit is cleared.
__global__ void __launch_bounds__(kThreads)
ClearMergedBitsKernel(const uint64_t* __restrict__ nodes, const uint32_t* __restrict__ node_roots,
                      uint32_t count, uint32_t node_first, uint64_t base,
                      const uint32_t* __restrict__ mask, const uint32_t* __restrict__ word_prefix,
                      uint32_t* bits)
{
  const uint32_t k = blockIdx.x * kThreads + threadIdx.x;
  if (k < count && node_roots[k] != node_first + k)
  {
    const uint32_t rank = RootRank(mask, word_prefix, static_cast<uint32_t>(nodes[k] - base));
    atomicAnd(bits + (rank >> 5), ~(1u << (rank & 31)));
  }
}

__global__ void __launch_bounds__(kThreads)
BitCountsKernel(const uint32_t* __restrict__ bits, uint32_t words, uint32_t* __restrict__ counts)
{
  const uint32_t w = blockIdx.x * kThreads + threadIdx.x;
  if (w < words)
  {
    counts[w] = static_cast<uint32_t>(__popc(bits[w]));
  }
}

// Step d: final[r] = offset + 1 + rank among the slab's global roots, 0 for merged components
// (overwritten by ApplyNodeIdsKernel).
__global__ void __launch_bounds__(kThreads)
FinalIdsKernel(const uint32_t* __restrict__ bits, const uint32_t* __restrict__ bit_prefix,
               uint32_t num_components, uint32_t offset, uint32_t* __restrict__ final_ids)
{
  const uint32_t r = blockIdx.x * kThreads + threadIdx.x;
  if (r < num_components)
  {
    const uint32_t word = __ldg(bits + (r >> 5));
    final_ids[r] = ((word >> (r & 31)) & 1u) == 0u
                 ? 0u
                 : offset + 1u + __ldg(bit_prefix + (r >> 5))
                       + static_cast<uint32_t>(__popc(word & ((1u << (r & 31)) - 1u)));
  }
}

// ids[k] = final[local rank of node k]: the published id of each root node of the slab.
__global__ void __launch_bounds__(kThreads)
PublishNodeIdsKernel(const uint64_t* __restrict__ nodes, uint32_t count, uint64_t base,
                     const uint32_t* __restrict__ mask, const uint32_t* __restrict__ word_prefix,
                     const uint32_t* __restrict__ final_ids, uint32_t* __restrict__ ids)
{
  const uint32_t k = blockIdx.x * kThreads + threadIdx.x;
  if (k < count)
  {
    ids[k] = final_ids[RootRank(mask, word_prefix, static_cast<uint32_t>(nodes[k] - base))];
  }
}

// On devices[0]: every node takes the id its compact root published (roots keep theirs).
__global__ void __launch_bounds__(kThreads)
NodeIdsFromRootsKernel(const uint32_t* __restrict__ node_roots, uint32_t num_nodes, uint32_t* ids)
{
  const uint32_t k = blockIdx.x * kThreads + threadIdx.x;
  if (k < num_nodes && node_roots[k] != k)
  {
    ids[k] = ids[node_roots[k]];
  }
}

__global__ void __launch_bounds__(kThreads)
ApplyNodeIdsKernel(const uint64_t* __restrict__ nodes, const uint32_t* __restrict__ ids,
                   uint32_t count, uint64_t base, const uint32_t* __restrict__ mask,
                   const uint32_t* __restrict__ word_prefix, uint32_t* __restrict__ final_ids)
{
  const uint32_t k = blockIdx.x * kThreads + threadIdx.x;
  if (k < count)
  {
    final_ids[RootRank(mask, word_prefix, static_cast<uint32_t>(nodes[k] - base))] = ids[k];
  }
}

// Step 5 of a slab: the component word = final[local rank of the cell's local root]; the other
// words are copied as read.
template <int kCellWords>
__global__ void __launch_bounds__(kThreads)
WriteSlabComponentsKernel(uint32_t* __restrict__ cells, uint32_t count, uint32_t* parent,
                          const uint32_t* __restrict__ mask,
                          const uint32_t* __restrict__ word_prefix,
                          const uint32_t* __restrict__ final_ids)
{
  const uint32_t i = blockIdx.x * kThreads + threadIdx.x;
  if (i >= count)
  {
    return;
  }
  const uint32_t component = __ldg(final_ids + RootRank(mask, word_prefix, Find(parent, i)));
  uint32_t* cell = cells + static_cast<size_t>(i) * kCellWords;
  uint32_t words[kCellWords];
#pragma unroll
  for (int w = 0; w < kCellWords; w++)
  {
    words[w] = __ldcs(cell + w);
  }
  words[kComponentWord<kCellWords>] = component;
#pragma unroll
  for (int w = 0; w < kCellWords; w++)
  {
    __stcs(cell + w, words[w]);
  }
}

inline uint32_t Blocks(uint64_t threads)
{
  return static_cast<uint32_t>((threads + kThreads - 1) / kThreads);
}

#define VGT_LAUNCHED(what)                                  \
  do                                                        \
  {                                                         \
    NoteKernelLaunch();                                     \
    VGT_CUDA_TRY(cudaGetLastError(), what " launch");       \
  } while (0)

// ---------------------------------------------------------------------------------------------
// The phases of one slab, each asynchronous on `stream`: steps 1-5 of the slab scheme above.
// vgt_b200_connected_components_multi runs them on host threads and passes what crosses slabs
// through host memory; the vgt_b200_components_* entries run one slab per process and leave the
// crossing to the caller (collectives). Every array that lives from one phase to the next is the
// caller's.
// ---------------------------------------------------------------------------------------------
struct SlabArrays
{
  Grid grid;
  uint64_t base;          // global index of the slab's first cell
  uint32_t* cells;
  uint32_t* parent;       // grid.count
  uint32_t* mask;         // (grid.count + 31) / 32
  uint32_t* word_prefix;  // (grid.count + 31) / 32 + 1; the last entry ends as K_g
  void* scan_storage;     // ScanBytes(grid.count): both scans of the slab
  size_t scan_bytes;
};

// The face graph's nodes as ResolvePhase leaves them, and the slab's share of them.
struct SlabNodes
{
  const uint64_t* nodes;       // the sorted unique endpoints of all edges
  const uint32_t* node_roots;  // their compact roots
  uint32_t num_nodes;
  uint32_t first;              // the slab's nodes are [first, first + count)
  uint32_t count;
};

uint32_t RootWords(uint32_t cells)
{
  return (cells + 31) / 32;
}

// Temporary storage of the scan of a slab's word counts (words + 1 entries); it also fits the
// scan of the root bits (at most as many words).
int ScanBytes(uint32_t count, size_t* bytes)
{
  size_t needed = 0;
  VGT_CUDA_TRY(cub::DeviceScan::ExclusiveSum(nullptr, needed, static_cast<uint32_t*>(nullptr),
                                             static_cast<uint32_t*>(nullptr),
                                             static_cast<int>(RootWords(count)) + 1),
               "scan size query");
  *bytes = std::max<size_t>(needed, 1);
  return VGT_B200_OK;
}

// Step 1: steps 1-4 of the whole-grid labelling on the slab alone; K_g ends in
// word_prefix[words]. face_roots (may be null): the local roots of the slab's last x-plane.
template <int kCellWords>
int LocalPhase(const SlabArrays& slab, uint32_t* face_roots, cudaStream_t stream)
{
  const Grid& grid = slab.grid;
  const uint32_t words = RootWords(grid.count);
  const uint32_t blocks = Blocks(grid.count);
  VGT_CUDA_TRY(cudaMemsetAsync(slab.word_prefix + words, 0, sizeof(uint32_t), stream),
               "count reset");
  InitRunsKernel<kCellWords><<<blocks, kThreads, 0, stream>>>(slab.cells, grid, slab.parent);
  VGT_LAUNCHED("InitRunsKernel");
  MergeKernel<kCellWords><<<blocks, kThreads, 0, stream>>>(slab.cells, grid, slab.parent);
  VGT_LAUNCHED("MergeKernel");
  MarkRootsKernel<<<blocks, kThreads, 0, stream>>>(slab.parent, grid.count, slab.mask,
                                                   slab.word_prefix);
  VGT_LAUNCHED("MarkRootsKernel");
  size_t scan_bytes = slab.scan_bytes;
  VGT_CUDA_TRY(cub::DeviceScan::ExclusiveSum(slab.scan_storage, scan_bytes, slab.word_prefix,
                                             slab.word_prefix, static_cast<int>(words) + 1,
                                             stream),
               "root rank scan");
  NoteKernelLaunch();  // the scan is two kernels (tile-state init, then the scan)
  NoteKernelLaunch();
  if (face_roots != nullptr)
  {
    const uint32_t plane = grid.ny * grid.nz;
    FaceRootsKernel<<<Blocks(plane), kThreads, 0, stream>>>(slab.parent, grid.count - plane,
                                                            plane, face_roots);
    VGT_LAUNCHED("FaceRootsKernel");
  }
  return VGT_B200_OK;
}

// Step 2, on the slab above the face: below_cells / below_roots are the last x-plane of the slab
// below (its cells as stored and their local roots), below_base that slab's first global index.
// At most ny * nz edges; their number ends in *edge_count.
template <int kCellWords>
int FaceEdgesPhase(const uint32_t* below_cells, const uint32_t* below_roots, uint64_t below_base,
                   const SlabArrays& slab, Edge* edges, uint32_t* edge_count, cudaStream_t stream)
{
  const uint32_t plane = slab.grid.ny * slab.grid.nz;
  VGT_CUDA_TRY(cudaMemsetAsync(edge_count, 0, sizeof(uint32_t), stream), "edge count reset");
  FaceEdgesKernel<kCellWords><<<Blocks(plane), kThreads, 0, stream>>>(
      below_cells, below_roots, below_base, slab.cells, slab.parent, slab.base, plane,
      slab.grid.nz, edges, edge_count);
  VGT_LAUNCHED("FaceEdgesKernel");
  return VGT_B200_OK;
}

// Step 3: the edges of all faces (any order) sorted and made unique into nodes, joined and
// flattened. nodes / node_roots hold max(1, 2 * num_edges) entries: nodes past the node count
// are all ones (so binary searches over the whole array find the real ones) and their roots are
// themselves. node_words[0] = the node count, node_words[1 + b] = the first node >= bases[b]
// (host array, num_bases entries below num_cells). Compact roots are set minima, so every caller
// that passes the same edges gets the same nodes and roots whatever their order.
int ResolvePhase(const Edge* edges, uint32_t num_edges, uint64_t num_cells,
                 const uint64_t* bases, int num_bases, uint64_t* nodes, uint32_t* node_roots,
                 uint32_t* node_words, cudaStream_t stream)
{
  const int num_endpoints = static_cast<int>(2 * num_edges);
  const uint32_t capacity = std::max<uint32_t>(1, 2 * num_edges);
  StreamScratch<uint64_t> sorted;
  StreamScratch<uint32_t> node_parent;
  StreamScratch<uint64_t> d_bases;
  StreamScratch<char> storage;
  VGT_CUDA_TRY(sorted.Allocate(capacity, stream), "endpoint allocation");
  VGT_CUDA_TRY(node_parent.Allocate(capacity, stream), "node parent allocation");
  VGT_CUDA_TRY(d_bases.Allocate(num_bases, stream), "base allocation");
  VGT_CUDA_TRY(cudaMemcpyAsync(d_bases.get(), bases, sizeof(uint64_t) * num_bases,
                               cudaMemcpyHostToDevice, stream),
               "copy bases");
  VGT_CUDA_TRY(cudaMemsetAsync(nodes, 0xff, sizeof(uint64_t) * capacity, stream), "node reset");
  VGT_CUDA_TRY(cudaMemsetAsync(node_words, 0, sizeof(uint32_t), stream), "node count reset");
  int end_bit = 1;
  while (end_bit < 64 && (num_cells >> end_bit) != 0)
  {
    end_bit++;
  }
  const uint64_t* endpoints = reinterpret_cast<const uint64_t*>(edges);
  size_t sort_bytes = 0;
  size_t unique_bytes = 0;
  VGT_CUDA_TRY(cub::DeviceRadixSort::SortKeys(nullptr, sort_bytes, endpoints, sorted.get(),
                                              num_endpoints, 0, end_bit, stream),
               "sort size query");
  VGT_CUDA_TRY(cub::DeviceSelect::Unique(nullptr, unique_bytes, sorted.get(), nodes, node_words,
                                         num_endpoints, stream),
               "unique size query");
  const size_t storage_bytes = std::max<size_t>({sort_bytes, unique_bytes, 1});
  VGT_CUDA_TRY(storage.Allocate(static_cast<int64_t>(storage_bytes), stream),
               "resolve storage allocation");
  if (num_edges > 0)
  {
    VGT_CUDA_TRY(cub::DeviceRadixSort::SortKeys(storage.get(), sort_bytes, endpoints, sorted.get(),
                                                num_endpoints, 0, end_bit, stream),
                 "endpoint sort");
    NoteKernelLaunch();
    VGT_CUDA_TRY(cub::DeviceSelect::Unique(storage.get(), unique_bytes, sorted.get(), nodes,
                                           node_words, num_endpoints, stream),
                 "endpoint unique");
    NoteKernelLaunch();
    NodeInitKernel<<<Blocks(capacity), kThreads, 0, stream>>>(node_parent.get(), capacity);
    VGT_LAUNCHED("NodeInitKernel");
    NodeUnionKernel<<<Blocks(num_edges), kThreads, 0, stream>>>(edges, num_edges, nodes,
                                                                capacity, node_parent.get());
    VGT_LAUNCHED("NodeUnionKernel");
  }
  const uint32_t flattened = num_edges > 0 ? capacity : 0;
  NodeFlattenKernel<<<Blocks(std::max<uint32_t>(capacity, num_bases)), kThreads, 0, stream>>>(
      node_parent.get(), nodes, flattened, d_bases.get(), num_bases, node_roots, node_words + 1);
  VGT_LAUNCHED("NodeFlattenKernel");
  return VGT_B200_OK;
}

// Step 4: one bit per local component, cleared for the slab's nodes whose compact root is another
// node; count_g (the bits left) ends in bit_prefix[bit words].
int CountPhase(const SlabArrays& slab, uint32_t num_components, const SlabNodes& graph,
               uint32_t* bits, uint32_t* bit_prefix, cudaStream_t stream)
{
  const uint32_t bit_words = RootWords(num_components);
  GlobalRootBitsInitKernel<<<Blocks(bit_words), kThreads, 0, stream>>>(bits, num_components);
  VGT_LAUNCHED("GlobalRootBitsInitKernel");
  if (graph.count > 0)
  {
    ClearMergedBitsKernel<<<Blocks(graph.count), kThreads, 0, stream>>>(
        graph.nodes + graph.first, graph.node_roots + graph.first, graph.count, graph.first,
        slab.base, slab.mask, slab.word_prefix, bits);
    VGT_LAUNCHED("ClearMergedBitsKernel");
  }
  VGT_CUDA_TRY(cudaMemsetAsync(bit_prefix + bit_words, 0, sizeof(uint32_t), stream),
               "count reset");
  BitCountsKernel<<<Blocks(bit_words), kThreads, 0, stream>>>(bits, bit_words, bit_prefix);
  VGT_LAUNCHED("BitCountsKernel");
  size_t scan_bytes = slab.scan_bytes;
  VGT_CUDA_TRY(cub::DeviceScan::ExclusiveSum(slab.scan_storage, scan_bytes, bit_prefix, bit_prefix,
                                             static_cast<int>(bit_words) + 1, stream),
               "global root scan");
  NoteKernelLaunch();
  NoteKernelLaunch();
  return VGT_B200_OK;
}

// Step 5a: final[r] = offset + 1 + rank among the slab's global roots (0 for merged components);
// node_ids[first + k] = the final id of the slab's node k (node_ids: one word per node, zero
// elsewhere; after the ids of all slabs are added up, every root node holds its id).
int PublishPhase(const SlabArrays& slab, uint32_t num_components, uint32_t offset,
                 const SlabNodes& graph, const uint32_t* bits, const uint32_t* bit_prefix,
                 uint32_t* final_ids, uint32_t* node_ids, cudaStream_t stream)
{
  FinalIdsKernel<<<Blocks(num_components), kThreads, 0, stream>>>(bits, bit_prefix,
                                                                  num_components, offset,
                                                                  final_ids);
  VGT_LAUNCHED("FinalIdsKernel");
  if (graph.count > 0)
  {
    PublishNodeIdsKernel<<<Blocks(graph.count), kThreads, 0, stream>>>(
        graph.nodes + graph.first, graph.count, slab.base, slab.mask, slab.word_prefix, final_ids,
        node_ids + graph.first);
    VGT_LAUNCHED("PublishNodeIdsKernel");
  }
  return VGT_B200_OK;
}

// Step 5b, on the ids of every slab added up: every node takes its compact root's id, the
// slab's merged components take their nodes' ids, and every cell's component word is written.
template <int kCellWords>
int WritePhase(const SlabArrays& slab, const SlabNodes& graph, uint32_t* node_ids,
               uint32_t* final_ids, cudaStream_t stream)
{
  if (graph.num_nodes > 0)
  {
    NodeIdsFromRootsKernel<<<Blocks(graph.num_nodes), kThreads, 0, stream>>>(
        graph.node_roots, graph.num_nodes, node_ids);
    VGT_LAUNCHED("NodeIdsFromRootsKernel");
  }
  if (graph.count > 0)
  {
    ApplyNodeIdsKernel<<<Blocks(graph.count), kThreads, 0, stream>>>(
        graph.nodes + graph.first, node_ids + graph.first, graph.count, slab.base, slab.mask,
        slab.word_prefix, final_ids);
    VGT_LAUNCHED("ApplyNodeIdsKernel");
  }
  WriteSlabComponentsKernel<kCellWords><<<Blocks(slab.grid.count), kThreads, 0, stream>>>(
      slab.cells, slab.grid.count, slab.parent, slab.mask, slab.word_prefix, final_ids);
  VGT_LAUNCHED("WriteSlabComponentsKernel");
  return VGT_B200_OK;
}

// Every check of vgt_b200_connected_components_multi, before any device call.
int CheckMultiArguments(const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz,
                        const int* devices, int num_slabs, const void* num_components)
{
  if (cells == nullptr)
  {
    return FailInvalid("null cell array");
  }
  if (devices == nullptr)
  {
    return FailInvalid("null device list");
  }
  if (num_components == nullptr)
  {
    return FailInvalid("null component count");
  }
  if (num_slabs < 1 || num_slabs > 8)
  {
    return FailInvalid("1..8 slabs are supported (%d requested)", num_slabs);
  }
  if (cell_bytes != 8 && cell_bytes != 16)
  {
    return FailInvalid("cell size must be 8 (OccupancyComponentCell) or 16 "
                       "(TaggedObjectOccupancyComponentCell) bytes");
  }
  if (!ValidDims(nx, ny, nz))
  {
    return FailInvalid("grid dimensions %lld x %lld x %lld out of range",
                       static_cast<long long>(nx), static_cast<long long>(ny),
                       static_cast<long long>(nz));
  }
  if (num_slabs > nx)
  {
    return FailInvalid("more slabs (%d) than x-planes (%lld)", num_slabs,
                       static_cast<long long>(nx));
  }
  for (int g = 0; g < num_slabs; g++)
  {
    if (devices[g] < 0)
    {
      return FailInvalid("device ordinal %d out of range", devices[g]);
    }
  }
  const int64_t widest = (nx + num_slabs - 1) / num_slabs * ny * nz;
  if (widest >= (int64_t{1} << 32))
  {
    SetLastError("connected components: slabs of 2^32 cells or more are not supported "
                 "(%lld cells in the widest of %d slabs)", static_cast<long long>(widest),
                 num_slabs);
    return VGT_B200_ERR_UNSUPPORTED;
  }
  return VGT_B200_OK;
}

template <int kCellWords>
int ConnectedComponentsSlabs(char* h_cells, int64_t nx, int64_t ny, int64_t nz,
                             const int* devices, int num_slabs, uint32_t* out_num_components)
{
  constexpr size_t kCellBytes = sizeof(uint32_t) * kCellWords;
  const uint32_t plane = static_cast<uint32_t>(ny * nz);
  std::vector<int64_t> x_begin(static_cast<size_t>(num_slabs) + 1);
  for (int g = 0; g < num_slabs; g++)
  {
    int64_t end;
    SplitRange(nx, num_slabs, g, &x_begin[static_cast<size_t>(g)], &end);
  }
  x_begin[static_cast<size_t>(num_slabs)] = nx;
  std::vector<uint64_t> slab_base(static_cast<size_t>(num_slabs) + 1);
  for (int g = 0; g <= num_slabs; g++)
  {
    slab_base[static_cast<size_t>(g)] = static_cast<uint64_t>(x_begin[static_cast<size_t>(g)])
                                      * plane;
  }
  const uint64_t num_cells = slab_base[static_cast<size_t>(num_slabs)];

  // What one slab's thread shows the others between phases (written before a barrier, read
  // after it). Everything that crosses slabs goes through host memory with plain async copies:
  // it is O(num_slabs * ny * nz), and neither peer access nor access to another device's
  // stream-ordered pool is needed.
  struct Shared
  {
    std::vector<uint32_t> last_plane;  // the slab's last x-plane of cells
    std::vector<uint32_t> face_roots;  // and the local roots of its cells
    std::vector<Edge> edges;           // the edges of the face below the slab
    uint64_t num_global_roots = 0;     // count_g
    std::vector<uint32_t> node_ids;    // the ids of the slab's nodes (PublishPhase)
    uint32_t first_node = 0;
  };
  std::vector<Shared> shared(static_cast<size_t>(num_slabs));
  std::atomic<uint64_t> total_components{0};

  ThreadBarrier barrier(num_slabs);
  std::vector<int> statuses(static_cast<size_t>(num_slabs), VGT_B200_OK);
  std::vector<std::string> messages(static_cast<size_t>(num_slabs));
  std::atomic<int> failed{0};
  const char* const kStoodDown = "another slab failed";

  const auto worker = [&](const int g)
  {
    const size_t s = static_cast<size_t>(g);
    const int device = devices[g];
    ScopedDevice scoped(device);
    const int64_t slab_x = x_begin[s + 1] - x_begin[s];
    const Grid grid{static_cast<uint32_t>(slab_x), static_cast<uint32_t>(ny),
                    static_cast<uint32_t>(nz), static_cast<uint32_t>(slab_x * plane)};
    const uint32_t words = RootWords(grid.count);
    const size_t slab_bytes = kCellBytes * grid.count;
    char* const h_slab = h_cells + kCellBytes * slab_base[s];
    uint32_t num_components = 0;
    uint32_t node_words[3] = {0, 0, 0};  // node count, the slab's first node, its end
    SlabNodes graph{};

    StreamGuard guard;
    StreamScratch<uint32_t> d_cells;
    StreamScratch<uint32_t> parent;
    StreamScratch<uint32_t> mask;
    StreamScratch<uint32_t> word_prefix;
    StreamScratch<char> scan_storage;
    StreamScratch<uint32_t> face_roots;
    StreamScratch<uint32_t> below_plane;
    StreamScratch<uint32_t> below_roots;
    StreamScratch<Edge> edges;
    StreamScratch<uint32_t> edge_count;
    StreamScratch<Edge> all_edges;
    StreamScratch<uint64_t> nodes;
    StreamScratch<uint32_t> node_roots;
    StreamScratch<uint32_t> d_node_words;
    StreamScratch<uint32_t> bits;
    StreamScratch<uint32_t> bit_prefix;
    StreamScratch<uint32_t> final_ids;
    StreamScratch<uint32_t> node_ids;
    SlabArrays slab{grid, slab_base[s], nullptr, nullptr, nullptr, nullptr, nullptr, 0};
    StagedTransfer transfer;
    if (num_slabs >= 6)
    {
      // enough slab threads to be the parallel copy workers themselves (the shared workers serve
      // one caller at a time)
      transfer.UseCallingThreadOnly();
    }
    struct DrainOnExit
    {
      const StreamGuard& guard;
      ~DrainOnExit()
      {
        if (guard.stream != nullptr)
        {
          cudaStreamSynchronize(guard.stream);
        }
      }
    } drain{guard};

    // 1. the slab up, labelled on its own, K_g; the local roots of its last plane for the slab
    //    above
    const auto local_labelling = [&]() -> int
    {
      VGT_CUDA_TRY(scoped.Status(), "cudaSetDevice");
      KeepPoolMemory(device);
      VGT_CUDA_TRY(cudaStreamCreateWithFlags(&guard.stream, cudaStreamNonBlocking), "stream");
      cudaStream_t stream = guard.stream;
      const int scanned = ScanBytes(grid.count, &slab.scan_bytes);
      if (scanned != VGT_B200_OK)
      {
        return scanned;
      }
      VGT_CUDA_TRY(d_cells.Allocate(static_cast<int64_t>(grid.count) * kCellWords, stream),
                   "cell slab allocation");
      VGT_CUDA_TRY(parent.Allocate(grid.count, stream), "parent allocation");
      VGT_CUDA_TRY(mask.Allocate(words, stream), "root mask allocation");
      VGT_CUDA_TRY(word_prefix.Allocate(int64_t{words} + 1, stream), "word count allocation");
      VGT_CUDA_TRY(scan_storage.Allocate(static_cast<int64_t>(slab.scan_bytes), stream),
                   "scan storage allocation");
      slab.cells = d_cells.get();
      slab.parent = parent.get();
      slab.mask = mask.get();
      slab.word_prefix = word_prefix.get();
      slab.scan_storage = scan_storage.get();
      VGT_CUDA_TRY(transfer.ToDevice(reinterpret_cast<char*>(d_cells.get()), slab_bytes, h_slab,
                                     slab_bytes, slab_bytes, 1, stream),
                   "copy cell slab to device");
      const bool above = g + 1 < num_slabs;
      if (above)
      {
        VGT_CUDA_TRY(face_roots.Allocate(plane, stream), "face root allocation");
      }
      const int labelled = LocalPhase<kCellWords>(slab, above ? face_roots.get() : nullptr,
                                                  stream);
      if (labelled != VGT_B200_OK)
      {
        return labelled;
      }
      if (above)
      {
        Shared& face = shared[s];
        face.last_plane.resize(size_t{plane} * kCellWords);
        face.face_roots.resize(plane);
        VGT_CUDA_TRY(cudaMemcpyAsync(face.face_roots.data(), face_roots.get(),
                                     sizeof(uint32_t) * plane, cudaMemcpyDeviceToHost, stream),
                     "copy face roots to host");
        VGT_CUDA_TRY(cudaMemcpyAsync(face.last_plane.data(),
                                     d_cells.get() + size_t{grid.count - plane} * kCellWords,
                                     kCellBytes * plane, cudaMemcpyDeviceToHost, stream),
                     "copy face cells to host");
      }
      VGT_CUDA_TRY(cudaMemcpyAsync(&num_components, word_prefix.get() + words, sizeof(uint32_t),
                                   cudaMemcpyDeviceToHost, stream),
                   "copy local component count");
      VGT_CUDA_TRY(cudaStreamSynchronize(stream), "slab labelling");
      return VGT_B200_OK;
    };

    // 2. the edges of the face below the slab, on the slab's device
    const auto face_edges = [&]() -> int
    {
      if (g == 0)
      {
        return VGT_B200_OK;
      }
      cudaStream_t stream = guard.stream;
      const Shared& below = shared[s - 1];
      VGT_CUDA_TRY(below_plane.Allocate(int64_t{plane} * kCellWords, stream),
                   "face cell allocation");
      VGT_CUDA_TRY(below_roots.Allocate(plane, stream), "face root allocation");
      VGT_CUDA_TRY(edges.Allocate(plane, stream), "edge allocation");
      VGT_CUDA_TRY(edge_count.Allocate(1, stream), "edge count allocation");
      VGT_CUDA_TRY(cudaMemcpyAsync(below_plane.get(), below.last_plane.data(),
                                   kCellBytes * plane, cudaMemcpyHostToDevice, stream),
                   "copy face cells to device");
      VGT_CUDA_TRY(cudaMemcpyAsync(below_roots.get(), below.face_roots.data(),
                                   sizeof(uint32_t) * plane, cudaMemcpyHostToDevice, stream),
                   "copy face roots to device");
      const int emitted = FaceEdgesPhase<kCellWords>(below_plane.get(), below_roots.get(),
                                                     slab_base[s - 1], slab, edges.get(),
                                                     edge_count.get(), stream);
      if (emitted != VGT_B200_OK)
      {
        return emitted;
      }
      uint32_t count = 0;
      VGT_CUDA_TRY(cudaMemcpyAsync(&count, edge_count.get(), sizeof(uint32_t),
                                   cudaMemcpyDeviceToHost, stream),
                   "copy edge count");
      VGT_CUDA_TRY(cudaStreamSynchronize(stream), "face edges");
      shared[s].edges.resize(count);
      VGT_CUDA_TRY(cudaMemcpyAsync(shared[s].edges.data(), edges.get(), sizeof(Edge) * count,
                                   cudaMemcpyDeviceToHost, stream),
                   "copy face edges to host");
      VGT_CUDA_TRY(cudaStreamSynchronize(stream), "face edges");
      return VGT_B200_OK;
    };

    // 3. the edges of every face gathered, the face graph resolved (on every slab's device)
    const auto resolve = [&]() -> int
    {
      cudaStream_t stream = guard.stream;
      uint64_t total = 0;
      for (int f = 1; f < num_slabs; f++)
      {
        total += shared[static_cast<size_t>(f)].edges.size();
      }
      const uint32_t num_edges = static_cast<uint32_t>(total);  // <= 7 * 2^26
      const int64_t capacity = std::max<int64_t>(1, 2 * total);
      VGT_CUDA_TRY(all_edges.Allocate(std::max<int64_t>(1, num_edges), stream), "edge allocation");
      VGT_CUDA_TRY(nodes.Allocate(capacity, stream), "node allocation");
      VGT_CUDA_TRY(node_roots.Allocate(capacity, stream), "node root allocation");
      VGT_CUDA_TRY(d_node_words.Allocate(3, stream), "node count allocation");
      uint32_t at = 0;
      for (int f = 1; f < num_slabs; f++)
      {
        const std::vector<Edge>& face = shared[static_cast<size_t>(f)].edges;
        if (!face.empty())
        {
          VGT_CUDA_TRY(cudaMemcpyAsync(all_edges.get() + at, face.data(),
                                       sizeof(Edge) * face.size(), cudaMemcpyHostToDevice, stream),
                       "gather face edges");
        }
        at += static_cast<uint32_t>(face.size());
      }
      const uint64_t range[2] = {slab_base[s], slab_base[s + 1]};
      const int resolved = ResolvePhase(all_edges.get(), num_edges, num_cells, range, 2,
                                        nodes.get(), node_roots.get(), d_node_words.get(), stream);
      if (resolved != VGT_B200_OK)
      {
        return resolved;
      }
      VGT_CUDA_TRY(cudaMemcpyAsync(node_words, d_node_words.get(), sizeof(node_words),
                                   cudaMemcpyDeviceToHost, stream),
                   "copy node count");
      VGT_CUDA_TRY(cudaStreamSynchronize(stream), "face graph");
      graph = SlabNodes{nodes.get(), node_roots.get(), node_words[0], node_words[1],
                        node_words[2] - node_words[1]};
      return VGT_B200_OK;
    };

    // 4. the slab's global roots: bits, their count (count_g)
    const auto count_global_roots = [&]() -> int
    {
      cudaStream_t stream = guard.stream;
      const uint32_t bit_words = RootWords(num_components);
      VGT_CUDA_TRY(bits.Allocate(bit_words, stream), "root bit allocation");
      VGT_CUDA_TRY(bit_prefix.Allocate(int64_t{bit_words} + 1, stream), "root bit prefix allocation");
      const int counted = CountPhase(slab, num_components, graph, bits.get(), bit_prefix.get(),
                                     stream);
      if (counted != VGT_B200_OK)
      {
        return counted;
      }
      uint32_t count = 0;
      VGT_CUDA_TRY(cudaMemcpyAsync(&count, bit_prefix.get() + bit_words, sizeof(uint32_t),
                                   cudaMemcpyDeviceToHost, stream),
                   "copy global root count");
      VGT_CUDA_TRY(cudaStreamSynchronize(stream), "global roots");
      shared[s].num_global_roots = count;
      return VGT_B200_OK;
    };

    // 5. offsets (refused past 0xFFFFFFFF, before any cell is written), the final ids of the
    //    slab's global roots, the ids of its nodes published to the other slabs
    const auto publish = [&]() -> int
    {
      uint64_t total = 0;
      uint64_t offset = 0;
      for (int f = 0; f < num_slabs; f++)
      {
        if (f == g)
        {
          offset = total;
        }
        total += shared[static_cast<size_t>(f)].num_global_roots;
      }
      if (total > 0xFFFFFFFFull)
      {
        SetLastError("connected components: %llu components do not fit the 32-bit component word",
                     static_cast<unsigned long long>(total));
        return VGT_B200_ERR_UNSUPPORTED;
      }
      cudaStream_t stream = guard.stream;
      VGT_CUDA_TRY(final_ids.Allocate(num_components, stream), "final id allocation");
      VGT_CUDA_TRY(node_ids.Allocate(std::max<uint32_t>(1, graph.num_nodes), stream),
                   "node id allocation");
      const int published = PublishPhase(slab, num_components, static_cast<uint32_t>(offset),
                                         graph, bits.get(), bit_prefix.get(), final_ids.get(),
                                         node_ids.get(), stream);
      if (published != VGT_B200_OK)
      {
        return published;
      }
      shared[s].first_node = graph.first;
      shared[s].node_ids.resize(graph.count);
      if (graph.count > 0)
      {
        VGT_CUDA_TRY(cudaMemcpyAsync(shared[s].node_ids.data(), node_ids.get() + graph.first,
                                     sizeof(uint32_t) * graph.count, cudaMemcpyDeviceToHost,
                                     stream),
                     "publish node ids");
      }
      VGT_CUDA_TRY(cudaStreamSynchronize(stream), "node id publication");
      total_components = total;  // (the same sum in every slab)
      return VGT_B200_OK;
    };

    // 6. the published ids of every slab together (their node ranges do not overlap), then the
    //    component word of every cell
    const auto write = [&]() -> int
    {
      cudaStream_t stream = guard.stream;
      std::vector<uint32_t> ids(graph.num_nodes, 0);
      for (const Shared& other : shared)
      {
        std::copy(other.node_ids.begin(), other.node_ids.end(),
                  ids.begin() + other.first_node);
      }
      if (!ids.empty())
      {
        VGT_CUDA_TRY(cudaMemcpyAsync(node_ids.get(), ids.data(), sizeof(uint32_t) * ids.size(),
                                     cudaMemcpyHostToDevice, stream),
                     "copy node ids to device");
      }
      const int written = WritePhase<kCellWords>(slab, graph, node_ids.get(), final_ids.get(),
                                                 stream);
      if (written != VGT_B200_OK)
      {
        return written;
      }
      VGT_CUDA_TRY(cudaStreamSynchronize(stream), "component write");
      return VGT_B200_OK;
    };

    // 7. every slab has written: the cells back
    const auto copy_back = [&]() -> int
    {
      VGT_CUDA_TRY(transfer.ToHost(h_slab, slab_bytes, reinterpret_cast<char*>(d_cells.get()),
                                   slab_bytes, slab_bytes, 1, guard.stream),
                   "copy cell slab to host");
      VGT_CUDA_TRY(cudaStreamSynchronize(guard.stream), "cell copy");
      return VGT_B200_OK;
    };

    // Every thread passes every barrier; after the first failure (here or in another slab) the
    // remaining phases are skipped.
    int status = VGT_B200_OK;
    const std::function<int()> phases[] = {local_labelling, face_edges, resolve,
                                           count_global_roots, publish, write, copy_back};
    for (const auto& phase : phases)
    {
      if (status == VGT_B200_OK && failed.load() != 0)
      {
        status = VGT_B200_ERR_DEVICE;
        messages[s] = kStoodDown;
      }
      if (status == VGT_B200_OK)
      {
        status = phase();
        if (status != VGT_B200_OK)
        {
          messages[s] = vgt_b200_last_error();  // thread-local text
          failed.store(1);
        }
      }
      barrier.Wait();
    }
    statuses[s] = status;
  };

  std::vector<std::thread> threads;
  for (int g = 1; g < num_slabs; g++)
  {
    threads.emplace_back(worker, g);
  }
  worker(0);
  for (auto& thread : threads)
  {
    thread.join();
  }
  // the slab that failed first-hand, not the ones that stood down because of it
  for (const bool first_hand : {true, false})
  {
    for (int g = 0; g < num_slabs; g++)
    {
      const size_t s = static_cast<size_t>(g);
      const bool stood_down = messages[s] == kStoodDown;
      if (statuses[s] != VGT_B200_OK && stood_down != first_hand)
      {
        SetLastError("slab %d (device %d): %s", g, devices[g], messages[s].c_str());
        return statuses[s];
      }
    }
  }
  *out_num_components = static_cast<uint32_t>(total_components);
  return VGT_B200_OK;
}

// ---- checks of the per-slab entries (vgt_b200_components_*), before any device call ---------
int CheckSlab(int cell_bytes, int64_t nx, int64_t ny, int64_t nz, Grid* grid)
{
  if (cell_bytes != 8 && cell_bytes != 16)
  {
    return FailInvalid("cell size must be 8 (OccupancyComponentCell) or 16 "
                       "(TaggedObjectOccupancyComponentCell) bytes");
  }
  if (!ValidDims(nx, ny, nz))
  {
    return FailInvalid("slab dimensions %lld x %lld x %lld out of range (a slab has at least one "
                       "x-plane)", static_cast<long long>(nx), static_cast<long long>(ny),
                       static_cast<long long>(nz));
  }
  const int64_t count = nx * ny * nz;
  if (count >= (int64_t{1} << 32))
  {
    SetLastError("connected components: slabs of 2^32 cells or more are not supported "
                 "(%lld cells)", static_cast<long long>(count));
    return VGT_B200_ERR_UNSUPPORTED;
  }
  *grid = Grid{static_cast<uint32_t>(nx), static_cast<uint32_t>(ny), static_cast<uint32_t>(nz),
               static_cast<uint32_t>(count)};
  return VGT_B200_OK;
}

int CheckPointers(std::initializer_list<std::pair<const void*, const char*>> pointers)
{
  for (const auto& pointer : pointers)
  {
    if (pointer.first == nullptr)
    {
      return FailInvalid("null %s", pointer.second);
    }
  }
  return VGT_B200_OK;
}

// The slab's arrays and its share of the face graph, checked.
int CheckSlabState(int64_t nx, int64_t ny, int64_t nz, int64_t base, int64_t num_components,
                   int64_t num_nodes, int64_t first_node, int64_t num_slab_nodes, Grid* grid)
{
  const int checked = CheckSlab(8, nx, ny, nz, grid);
  if (checked != VGT_B200_OK)
  {
    return checked;
  }
  if (base < 0 || base > (int64_t{1} << 62))
  {
    return FailInvalid("slab base %lld out of range", static_cast<long long>(base));
  }
  if (num_components < 1 || num_components > grid->count)
  {
    return FailInvalid("%lld local components in a slab of %u cells",
                       static_cast<long long>(num_components), grid->count);
  }
  if (num_nodes < 0 || num_nodes > 0xFFFFFFFFll || first_node < 0 || num_slab_nodes < 0
      || first_node + num_slab_nodes > num_nodes)
  {
    return FailInvalid("node range [%lld, %lld) outside the %lld nodes",
                       static_cast<long long>(first_node),
                       static_cast<long long>(first_node + num_slab_nodes),
                       static_cast<long long>(num_nodes));
  }
  return VGT_B200_OK;
}
}  // namespace
}  // namespace components
}  // namespace vgt_b200

using namespace vgt_b200;
using namespace vgt_b200::components;

extern "C"
{
int vgt_b200_connected_components_dev(void* d_cells, int cell_bytes, int64_t nx, int64_t ny,
                                      int64_t nz, int device, uint32_t* d_num_components,
                                      void* stream)
{
  Grid grid;
  const int check = CheckArguments(d_cells, cell_bytes, nx, ny, nz, d_num_components, &grid);
  if (check != VGT_B200_OK)
  {
    return check;
  }
  if ((reinterpret_cast<uintptr_t>(d_cells) & 3u) != 0)
  {
    return FailInvalid("cell array must be 4-byte aligned");
  }
  ScopedDevice scoped(device);
  VGT_CUDA_TRY(scoped.Status(), "cudaSetDevice");
  KeepPoolMemory(device);
  return Launch(d_cells, cell_bytes, grid, d_num_components, static_cast<cudaStream_t>(stream));
}

int vgt_b200_connected_components(void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz,
                                  int device, uint32_t* out_num_components)
{
  Grid grid;
  const int check = CheckArguments(cells, cell_bytes, nx, ny, nz, out_num_components, &grid);
  if (check != VGT_B200_OK)
  {
    return check;
  }
  ScopedDevice scoped(device);
  VGT_CUDA_TRY(scoped.Status(), "cudaSetDevice");
  KeepPoolMemory(device);
  cudaStream_t stream = nullptr;
  VGT_CUDA_TRY(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking), "cudaStreamCreate");
  struct StreamOwner
  {
    cudaStream_t stream;
    ~StreamOwner()
    {
      cudaStreamSynchronize(stream);
      cudaStreamDestroy(stream);
    }
  } owner{stream};
  const size_t grid_bytes = static_cast<size_t>(grid.count) * static_cast<size_t>(cell_bytes);
  uint32_t num_components = 0;
  {
    // (declared inside the stream owner's scope: freed on the stream before it is destroyed)
    StreamScratch<char> d_cells;
    StreamScratch<uint32_t> d_num_components;
    VGT_CUDA_TRY(d_cells.Allocate(static_cast<int64_t>(grid_bytes), stream), "cell allocation");
    VGT_CUDA_TRY(d_num_components.Allocate(1, stream), "count allocation");
    // Whole cells go both ways (no gather / scatter of the component words on the host).
    StagedTransfer transfer;
    VGT_CUDA_TRY(transfer.ToDevice(d_cells.get(), grid_bytes, static_cast<const char*>(cells),
                                   grid_bytes, grid_bytes, 1, stream),
                 "copy cells to device");
    const int launched = Launch(d_cells.get(), cell_bytes, grid, d_num_components.get(), stream);
    if (launched != VGT_B200_OK)
    {
      cudaStreamSynchronize(stream);
      return launched;
    }
    VGT_CUDA_TRY(cudaMemcpyAsync(&num_components, d_num_components.get(), sizeof(uint32_t),
                                 cudaMemcpyDeviceToHost, stream),
                 "copy component count to host");
    VGT_CUDA_TRY(transfer.ToHost(static_cast<char*>(cells), grid_bytes, d_cells.get(), grid_bytes,
                                 grid_bytes, 1, stream),
                 "copy cells to host");
    VGT_CUDA_TRY(cudaStreamSynchronize(stream), "connected components");
  }
  *out_num_components = num_components;
  return VGT_B200_OK;
}

int vgt_b200_connected_components_multi(void* cells, int cell_bytes, int64_t nx, int64_t ny,
                                        int64_t nz, const int* devices, int num_slabs,
                                        uint32_t* out_num_components)
{
  const int check = CheckMultiArguments(cells, cell_bytes, nx, ny, nz, devices, num_slabs,
                                        out_num_components);
  if (check != VGT_B200_OK)
  {
    return check;
  }
  if (num_slabs == 1)
  {
    return vgt_b200_connected_components(cells, cell_bytes, nx, ny, nz, devices[0],
                                         out_num_components);
  }
  if (cell_bytes == 8)
  {
    return ConnectedComponentsSlabs<2>(static_cast<char*>(cells), nx, ny, nz, devices, num_slabs,
                                       out_num_components);
  }
  return ConnectedComponentsSlabs<4>(static_cast<char*>(cells), nx, ny, nz, devices, num_slabs,
                                     out_num_components);
}

int vgt_b200_components_slab_scan_bytes(int64_t nx, int64_t ny, int64_t nz, int device,
                                        size_t* out_bytes)
{
  Grid grid;
  const int check = CheckSlab(8, nx, ny, nz, &grid);
  if (check != VGT_B200_OK)
  {
    return check;
  }
  const int pointers = CheckPointers({{out_bytes, "scan size"}});
  if (pointers != VGT_B200_OK)
  {
    return pointers;
  }
  ScopedDevice scoped(device);
  VGT_CUDA_TRY(scoped.Status(), "cudaSetDevice");
  return ScanBytes(grid.count, out_bytes);
}

int vgt_b200_components_slab_local(void* d_cells, int cell_bytes, int64_t nx, int64_t ny,
                                   int64_t nz, int device, uint32_t* d_parent, uint32_t* d_mask,
                                   uint32_t* d_word_prefix, void* d_scan_storage,
                                   size_t scan_bytes, uint32_t* d_face_roots, void* stream)
{
  Grid grid;
  int check = CheckSlab(cell_bytes, nx, ny, nz, &grid);
  if (check == VGT_B200_OK)
  {
    check = CheckPointers({{d_cells, "cell array"}, {d_parent, "parent array"},
                           {d_mask, "root mask"}, {d_word_prefix, "word prefix"},
                           {d_scan_storage, "scan storage"}});
  }
  if (check != VGT_B200_OK)
  {
    return check;
  }
  ScopedDevice scoped(device);
  VGT_CUDA_TRY(scoped.Status(), "cudaSetDevice");
  const SlabArrays slab{grid, 0, static_cast<uint32_t*>(d_cells), d_parent, d_mask,
                        d_word_prefix, d_scan_storage, scan_bytes};
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  return cell_bytes == 8 ? LocalPhase<2>(slab, d_face_roots, s)
                         : LocalPhase<4>(slab, d_face_roots, s);
}

int vgt_b200_components_slab_face_edges(const void* d_below_cells, const uint32_t* d_below_roots,
                                        int64_t below_base, void* d_cells, int cell_bytes,
                                        int64_t nx, int64_t ny, int64_t nz, int64_t base,
                                        int device, uint32_t* d_parent, int64_t* d_edges,
                                        uint32_t* d_edge_count, void* stream)
{
  Grid grid;
  int check = CheckSlab(cell_bytes, nx, ny, nz, &grid);
  if (check == VGT_B200_OK)
  {
    check = CheckPointers({{d_below_cells, "face cell array"}, {d_below_roots, "face roots"},
                           {d_cells, "cell array"}, {d_parent, "parent array"},
                           {d_edges, "edge array"}, {d_edge_count, "edge count"}});
  }
  if (check != VGT_B200_OK)
  {
    return check;
  }
  if (below_base < 0 || base < below_base + ny * nz)
  {
    return FailInvalid("slab bases %lld (below) and %lld out of order",
                       static_cast<long long>(below_base), static_cast<long long>(base));
  }
  ScopedDevice scoped(device);
  VGT_CUDA_TRY(scoped.Status(), "cudaSetDevice");
  const SlabArrays slab{grid, static_cast<uint64_t>(base), static_cast<uint32_t*>(d_cells),
                        d_parent, nullptr, nullptr, nullptr, 0};
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  const uint32_t* below = static_cast<const uint32_t*>(d_below_cells);
  Edge* edges = reinterpret_cast<Edge*>(d_edges);
  return cell_bytes == 8
             ? FaceEdgesPhase<2>(below, d_below_roots, static_cast<uint64_t>(below_base), slab,
                                 edges, d_edge_count, s)
             : FaceEdgesPhase<4>(below, d_below_roots, static_cast<uint64_t>(below_base), slab,
                                 edges, d_edge_count, s);
}

int vgt_b200_components_resolve(const int64_t* d_edges, int64_t num_edges, int64_t num_cells,
                                int64_t base, int64_t end, int device, int64_t* d_nodes,
                                uint32_t* d_node_roots, uint32_t* d_node_range, void* stream)
{
  int check = CheckPointers({{d_nodes, "node array"}, {d_node_roots, "node roots"},
                             {d_node_range, "node range"}});
  if (check != VGT_B200_OK)
  {
    return check;
  }
  if (num_edges < 0 || num_edges > (int64_t{1} << 30) || (num_edges > 0 && d_edges == nullptr))
  {
    return FailInvalid("%lld edges (at most 2^30, and a null edge array only without edges)",
                       static_cast<long long>(num_edges));
  }
  if (num_cells < 1 || base < 0 || end <= base || end > num_cells)
  {
    return FailInvalid("slab [%lld, %lld) outside a map of %lld cells",
                       static_cast<long long>(base), static_cast<long long>(end),
                       static_cast<long long>(num_cells));
  }
  ScopedDevice scoped(device);
  VGT_CUDA_TRY(scoped.Status(), "cudaSetDevice");
  KeepPoolMemory(device);
  const uint64_t range[2] = {static_cast<uint64_t>(base), static_cast<uint64_t>(end)};
  return ResolvePhase(reinterpret_cast<const Edge*>(d_edges), static_cast<uint32_t>(num_edges),
                      static_cast<uint64_t>(num_cells), range, 2,
                      reinterpret_cast<uint64_t*>(d_nodes), d_node_roots, d_node_range,
                      static_cast<cudaStream_t>(stream));
}

int vgt_b200_components_slab_count(int64_t nx, int64_t ny, int64_t nz, int64_t base,
                                   int64_t num_components, int device, const uint32_t* d_mask,
                                   const uint32_t* d_word_prefix, const int64_t* d_nodes,
                                   const uint32_t* d_node_roots, int64_t num_nodes,
                                   int64_t first_node, int64_t num_slab_nodes, uint32_t* d_bits,
                                   uint32_t* d_bit_prefix, void* d_scan_storage,
                                   size_t scan_bytes, void* stream)
{
  Grid grid;
  int check = CheckSlabState(nx, ny, nz, base, num_components, num_nodes, first_node,
                             num_slab_nodes, &grid);
  if (check == VGT_B200_OK)
  {
    check = CheckPointers({{d_mask, "root mask"}, {d_word_prefix, "word prefix"},
                           {d_bits, "root bits"}, {d_bit_prefix, "root bit prefix"},
                           {d_scan_storage, "scan storage"}});
  }
  if (check == VGT_B200_OK && num_slab_nodes > 0)
  {
    check = CheckPointers({{d_nodes, "node array"}, {d_node_roots, "node roots"}});
  }
  if (check != VGT_B200_OK)
  {
    return check;
  }
  ScopedDevice scoped(device);
  VGT_CUDA_TRY(scoped.Status(), "cudaSetDevice");
  const SlabArrays slab{grid, static_cast<uint64_t>(base), nullptr, nullptr,
                        const_cast<uint32_t*>(d_mask), const_cast<uint32_t*>(d_word_prefix),
                        d_scan_storage, scan_bytes};
  const SlabNodes graph{reinterpret_cast<const uint64_t*>(d_nodes), d_node_roots,
                        static_cast<uint32_t>(num_nodes), static_cast<uint32_t>(first_node),
                        static_cast<uint32_t>(num_slab_nodes)};
  return CountPhase(slab, static_cast<uint32_t>(num_components), graph, d_bits, d_bit_prefix,
                    static_cast<cudaStream_t>(stream));
}

int vgt_b200_components_slab_publish(int64_t nx, int64_t ny, int64_t nz, int64_t base,
                                     int64_t num_components, int64_t offset, int device,
                                     const uint32_t* d_mask, const uint32_t* d_word_prefix,
                                     const int64_t* d_nodes, int64_t num_nodes,
                                     int64_t first_node, int64_t num_slab_nodes,
                                     const uint32_t* d_bits, const uint32_t* d_bit_prefix,
                                     uint32_t* d_final_ids, uint32_t* d_node_ids, void* stream)
{
  Grid grid;
  int check = CheckSlabState(nx, ny, nz, base, num_components, num_nodes, first_node,
                             num_slab_nodes, &grid);
  if (check == VGT_B200_OK)
  {
    check = CheckPointers({{d_mask, "root mask"}, {d_word_prefix, "word prefix"},
                           {d_bits, "root bits"}, {d_bit_prefix, "root bit prefix"},
                           {d_final_ids, "final id array"}});
  }
  if (check == VGT_B200_OK && num_slab_nodes > 0)
  {
    check = CheckPointers({{d_nodes, "node array"}, {d_node_ids, "node id array"}});
  }
  if (check != VGT_B200_OK)
  {
    return check;
  }
  if (offset < 0 || offset > 0xFFFFFFFFll)
  {
    return FailInvalid("component offset %lld out of range", static_cast<long long>(offset));
  }
  ScopedDevice scoped(device);
  VGT_CUDA_TRY(scoped.Status(), "cudaSetDevice");
  const SlabArrays slab{grid, static_cast<uint64_t>(base), nullptr, nullptr,
                        const_cast<uint32_t*>(d_mask), const_cast<uint32_t*>(d_word_prefix),
                        nullptr, 0};
  const SlabNodes graph{reinterpret_cast<const uint64_t*>(d_nodes), nullptr,
                        static_cast<uint32_t>(num_nodes), static_cast<uint32_t>(first_node),
                        static_cast<uint32_t>(num_slab_nodes)};
  return PublishPhase(slab, static_cast<uint32_t>(num_components), static_cast<uint32_t>(offset),
                      graph, d_bits, d_bit_prefix, d_final_ids, d_node_ids,
                      static_cast<cudaStream_t>(stream));
}

int vgt_b200_components_slab_write(void* d_cells, int cell_bytes, int64_t nx, int64_t ny,
                                   int64_t nz, int64_t base, int64_t num_components, int device,
                                   uint32_t* d_parent, const uint32_t* d_mask,
                                   const uint32_t* d_word_prefix, const int64_t* d_nodes,
                                   const uint32_t* d_node_roots, int64_t num_nodes,
                                   int64_t first_node, int64_t num_slab_nodes,
                                   uint32_t* d_node_ids, uint32_t* d_final_ids, void* stream)
{
  Grid grid;
  int check = CheckSlab(cell_bytes, nx, ny, nz, &grid);
  if (check == VGT_B200_OK)
  {
    check = CheckSlabState(nx, ny, nz, base, num_components, num_nodes, first_node,
                           num_slab_nodes, &grid);
  }
  if (check == VGT_B200_OK)
  {
    check = CheckPointers({{d_cells, "cell array"}, {d_parent, "parent array"},
                           {d_mask, "root mask"}, {d_word_prefix, "word prefix"},
                           {d_final_ids, "final id array"}});
  }
  if (check == VGT_B200_OK && num_nodes > 0)
  {
    check = CheckPointers({{d_nodes, "node array"}, {d_node_roots, "node roots"},
                           {d_node_ids, "node id array"}});
  }
  if (check != VGT_B200_OK)
  {
    return check;
  }
  ScopedDevice scoped(device);
  VGT_CUDA_TRY(scoped.Status(), "cudaSetDevice");
  const SlabArrays slab{grid, static_cast<uint64_t>(base), static_cast<uint32_t*>(d_cells),
                        d_parent, const_cast<uint32_t*>(d_mask),
                        const_cast<uint32_t*>(d_word_prefix), nullptr, 0};
  const SlabNodes graph{reinterpret_cast<const uint64_t*>(d_nodes), d_node_roots,
                        static_cast<uint32_t>(num_nodes), static_cast<uint32_t>(first_node),
                        static_cast<uint32_t>(num_slab_nodes)};
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  return cell_bytes == 8 ? WritePhase<2>(slab, graph, d_node_ids, d_final_ids, s)
                         : WritePhase<4>(slab, graph, d_node_ids, d_final_ids, s);
}
}  // extern "C"
