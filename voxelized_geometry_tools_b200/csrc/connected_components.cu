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
#include <cub/device/device_scan.cuh>

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
}  // extern "C"
