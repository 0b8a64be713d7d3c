// Occupancy cells of the other map types -> filled mask, and the merge of the "free" and "named
// objects" fields (sm_100a). Included by edt_kernels.cu.
//
// The reference's other three map types store 8- or 16-byte cells
//   OccupancyComponentCell             { float occupancy; uint32 component; }
//     (include/voxelized_geometry_tools/occupancy_component_map.hpp:28-64)
//   TaggedObjectOccupancyCell          { float occupancy; uint32 object_id; }
//     (include/.../tagged_object_occupancy_map.hpp:28-68)
//   TaggedObjectOccupancyComponentCell { float occupancy; uint32 object_id; uint32 component;
//                                        uint32 spatial_segment; }
//     (include/.../tagged_object_occupancy_component_map.hpp:17-60)
// and their ExtractSignedDistanceField differs from OccupancyMap's only in the filled predicate
// (occupancy_component_map.hpp:270-306, tagged_object_occupancy_map.hpp:199-247,
// tagged_object_occupancy_component_map.hpp:360-410). The predicate is evaluated here, on the
// device, straight from the raw cell array (read once, 1 byte per voxel out); the mask then
// takes the same three passes as every other grid.
#pragma once

#include <cstdint>

#include "edt_device.cuh"

namespace vgt_b200
{
namespace edt
{
namespace
{
// What a cell must satisfy, besides the occupancy rule, to count as filled.
enum ObjectRule
{
  kAnyObject = 0,     // no object restriction (objects_to_use empty / maps without object ids)
  kListedObjects = 1, // object_id in the sorted list (tagged_object_occupancy_map.hpp:219-222)
  kNamedObjects = 2   // object_id > 0 (tagged_object_occupancy_map.hpp:321-324)
};

// cells: raw array of `cell_words` 32-bit words per voxel; word 0 = occupancy (float), word 1 =
// object id (only read for the object rules). sorted_ids: ascending, num_ids entries.
__global__ void CellsToMaskKernel(const uint32_t* __restrict__ cells, int cell_words,
                                  int64_t count, int unknown_is_filled, int object_rule,
                                  const uint32_t* __restrict__ sorted_ids, int num_ids,
                                  uint8_t* __restrict__ mask)
{
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= count)
  {
    return;
  }
  const uint32_t* cell = cells + i * cell_words;
  bool filled = IsFilled(__uint_as_float(__ldcs(cell)), unknown_is_filled);
  if (filled && object_rule != kAnyObject)
  {
    const uint32_t object_id = __ldcs(cell + 1);
    if (object_rule == kNamedObjects)
    {
      filled = object_id > 0u;
    }
    else
    {
      int low = 0;
      int high = num_ids;
      while (low < high)
      {
        const int middle = (low + high) >> 1;
        if (__ldg(sorted_ids + middle) < object_id)
        {
          low = middle + 1;
        }
        else
        {
          high = middle;
        }
      }
      filled = (low < num_ids) && (__ldg(sorted_ids + low) == object_id);
    }
  }
  mask[i] = filled ? 1 : 0;
}

// The per-object batch on device cells (MakeSeparateObjectSDFs, tagged_object_occupancy_map.hpp:
// 249-262) classifies the cells once per group of at most kSlotGroupSize distinct object ids into
// a 1-byte slot map; SDF k of the batch then takes the three passes on "slot == key of object k".
// Slot 0 is "not filled, or an object outside the group", so one byte tells 255 ids apart.
constexpr int kSlotGroupSize = 255;

// A kernel parameter (1 KB), so the host's id list needs no device copy.
struct SlotGroup
{
  uint32_t ids[kSlotGroupSize];  // ascending, distinct
  int count;
};

// slots[i] = 0 when the occupancy rule fails or cell i's object id (word 1) is not in the group,
// else 1 + the id's position in group.ids. Grid-stride over a fixed grid, so that the copy of the
// group into shared memory is paid per resident block, not per 256 voxels; four voxels per thread
// and round, their loads issued before any is used.
__global__ void __launch_bounds__(256) CellsToObjectSlotsKernel(
    const uint32_t* __restrict__ cells, int cell_words, int64_t count, int unknown_is_filled,
    const SlotGroup group, uint8_t* __restrict__ slots)
{
  constexpr int kPerThread = 4;
  __shared__ uint32_t ids[kSlotGroupSize];
  for (int j = threadIdx.x; j < group.count; j += blockDim.x)
  {
    ids[j] = group.ids[j];
  }
  __syncthreads();
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x * kPerThread;
  for (int64_t base = static_cast<int64_t>(blockIdx.x) * blockDim.x * kPerThread + threadIdx.x;
       base < count; base += stride)
  {
    uint32_t occupancy[kPerThread];
    uint32_t object_id[kPerThread];
#pragma unroll
    for (int j = 0; j < kPerThread; j++)
    {
      const int64_t i = base + static_cast<int64_t>(j) * blockDim.x;
      if (i < count)
      {
        occupancy[j] = __ldcs(cells + i * cell_words);
        object_id[j] = __ldcs(cells + i * cell_words + 1);
      }
    }
#pragma unroll
    for (int j = 0; j < kPerThread; j++)
    {
      const int64_t i = base + static_cast<int64_t>(j) * blockDim.x;
      if (i >= count)
      {
        break;
      }
      uint8_t slot = 0;
      if (IsFilled(__uint_as_float(occupancy[j]), unknown_is_filled))
      {
        int low = 0;
        int high = group.count;
        while (low < high)
        {
          const int middle = (low + high) >> 1;
          if (ids[middle] < object_id[j])
          {
            low = middle + 1;
          }
          else
          {
            high = middle;
          }
        }
        if (low < group.count && ids[low] == object_id[j])
        {
          slot = static_cast<uint8_t>(low + 1);
        }
      }
      slots[i] = slot;
    }
  }
}

// A byte of the slot map as the input of the scalar z scan: filled iff the slot equals the key of
// the object whose SDF is computed, which the scans take where occupancy inputs take
// unknown_is_filled.
struct ObjectSlot
{
  uint8_t slot;
};

__device__ __forceinline__ bool IsFilled(ObjectSlot cell, int key) { return cell.slot == key; }

__device__ __forceinline__ ObjectSlot LoadStreaming(const ObjectSlot* p)
{
  return ObjectSlot{__ldcs(reinterpret_cast<const uint8_t*>(p))};
}

// The same test four slots at a time, for the register and Vec4 scans.
struct SlotEquals4Source
{
  using Vector = uchar4;
  __device__ static __forceinline__ uint32_t Nibble(const uchar4& v, int key)
  {
    return (v.x == key ? 1u : 0u) | (v.y == key ? 2u : 0u) | (v.z == key ? 4u : 0u)
        | (v.w == key ? 8u : 0u);
  }
};

// ExtractFreeAndNamedObjectsSignedDistanceField's merge (tagged_object_occupancy_map.hpp:344-369):
//   free >= 0 -> free;  else named <= -0 -> named;  else 0.   Then Lock()'s min/max.
// Grid-stride: a fixed grid, so the min/max atomics are two per warp of the grid, not two per
// 32 voxels (all to the same two addresses, which the L2 serialises).
template <typename Out, typename Key>
__global__ void MergeFreeAndNamedKernel(const Out* __restrict__ free_sdf,
                                        const Out* __restrict__ named_sdf, int64_t count,
                                        Out* __restrict__ combined, Key* min_max_keys)
{
  Out low = PositiveInfinity<Out>();
  Out high = -PositiveInfinity<Out>();
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < count;
       i += stride)
  {
    const Out free_value = free_sdf[i];
    const Out named_value = named_sdf[i];
    const Out value =
        (free_value >= Out(0)) ? free_value : ((named_value <= Out(0)) ? named_value : Out(0));
    combined[i] = value;
    low = (value < low) ? value : low;
    high = (value > high) ? value : high;
  }
  Key key_min = OrderedKey(low);
  Key key_max = OrderedKey(high);
#pragma unroll
  for (int offset = 16; offset > 0; offset >>= 1)
  {
    const Key other_min = __shfl_xor_sync(0xffffffffu, key_min, offset);
    const Key other_max = __shfl_xor_sync(0xffffffffu, key_max, offset);
    key_min = (other_min < key_min) ? other_min : key_min;
    key_max = (other_max > key_max) ? other_max : key_max;
  }
  if ((threadIdx.x & 31) == 0 && min_max_keys != nullptr)
  {
    atomicMin(min_max_keys + 0, key_min);
    atomicMax(min_max_keys + 1, key_max);
  }
}
}  // namespace
}  // namespace edt
}  // namespace vgt_b200
