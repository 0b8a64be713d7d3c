// C++ host adapter for the reference's three cell-map types: the packed 8- / 16-byte cells go to
// the device as they are and the filled predicate runs there (vgt_b200_sdf_from_cells_*,
// vgt_b200_sdf_per_object_*, vgt_b200_sdf_free_and_named_* in include/vgt_b200.h).
//
// Same names, argument meaning and results as the member templates they stand in for:
//   OccupancyComponentMap::ExtractSignedDistanceField<T>(parameters)
//       include/voxelized_geometry_tools/occupancy_component_map.hpp:270-306
//   TaggedObjectOccupancyMap::ExtractSignedDistanceField<T>(objects_to_use, parameters)
//   TaggedObjectOccupancyMap::MakeSeparateObjectSDFs<T> / MakeAllObjectSDFs<T>
//   TaggedObjectOccupancyMap::ExtractFreeAndNamedObjectsSignedDistanceField<T>(parameters)
//       include/voxelized_geometry_tools/tagged_object_occupancy_map.hpp:199-378
//   and the same four on TaggedObjectOccupancyComponentMap
//       include/voxelized_geometry_tools/tagged_object_occupancy_component_map.hpp:360-575
// as free functions taking the map, in namespace ...::signed_distance_field_generation::b200
// (a maintainer replaces the member bodies by calls to these, INTEGRATION.md section 2).
#pragma once

#include <cstdint>
#include <map>
#include <set>
#include <stdexcept>
#include <string>
#include <vector>

#include <voxelized_geometry_tools/signed_distance_field.hpp>
#include <voxelized_geometry_tools/vgt_namespace.hpp>

#include "b200_signed_distance_field_generation.hpp"
#include "vgt_b200.h"

namespace voxelized_geometry_tools
{
VGT_NAMESPACE_BEGIN
namespace signed_distance_field_generation
{
namespace b200
{
namespace detail
{
// (float / double overloads over the C-ABI pairs; `int device` or a device list)
inline int CallCells(const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz,
                     double resolution, bool unknown_is_filled, bool border,
                     const uint32_t* ids, int64_t num_ids, int device, float* out, float* lo,
                     float* hi)
{
  return vgt_b200_sdf_from_cells_f32(cells, cell_bytes, nx, ny, nz, resolution,
                                     unknown_is_filled ? 1 : 0, border ? 1 : 0, ids, num_ids,
                                     device, out, lo, hi);
}
inline int CallCells(const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz,
                     double resolution, bool unknown_is_filled, bool border,
                     const uint32_t* ids, int64_t num_ids, int device, double* out, double* lo,
                     double* hi)
{
  return vgt_b200_sdf_from_cells_f64(cells, cell_bytes, nx, ny, nz, resolution,
                                     unknown_is_filled ? 1 : 0, border ? 1 : 0, ids, num_ids,
                                     device, out, lo, hi);
}
inline int CallPerObject(const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz,
                         double resolution, bool unknown_is_filled, bool border,
                         const uint32_t* ids, int64_t num_ids, int device, float* out, float* lo,
                         float* hi)
{
  return vgt_b200_sdf_per_object_f32(cells, cell_bytes, nx, ny, nz, resolution,
                                     unknown_is_filled ? 1 : 0, border ? 1 : 0, ids, num_ids,
                                     device, out, lo, hi);
}
inline int CallPerObject(const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz,
                         double resolution, bool unknown_is_filled, bool border,
                         const uint32_t* ids, int64_t num_ids, int device, double* out,
                         double* lo, double* hi)
{
  return vgt_b200_sdf_per_object_f64(cells, cell_bytes, nx, ny, nz, resolution,
                                     unknown_is_filled ? 1 : 0, border ? 1 : 0, ids, num_ids,
                                     device, out, lo, hi);
}
inline int CallFreeAndNamed(const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz,
                            double resolution, bool unknown_is_filled, bool border, int device,
                            float* out, float* lo, float* hi)
{
  return vgt_b200_sdf_free_and_named_f32(cells, cell_bytes, nx, ny, nz, resolution,
                                         unknown_is_filled ? 1 : 0, border ? 1 : 0, device, out,
                                         lo, hi);
}
inline int CallFreeAndNamed(const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz,
                            double resolution, bool unknown_is_filled, bool border, int device,
                            double* out, double* lo, double* hi)
{
  return vgt_b200_sdf_free_and_named_f64(cells, cell_bytes, nx, ny, nz, resolution,
                                         unknown_is_filled ? 1 : 0, border ? 1 : 0, device, out,
                                         lo, hi);
}
// the same over the multi-device entries, the device list in place of `device`
inline int CallCells(const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz,
                     double resolution, bool unknown_is_filled, bool border,
                     const uint32_t* ids, int64_t num_ids, const std::vector<int>& devices,
                     float* out, float* lo, float* hi)
{
  return vgt_b200_sdf_from_cells_f32_multi(
      cells, cell_bytes, nx, ny, nz, resolution, unknown_is_filled ? 1 : 0, border ? 1 : 0,
      ids, num_ids, devices.data(), static_cast<int>(devices.size()), out, lo, hi);
}
inline int CallCells(const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz,
                     double resolution, bool unknown_is_filled, bool border,
                     const uint32_t* ids, int64_t num_ids, const std::vector<int>& devices,
                     double* out, double* lo, double* hi)
{
  return vgt_b200_sdf_from_cells_f64_multi(
      cells, cell_bytes, nx, ny, nz, resolution, unknown_is_filled ? 1 : 0, border ? 1 : 0,
      ids, num_ids, devices.data(), static_cast<int>(devices.size()), out, lo, hi);
}
inline int CallPerObject(const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz,
                         double resolution, bool unknown_is_filled, bool border,
                         const uint32_t* ids, int64_t num_ids, const std::vector<int>& devices,
                         float* out, float* lo, float* hi)
{
  return vgt_b200_sdf_per_object_f32_multi(
      cells, cell_bytes, nx, ny, nz, resolution, unknown_is_filled ? 1 : 0, border ? 1 : 0,
      ids, num_ids, devices.data(), static_cast<int>(devices.size()), out, lo, hi);
}
inline int CallPerObject(const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz,
                         double resolution, bool unknown_is_filled, bool border,
                         const uint32_t* ids, int64_t num_ids, const std::vector<int>& devices,
                         double* out, double* lo, double* hi)
{
  return vgt_b200_sdf_per_object_f64_multi(
      cells, cell_bytes, nx, ny, nz, resolution, unknown_is_filled ? 1 : 0, border ? 1 : 0,
      ids, num_ids, devices.data(), static_cast<int>(devices.size()), out, lo, hi);
}
inline int CallFreeAndNamed(const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz,
                            double resolution, bool unknown_is_filled, bool border,
                            const std::vector<int>& devices,
                            float* out, float* lo, float* hi)
{
  return vgt_b200_sdf_free_and_named_f32_multi(
      cells, cell_bytes, nx, ny, nz, resolution, unknown_is_filled ? 1 : 0, border ? 1 : 0,
      devices.data(), static_cast<int>(devices.size()), out, lo, hi);
}
inline int CallFreeAndNamed(const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz,
                            double resolution, bool unknown_is_filled, bool border,
                            const std::vector<int>& devices,
                            double* out, double* lo, double* hi)
{
  return vgt_b200_sdf_free_and_named_f64_multi(
      cells, cell_bytes, nx, ny, nz, resolution, unknown_is_filled ? 1 : 0, border ? 1 : 0,
      devices.data(), static_cast<int>(devices.size()), out, lo, hi);
}

template <typename MapType>
struct CellsOf
{
  using Cell = typename std::remove_reference<
      decltype(std::declval<const MapType&>().GetImmutableRawData())>::type::value_type;
  static_assert(sizeof(Cell) == 8 || sizeof(Cell) == 16,
                "cells are {float occupancy; uint32 id-or-component; ...} of 8 or 16 bytes "
                "(the reference pins both sizes with static_asserts)");
  static constexpr int kBytes = static_cast<int>(sizeof(Cell));
};

template <typename MapType>
inline void RequireUniform(const MapType& map)
{
  if (!map.HasUniformVoxelSize())
  {
    throw std::invalid_argument("Grid must have uniform resolution");  // sdfgen.hpp:123-126
  }
}

template <typename ScalarType>
inline void FinishSdf(SignedDistanceField<ScalarType>& sdf, ScalarType minimum, ScalarType maximum)
{
  FinishAndLock(sdf, minimum, maximum);
}
}  // namespace detail

// ExtractSignedDistanceField<T>(objects_to_use, parameters) of the tagged maps; with an empty
// list (or for OccupancyComponentMap, which has no object ids) every filled cell counts.
// `device` of each function below: one ordinal (int), or a std::vector<int> of several, which
// cuts the map into one x-slab per device (the *_multi entries) for maps one device cannot
// hold, with the same result.
template <typename MapType, typename ScalarType, typename Devices = int>
inline SignedDistanceField<ScalarType> ExtractSignedDistanceFieldFromCellMap(
    const MapType& map, const std::vector<uint32_t>& objects_to_use,
    const SignedDistanceFieldGenerationParameters<ScalarType>& parameters,
    const Devices& device = 0)
{
  detail::RequireUniform(map);
  SignedDistanceField<ScalarType> sdf(map.OriginTransform(), map.Frame(), map.ControlSizes(),
                                      parameters.OOBValue());
  ScalarType minimum = 0;
  ScalarType maximum = 0;
  ThrowOnError(detail::CallCells(
      map.GetImmutableRawData().data(), detail::CellsOf<MapType>::kBytes, map.NumXVoxels(),
      map.NumYVoxels(), map.NumZVoxels(), map.VoxelXSize(), parameters.UnknownIsFilled(),
      parameters.AddVirtualBorder(), objects_to_use.data(),
      static_cast<int64_t>(objects_to_use.size()), device, sdf.GetMutableRawData().data(),
      &minimum, &maximum));
  detail::FinishSdf(sdf, minimum, maximum);
  return sdf;
}

// MakeSeparateObjectSDFs<T>(object_ids, parameters): the cells are uploaded once, one SDF per id.
template <typename MapType, typename ScalarType, typename Devices = int>
inline std::map<uint32_t, SignedDistanceField<ScalarType>> MakeSeparateObjectSDFs(
    const MapType& map, const std::vector<uint32_t>& object_ids,
    const SignedDistanceFieldGenerationParameters<ScalarType>& parameters,
    const Devices& device = 0)
{
  detail::RequireUniform(map);
  std::map<uint32_t, SignedDistanceField<ScalarType>> per_object_sdfs;
  if (object_ids.empty())
  {
    return per_object_sdfs;
  }
  const size_t voxels = static_cast<size_t>(map.NumTotalVoxels());
  std::vector<ScalarType> values(voxels * object_ids.size());
  std::vector<ScalarType> minima(object_ids.size());
  std::vector<ScalarType> maxima(object_ids.size());
  ThrowOnError(detail::CallPerObject(
      map.GetImmutableRawData().data(), detail::CellsOf<MapType>::kBytes, map.NumXVoxels(),
      map.NumYVoxels(), map.NumZVoxels(), map.VoxelXSize(), parameters.UnknownIsFilled(),
      parameters.AddVirtualBorder(), object_ids.data(), static_cast<int64_t>(object_ids.size()),
      device, values.data(), minima.data(), maxima.data()));
  for (size_t k = 0; k < object_ids.size(); k++)
  {
    SignedDistanceField<ScalarType> sdf(map.OriginTransform(), map.Frame(), map.ControlSizes(),
                                        parameters.OOBValue());
    std::copy(values.begin() + static_cast<std::ptrdiff_t>(k * voxels),
              values.begin() + static_cast<std::ptrdiff_t>((k + 1) * voxels),
              sdf.GetMutableRawData().begin());
    detail::FinishSdf(sdf, minima[k], maxima[k]);
    per_object_sdfs[object_ids[k]] = sdf;   // (a repeated id keeps its last SDF, as in the reference)
  }
  return per_object_sdfs;
}

// MakeAllObjectSDFs<T>(parameters): every object id > 0 present in the map
// (tagged_object_occupancy_map.hpp:264-291).
template <typename MapType, typename ScalarType, typename Devices = int>
inline std::map<uint32_t, SignedDistanceField<ScalarType>> MakeAllObjectSDFs(
    const MapType& map, const SignedDistanceFieldGenerationParameters<ScalarType>& parameters,
    const Devices& device = 0)
{
  std::set<uint32_t> present;
  for (const auto& cell : map.GetImmutableRawData())
  {
    if (cell.ObjectId() > 0)
    {
      present.insert(cell.ObjectId());
    }
  }
  return MakeSeparateObjectSDFs<MapType, ScalarType, Devices>(
      map, std::vector<uint32_t>(present.begin(), present.end()), parameters, device);
}

// ExtractFreeAndNamedObjectsSignedDistanceField<T>(parameters): both SDFs and the merge on the
// device (tagged_object_occupancy_map.hpp:293-378).
template <typename MapType, typename ScalarType, typename Devices = int>
inline SignedDistanceField<ScalarType> ExtractFreeAndNamedObjectsSignedDistanceField(
    const MapType& map, const SignedDistanceFieldGenerationParameters<ScalarType>& parameters,
    const Devices& device = 0)
{
  detail::RequireUniform(map);
  SignedDistanceField<ScalarType> sdf(map.OriginTransform(), map.Frame(), map.ControlSizes(),
                                      parameters.OOBValue());
  ScalarType minimum = 0;
  ScalarType maximum = 0;
  ThrowOnError(detail::CallFreeAndNamed(
      map.GetImmutableRawData().data(), detail::CellsOf<MapType>::kBytes, map.NumXVoxels(),
      map.NumYVoxels(), map.NumZVoxels(), map.VoxelXSize(), parameters.UnknownIsFilled(),
      parameters.AddVirtualBorder(), device, sdf.GetMutableRawData().data(), &minimum, &maximum));
  detail::FinishSdf(sdf, minimum, maximum);
  return sdf;
}
}  // namespace b200
}  // namespace signed_distance_field_generation
VGT_NAMESPACE_END
}  // namespace voxelized_geometry_tools
